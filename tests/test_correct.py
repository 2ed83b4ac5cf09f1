"""garage_ec_correct: error-locating decode (DESIGN.md section 2).  Shards that are present but hold
the wrong bytes are found and repaired from the parity alone, up to t = floor((m - e) / 2) per byte
column (e = absent shards).

CPU: the GRS structure both matrix kinds rely on (pure-Python GF, independent of the library and of
the oracle), and the brute-force numpy oracle.  GPU: the kernels against that oracle byte for byte,
DEVICE / HOST / CUDA-graph agreement, a full-size batch, the HOST ownership contract under injected
faults, the block-manager GET path, and the matrix check of custom contexts."""
import os
import sys
from math import comb

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import rs_oracle_np as N  # noqa: E402
from correct_oracle import correct as oracle_correct  # noqa: E402

import garage_b200 as G  # noqa: E402


# ---------------------------------------------------------------- pure-Python GF(2^8)/0x11D
def _gmul(a, b):
    r = 0
    while b:
        if b & 1:
            r ^= a
        a <<= 1
        if a & 0x100:
            a ^= 0x11D
        b >>= 1
    return r


def _gpow(a, e):
    r = 1
    for _ in range(e):
        r = _gmul(r, a)
    return r


def _ginv(a):
    return _gpow(a, 254)


def _nullspace(rows, ncols):
    """basis of the null space of `rows` (lists of field elements) by Gauss-Jordan elimination"""
    A = [list(r) for r in rows]
    piv_cols, r0 = [], 0
    for c in range(ncols):
        pr = next((r for r in range(r0, len(A)) if A[r][c]), None)
        if pr is None:
            continue
        A[r0], A[pr] = A[pr], A[r0]
        iv = _ginv(A[r0][c])
        A[r0] = [_gmul(x, iv) for x in A[r0]]
        for r in range(len(A)):
            if r != r0 and A[r][c]:
                f = A[r][c]
                A[r] = [x ^ _gmul(f, y) for x, y in zip(A[r], A[r0])]
        piv_cols.append(c)
        r0 += 1
    basis = []
    for fc in (c for c in range(ncols) if c not in piv_cols):
        v = [0] * ncols
        v[fc] = 1
        for i, pc in enumerate(piv_cols):
            v[pc] = A[i][fc]
        basis.append(v)
    return basis


def _parity_rows(k, m, kind):
    if kind == 1:
        return [[_ginv((k + i) ^ j) for j in range(k)] for i in range(m)]
    # systematic Vandermonde: P = V[k..k+m) inv(V[0..k)), V[r][c] = r^c -- by solving V[0..k)^T X = V[k..)^T
    V = [[_gpow(r, c) for c in range(k)] for r in range(k + m)]
    P = []
    for i in range(m):
        rows = [[V[c][j] for c in range(k)] + [V[k + i][j]] for j in range(k)]
        ns = _nullspace(rows, k + 1)  # [x, -1] with top^T x = bottom^T
        assert len(ns) == 1 and ns[0][k] == 1
        P.append(ns[0][:k])
    return P


def _grs_multipliers(k, m, P):
    """v with sum_r v_r r^l c_r = 0 for every codeword c = (d, P d) and l < m"""
    rows = []
    for j in range(k):
        for l in range(m):
            row = [0] * (k + m)
            row[j] = _gpow(j, l)
            for i in range(m):
                row[k + i] = _gmul(_gpow(k + i, l), P[i][j])
            rows.append(row)
    return _nullspace(rows, k + m)


# ---------------------------------------------------------------- CPU tests
@pytest.mark.parametrize("kind", [G.VANDERMONDE, G.CAUCHY])
def test_builtin_matrices_are_grs_codes(kind):
    """every (k, m) with k <= 32, m <= 8: the dual-multiplier system has nullity exactly 1 and no
    multiplier is zero -- what lets the decoder work with syndromes"""
    for m in range(1, 9):
        for k in range(1, 33):
            P = _parity_rows(k, m, kind)
            if kind == G.VANDERMONDE and k in (1, 10, 32) and m in (1, 4, 8):
                assert np.array_equal(np.array(P, dtype=np.uint8), N.build_matrix(k, m, kind))
            ns = _grs_multipliers(k, m, P)
            assert len(ns) == 1, (k, m, kind, len(ns))
            assert all(ns[0]), (k, m, kind)


def test_random_matrix_is_not_grs():
    rng = np.random.default_rng(5)
    P = rng.integers(1, 256, (4, 10)).tolist()
    assert _grs_multipliers(10, 4, P) == []


def _codeword(k, m, P, L, rng):
    d = rng.integers(0, 256, (k, L), dtype=np.uint8)
    return np.concatenate([d, N.encode(P, d)])


@pytest.mark.parametrize("k,m", [(4, 2), (6, 3), (10, 4), (3, 5), (4, 8)])
@pytest.mark.parametrize("kind", [N.VANDERMONDE, N.CAUCHY])
def test_oracle_returns_the_original_within_t(k, m, kind):
    rng = np.random.default_rng(k * 100 + m * 10 + kind)
    P = N.build_matrix(k, m, kind)
    for trial in range(6):
        c = _codeword(k, m, P, 23, rng)
        e = int(rng.integers(0, m + 1))
        t = (m - e) // 2
        pres = np.ones(k + m, dtype=np.uint8)
        pres[rng.choice(k + m, e, replace=False)] = 0
        y = c.copy()
        y[pres == 0] = rng.integers(0, 256, (e, 23), dtype=np.uint8)
        cand = np.flatnonzero(pres)
        for col in range(23):
            for p in rng.choice(cand, int(rng.integers(0, t + 1)), replace=False):
                y[p, col] ^= int(rng.integers(1, 256))
        wrong = (y != c).any(axis=1) & (pres == 1)
        st, fixed = oracle_correct(k, m, P, y, pres)
        assert st == 0 and np.array_equal(y, c)
        assert np.array_equal(fixed.astype(bool), wrong)


@pytest.mark.parametrize("k,m", [(4, 2), (6, 3), (10, 4)])
def test_oracle_beyond_t_is_uncorrectable_or_within_radius(k, m):
    rng = np.random.default_rng(77 + k)
    P = N.build_matrix(k, m, 0)
    t = m // 2
    for trial in range(8):
        c = _codeword(k, m, P, 40, rng)
        y = c.copy()
        for col in range(40):
            for p in rng.choice(k + m, t + 1, replace=False):
                y[p, col] ^= int(rng.integers(1, 256))
        y0 = y.copy()
        st, fixed = oracle_correct(k, m, P, y, None)
        if st == -7:
            assert np.array_equal(y, y0) and not fixed.any()
        else:
            assert st == 0 and N.verify(k, m, P, y) == 0
            assert ((y != y0).sum(axis=0) <= t).all()


def test_oracle_more_than_m_absent_is_unrecoverable():
    P = N.build_matrix(4, 2, 0)
    y = _codeword(4, 2, P, 8, np.random.default_rng(1))
    y0 = y.copy()
    st, fixed = oracle_correct(4, 2, P, y, [0, 0, 0, 1, 1, 1])
    assert st == -4 and np.array_equal(y, y0) and not fixed.any()


def test_strerror_uncorrectable():
    L = G.load_library()
    s = L.garage_ec_strerror(G.E_UNCORRECTABLE)
    assert s and s != L.garage_ec_strerror(-99)


# ---------------------------------------------------------------- GPU helpers
PATTERNS = ["clean", "scattered", "stale", "erasures+errors", "beyond_t", "beyond_m"]


def _batch(k, m, kind, n, stride, seed):
    """n stripes (shard layout) with per-stripe patterns; returns (input, original, present, shard_len, pattern)"""
    rng = np.random.default_rng(seed)
    P = N.build_matrix(k, m, kind)
    tot = k + m
    lens = rng.integers(1, stride + 1, n).astype(np.uint32)
    lens[0] = stride
    orig = np.zeros((n, tot, stride), dtype=np.uint8)
    y = np.zeros_like(orig)
    pres = np.ones((n, tot), dtype=np.uint8)
    pats = []
    for s in range(n):
        L = int(lens[s])
        c = _codeword(k, m, P, L, rng)
        orig[s, :, :L] = c
        yc = c.copy()
        pat = PATTERNS[s % len(PATTERNS)]
        t = m // 2
        if pat == "scattered" and t:
            for col in rng.choice(L, min(L, 5), replace=False):
                for p in rng.choice(tot, int(rng.integers(1, t + 1)), replace=False):
                    yc[p, col] ^= int(rng.integers(1, 256))
        elif pat == "stale" and t:
            for p in rng.choice(tot, int(rng.integers(1, t + 1)), replace=False):
                yc[p] = rng.integers(0, 256, L, dtype=np.uint8)
        elif pat == "erasures+errors":
            e = int(rng.integers(1, m + 1))
            pres[s, rng.choice(tot, e, replace=False)] = 0
            te = (m - e) // 2
            cand = np.flatnonzero(pres[s])
            if te:
                for p in rng.choice(cand, te, replace=False):
                    yc[p, rng.choice(L, min(L, 3), replace=False)] ^= rng.integers(1, 256, min(L, 3), dtype=np.uint8)
        elif pat == "beyond_t":
            for p in rng.choice(tot, min(tot, t + 1), replace=False):
                yc[p] = rng.integers(0, 256, L, dtype=np.uint8)
        elif pat == "beyond_m":
            pres[s, rng.choice(tot, min(tot, m + 1), replace=False)] = 0
        yc[pres[s] == 0] = rng.integers(0, 256, ((pres[s] == 0).sum(), L), dtype=np.uint8)
        y[s, :, :L] = yc
        r16 = (L + 15) & ~15
        y[s, :, L:r16] = 0xA5  # sentinel: ignored as input, zero in every written shard
        y[s, :, r16:] = 0x5A  # never written
        pats.append(pat)
    return y, orig, pres, lens, pats


def _brute_force_cheap(k, m, e):
    t = (m - e) // 2
    return t <= 2 and sum(comb(k + m - e, j) for j in range(t + 1)) <= 120 or k + m <= 12


def _expected(k, m, kind, y, pres, lens, orig, pats):
    """expected output / status / fixed: the oracle where brute force is cheap, else the known original
    (stripes whose outcome is not known a priori are returned as None and checked for consistency)"""
    P = N.build_matrix(k, m, kind)
    n, tot, stride = y.shape
    out = y.copy()
    status = np.zeros(n, dtype=np.int32)
    fixed = np.zeros((n, tot), dtype=np.uint8)
    unknown = []
    for s in range(n):
        L = int(lens[s])
        e = int(tot - pres[s].sum())
        if e <= m and _brute_force_cheap(k, m, e):
            w = y[s, :, :L].copy()
            st, fx = oracle_correct(k, m, P, w, pres[s])
        elif e > m:
            st, fx = -4, np.zeros(tot, dtype=np.uint8)
        elif pats[s] != "beyond_t":
            w = orig[s, :, :L].copy()
            st, fx = 0, ((y[s, :, :L] != w).any(axis=1) & (pres[s] == 1)).astype(np.uint8)
        else:
            unknown.append(s)
            continue
        status[s] = st
        if st == 0:
            fixed[s] = fx
            r16 = (L + 15) & ~15
            for i in range(tot):
                if fx[i] or not pres[s, i]:
                    out[s, i, :L] = w[i]
                    out[s, i, L:r16] = 0
    return out, status, fixed, unknown


def _check(k, m, kind, y, pres, lens, orig, pats, got, st, fx):
    out, status, fixed, unknown = _expected(k, m, kind, y, pres, lens, orig, pats)
    P = N.build_matrix(k, m, kind)
    t = m // 2
    for s in range(y.shape[0]):
        if s in unknown:
            L = int(lens[s])
            assert st[s] in (0, G.E_UNCORRECTABLE), (s, st[s])
            if st[s] == G.E_UNCORRECTABLE:
                assert np.array_equal(got[s], y[s]) and not fx[s].any(), s
            else:  # miscorrected onto another codeword within radius t
                assert N.verify(k, m, P, got[s, :, :L].copy()) == 0
                assert ((got[s, :, :L] != y[s, :, :L]).sum(axis=0) <= t).all()
            continue
        assert st[s] == status[s], (s, pats[s], st[s], status[s])
        assert np.array_equal(fx[s], fixed[s]), (s, pats[s])
        assert np.array_equal(got[s], out[s]), (s, pats[s])
        if pats[s] in ("clean", "scattered", "stale", "erasures+errors") and m // 2:
            assert st[s] == 0 and np.array_equal(got[s, :, :int(lens[s])], orig[s, :, :int(lens[s])]), s


SHAPES = [(4, 2), (6, 3), (10, 4), (12, 4), (16, 4), (20, 4), (32, 4), (4, 8), (17, 8), (32, 8)]


@pytest.fixture(scope="module")
def torch():
    import torch as t

    assert t.cuda.is_available()
    return t


@pytest.mark.gpu
@pytest.mark.parametrize("k,m", SHAPES)
@pytest.mark.parametrize("kind", [G.VANDERMONDE, G.CAUCHY])
def test_correct_matches_oracle(torch, k, m, kind):
    n, stride = 18, 384
    y, orig, pres, lens, pats = _batch(k, m, kind, n, stride, seed=k * 1000 + m * 10 + kind)
    with G.GarageEc(0, k, m, kind=kind) as ec:
        d_sh = torch.from_numpy(y.reshape(-1).copy()).cuda()
        d_pr = torch.from_numpy(pres.reshape(-1).copy()).cuda()
        d_len = torch.from_numpy(lens.copy()).cuda()
        d_st = torch.full((n,), 99, dtype=torch.int32, device="cuda")
        d_fx = torch.full((n * (k + m),), 7, dtype=torch.uint8, device="cuda")
        ec.correct(d_sh, stride, n, present=d_pr, status=d_st, fixed=d_fx, shard_len=d_len)
        torch.cuda.synchronize()
        got = d_sh.cpu().numpy().reshape(y.shape)
        _check(k, m, kind, y, pres, lens, orig, pats, got, d_st.cpu().numpy(), d_fx.cpu().numpy().reshape(n, k + m))


@pytest.mark.gpu
@pytest.mark.parametrize("k,m", [(10, 4), (6, 3), (17, 8)])
def test_device_host_and_graph_agree(torch, k, m):
    n, stride = 30, 512
    y, orig, pres, lens, pats = _batch(k, m, 0, n, stride, seed=9 + k)
    with G.GarageEc(0, k, m) as ec:
        h_sh = y.reshape(-1).copy()
        h_st = np.zeros(n, dtype=np.int32)
        h_fx = np.zeros(n * (k + m), dtype=np.uint8)
        rc = ec.correct(h_sh, stride, n, present=pres.reshape(-1).copy(), status=h_st, fixed=h_fx, shard_len=lens.copy())
        assert rc == G.E_UNRECOVERABLE  # some stripes have more than m absent
        d_pr = torch.from_numpy(pres.reshape(-1).copy()).cuda()
        d_len = torch.from_numpy(lens.copy()).cuda()
        d_sh = torch.from_numpy(y.reshape(-1).copy()).cuda()
        d_st = torch.zeros(n, dtype=torch.int32, device="cuda")
        d_fx = torch.zeros(n * (k + m), dtype=torch.uint8, device="cuda")
        ec.correct(d_sh, stride, n, present=d_pr, status=d_st, fixed=d_fx, shard_len=d_len)
        torch.cuda.synchronize()
        assert np.array_equal(d_sh.cpu().numpy(), h_sh)
        assert np.array_equal(d_st.cpu().numpy(), h_st)
        assert np.array_equal(d_fx.cpu().numpy(), h_fx)
        # captured in a CUDA graph, replayed on a fresh copy of the input
        g_sh = torch.from_numpy(y.reshape(-1).copy()).cuda()
        g_st = torch.zeros(n, dtype=torch.int32, device="cuda")
        g_fx = torch.zeros(n * (k + m), dtype=torch.uint8, device="cuda")
        src = g_sh.clone()
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            ec.correct(g_sh, stride, n, present=d_pr, status=g_st, fixed=g_fx, shard_len=d_len)
        torch.cuda.synchronize()
        g_sh.copy_(src)
        g_st.zero_()
        g_fx.zero_()
        graph.replay()
        torch.cuda.synchronize()
        assert np.array_equal(g_sh.cpu().numpy(), h_sh)
        assert np.array_equal(g_st.cpu().numpy(), h_st)
        assert np.array_equal(g_fx.cpu().numpy(), h_fx)


@pytest.mark.gpu
def test_full_size_rs_10_4(torch):
    """4096 x 1 MiB RS(10,4): one stale shard in 1 % of the stripes, two byte-flipped shards in another
    1 %, the rest clean; afterwards every stripe equals the encode of its data"""
    k, m, n = 10, 4, 4096
    L = (1 << 20) // k + 1  # 104858
    stride = 104960
    tot = k + m
    with G.GarageEc(0, k, m) as ec:
        sh = torch.empty(n * tot * stride, dtype=torch.uint8, device="cuda")
        v = sh.view(n, tot, stride)
        data = torch.empty(n * k * stride, dtype=torch.uint8, device="cuda")
        ec.fill_random(data, data.numel(), 2024)
        par = torch.empty(n * m * stride, dtype=torch.uint8, device="cuda")
        lens = torch.full((n,), L, dtype=torch.int32, device="cuda")
        ec.encode(data, par, stride, n, shard_len=lens)
        v[:, :k] = data.view(n, k, stride)
        v[:, k:] = par.view(n, m, stride)
        v[:, :, L:] = 0
        ref = sh.clone()
        g = torch.Generator(device="cuda").manual_seed(3)
        perm = torch.randperm(n, device="cuda", generator=g)
        stale, flip = perm[:41].tolist(), perm[41:82].tolist()
        for i, s in enumerate(stale):
            v[s, (i * 3) % tot, :L] = torch.randint(0, 256, (L,), dtype=torch.uint8, device="cuda", generator=g)
        for i, s in enumerate(flip):
            for j in ((i + 1) % tot, (i + 5) % tot):
                cols = torch.randint(0, L, (64,), device="cuda", generator=g)
                v[s, j, cols] ^= torch.randint(1, 256, (64,), dtype=torch.uint8, device="cuda", generator=g)
        st = torch.full((n,), 99, dtype=torch.int32, device="cuda")
        fx = torch.zeros(n * tot, dtype=torch.uint8, device="cuda")
        ec.correct(sh, stride, n, status=st, fixed=fx, shard_len=lens)
        torch.cuda.synchronize()
        assert int(st.abs().sum()) == 0
        assert torch.equal(sh, ref)
        fxv = fx.view(n, tot).cpu().numpy()
        assert int(fxv.sum()) == 41 + 82
        assert all(fxv[s, (i * 3) % tot] == 1 for i, s in enumerate(stale))


@pytest.mark.gpu
@pytest.mark.parametrize("fail_at", [0, 1, 2, 4, 7, 11])
def test_host_fault_leaves_no_dma_in_flight(torch, fail_at):
    """HOST ownership under injected faults: after the error return, nothing writes the caller's buffers"""
    k, m, stride, n = 10, 4, 104960, 160  # several 48 MB chunks
    y, orig, pres, lens, pats = _batch(k, m, 0, n, stride, seed=31)
    with G.GarageEc(0, k, m) as ec:
        ref_sh = y.reshape(-1).copy()
        st0 = np.zeros(n, dtype=np.int32)
        fx0 = np.zeros(n * (k + m), dtype=np.uint8)
        ec.correct(ref_sh, stride, n, present=pres.reshape(-1).copy(), status=st0, fixed=fx0, shard_len=lens.copy())
        sh = y.reshape(-1).copy()
        st = np.zeros(n, dtype=np.int32)
        fx = np.zeros(n * (k + m), dtype=np.uint8)
        ec.debug_fail_after(fail_at)
        with pytest.raises(G.EcError) as ei:
            ec.correct(sh, stride, n, present=pres.reshape(-1).copy(), status=st, fixed=fx, shard_len=lens.copy())
        assert ei.value.code in (G.E_CUDA, G.E_NOMEM)
        ec.debug_fail_after(-1)
        sh[:] = 0xEE
        st[:] = 0x0EEEEEEE
        fx[:] = 0xEE
        torch.cuda.synchronize()
        assert (sh == 0xEE).all() and (st == 0x0EEEEEEE).all() and (fx == 0xEE).all()
        sh = y.reshape(-1).copy()
        ec.correct(sh, stride, n, present=pres.reshape(-1).copy(), status=st, fixed=fx, shard_len=lens.copy())
        assert np.array_equal(sh, ref_sh) and np.array_equal(st, st0) and np.array_equal(fx, fx0)


@pytest.mark.gpu
def test_block_manager_get_repairs_two_stale_shards(tmp_path):
    from garage_b200 import block_manager as BM

    sys.path.insert(0, HERE)
    import oracle_lib as O

    k, m = 10, 4
    b = O.fill_random(1 << 20, 71)
    with BM.BlockManager(k, m) as bm:
        h = BM.blake2sum(b)
        assert bm.rpc_put_block(h, b) == BM.OK
        who = bm.storage_nodes_of(h)
        for i in (2, 7):
            assert bm.plant_stale_shard(who[i], h) == BM.OK
        rc, got = bm.rpc_get_block(h)
        assert rc == BM.OK and np.array_equal(got, b)
        mt = bm.metrics()
        assert mt["corruption_counter"] == 2 and mt["resync_queue_length"] == 2
        assert bm.node_shard_index(who[2], h) == -1 and bm.node_shard_index(who[7], h) == -1
        assert bm.resync_all(who[2]) == (0, 1)
        assert bm.resync_all(who[7]) == (0, 1)
        assert bm.node_shard_index(who[2], h) == 2 and bm.node_shard_index(who[7], h) == 7
        rc, got = bm.rpc_get_block(h)
        assert rc == BM.OK and np.array_equal(got, b) and bm.metrics()["corrupt_data_errors"] == 1


@pytest.mark.gpu
def test_custom_matrix_needs_grs_structure(torch):
    k, m, n, stride = 10, 4, 6, 256
    rng = np.random.default_rng(8)
    y, orig, pres, lens, pats = _batch(k, m, 0, n, stride, seed=44)
    with G.GarageEc(0, k, m, matrix=rng.integers(1, 256, (m, k), dtype=np.uint8)) as ec:
        with pytest.raises(G.EcError) as ei:
            ec.correct(y.reshape(-1).copy(), stride, n)
        assert ei.value.code == G.E_INVALID
    with G.GarageEc(0, k, m, matrix=N.build_matrix(k, m, 0)) as ec:
        sh = y.reshape(-1).copy()
        st = np.zeros(n, dtype=np.int32)
        fx = np.zeros(n * (k + m), dtype=np.uint8)
        ec.correct(sh, stride, n, present=pres.reshape(-1).copy(), status=st, fixed=fx, shard_len=lens.copy())
        _check(k, m, 0, y, pres, lens, orig, pats, sh.reshape(y.shape), st, fx.reshape(n, k + m))
