"""Brute-force reference for garage_ec_correct (error-locating decode, DESIGN.md section 2).

TEST INFRASTRUCTURE ONLY.  Built on the independent numpy restatement of the arithmetic in
oracle/rs_oracle_np.py (shift-and-xor multiplication, composed decode matrices) and deliberately
unrelated to the product's syndrome decoder: no syndromes, no locator polynomials, just an exhaustive
search for the nearest codeword.
"""
import os
import sys
from itertools import combinations

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
from rs_oracle_np import reconstruct  # noqa: E402


def correct(k, m, P, shards, present=None):
    """Error-locating decode of one stripe by exhaustive nearest-codeword search.

    shards: (k+m, L) uint8, modified in place only on success.  present: k+m flags (None = all).
    Every byte column is decoded to the codeword that agrees with the received bytes at all present
    positions but at most t = (m - e) // 2 (e = absent shards).  The search tries every error support
    of size <= t: rebuild the column from k positions outside (erasures + support) and accept it where
    it agrees with every position outside (erasures + support).  Deliberately unrelated to the syndrome
    decoder of the product (no syndromes, no locator polynomials).

    Returns (status, fixed): status 0, -4 (e > m: untouched) or -7 (some column has no codeword within
    t: untouched); fixed[i] = 1 for the present shards that were rewritten.
    """
    n = k + m
    pres = np.ones(n, dtype=bool) if present is None else np.asarray(present).astype(bool)
    fixed = np.zeros(n, dtype=np.uint8)
    erased = [i for i in range(n) if not pres[i]]
    e = len(erased)
    if e > m:
        return -4, fixed
    t = (m - e) // 2
    y = shards.copy()
    y[erased] = 0
    L = y.shape[1]
    out = np.zeros_like(y)
    done = np.zeros(L, dtype=bool)
    cand = [i for i in range(n) if pres[i]]
    for size in range(t + 1):
        for sup in combinations(cand, size):
            keep = [i for i in cand if i not in sup]
            trial = y.copy()
            mask = np.zeros(n, dtype=np.uint8)
            mask[keep[:k]] = 1
            reconstruct(k, m, P, trial, mask)
            ok = np.all(trial[keep] == y[keep], axis=0) & ~done
            out[:, ok] = trial[:, ok]
            done |= ok
            if done.all():
                break
        if done.all():
            break
    if not done.all():
        return -7, fixed
    for i in cand:
        if not np.array_equal(out[i], y[i]):
            fixed[i] = 1
    shards[:] = out
    return 0, fixed
