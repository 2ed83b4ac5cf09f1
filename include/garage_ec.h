/*
 * garage_ec.h -- C ABI of libgarage_ec.so: the B200 (sm_100a) erasure-coding block path
 * for Garage.
 *
 * The reference (deuxfleurs-org/garage v1.2.0) has no FFI and no erasure coding; its
 * drop-in boundary is the Rust surface of garage_block::manager::BlockManager
 * (SURVEY.md section 8(b)).  Each entry point below names the reference call site whose
 * CPU-side per-block work it replaces; the Rust `src/block/cuda` shim that binds these
 * symbols is shown in INTEGRATION.md.
 *
 * Conventions (mirroring the reference's, SURVEY.md section 8(b)):
 *   errors     every call returns 0 or a negative GARAGE_EC_E_* code; nothing aborts or
 *              throws across the boundary (reference: Result<_, garage_util::error::Error>,
 *              src/util/error.rs:14-82; Rust maps non-zero to Error::Message /
 *              Error::CorruptData so resync's backoff handles it, src/block/resync.rs:300-315).
 *   ownership  caller owns every buffer; the library keeps no pointer after a HOST call
 *              returns, or after the stream work of a DEVICE call completes
 *              (reference: bytes::Bytes, immutable + refcounted).
 *   threading  a context may be used from many OS threads at once (reference: tokio
 *              spawn_blocking, src/block/block.rs:86, src/api/s3/put.rs:419,446).
 *   no CPU fallback: if there is no usable CUDA device, garage_ec_create fails with
 *              GARAGE_EC_E_NODEVICE.
 *
 * Arithmetic (normative definition in DESIGN.md; CPU oracle under oracle/):
 *   GF(2^8), polynomial 0x11D, alpha = 2.  One stripe = one block (post-compression bytes
 *   of DataBlock::from_buffer, src/block/block.rs:85-96).  shard_len = ceil(block_len/k);
 *   data shard j = block bytes [j*shard_len,(j+1)*shard_len) zero-padded; parity row
 *   i = XOR_j P[i][j] * data[j].
 *
 * Batch geometry ("shard layout"), shared by encode / reconstruct / verify:
 *   stride      bytes between consecutive shards; multiple of 16; >= every shard_len[s];
 *               (k+m)*stride < 4 GiB
 *   shard_len   per-stripe valid bytes per shard (NULL = `stride` for every stripe).
 *               Bytes in [shard_len, roundup16(shard_len)) of every OUTPUT shard are
 *               written as zero; input bytes there are ignored.  Beyond roundup16 nothing
 *               is written; input bytes up to `stride` may be read (the tile loads of the
 *               k >= 13 kernels fetch whole 512-byte rows) but never influence a result,
 *               so the whole n * shards * stride array must be addressable.
 *   all base pointers 16-byte aligned.
 */
#ifndef GARAGE_EC_H
#define GARAGE_EC_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GARAGE_EC_ABI_VERSION 1

/* error codes */
#define GARAGE_EC_OK 0
#define GARAGE_EC_E_INVALID (-1)       /* bad argument / geometry */
#define GARAGE_EC_E_CUDA (-2)          /* CUDA runtime error, see garage_ec_last_error */
#define GARAGE_EC_E_NOMEM (-3)         /* host or device allocation failed */
#define GARAGE_EC_E_UNRECOVERABLE (-4) /* >= 1 stripe had < k shards; see status[] */
#define GARAGE_EC_E_NODEVICE (-5)      /* no CUDA device / wrong architecture */
#define GARAGE_EC_E_ALIGN (-6)         /* pointer or stride alignment violated */
#define GARAGE_EC_E_UNCORRECTABLE (-7) /* >= 1 stripe had a column with more errors than t; see status[] */

/* matrix kinds */
#define GARAGE_EC_VANDERMONDE 0 /* systematic Vandermonde (default), G = V * inv(V[0..k)) */
#define GARAGE_EC_CAUCHY 1      /* P[i][j] = 1/((k+i) xor j) */

/* where the caller's buffers live */
#define GARAGE_EC_MEM_HOST 0   /* all pointers host; call is synchronous */
#define GARAGE_EC_MEM_DEVICE 1 /* all pointers device (this ctx's GPU); call enqueues on `stream` */

/* limits of this build */
#define GARAGE_EC_MAX_K 32
#define GARAGE_EC_MAX_M 8

typedef struct garage_ec_ctx garage_ec_ctx;

/* ---- lifecycle -------------------------------------------------------------------------
 * One context per (GPU, k, m, matrix).  Replaces nothing in the reference: it is the state
 * a BlockManager built with `erasure_coding = {data_shards, parity_shards}` would hold
 * next to `data_layout` (src/block/manager.rs:122-192).                                    */
int garage_ec_create(garage_ec_ctx **out, int cuda_device, int k, int m, int matrix_kind);
/* same, with an explicit m x k parity matrix (row-major) -- used by non-zero ranks after
 * the NCCL broadcast of rank 0's matrix (SURVEY.md section 8(e)).                          */
int garage_ec_create_with_matrix(garage_ec_ctx **out, int cuda_device, int k, int m,
                                 const uint8_t *parity_rows);
void garage_ec_destroy(garage_ec_ctx *ctx);

int garage_ec_matrix(const garage_ec_ctx *ctx, uint8_t *out_m_by_k); /* parity rows, row-major */
int garage_ec_params(const garage_ec_ctx *ctx, int *k, int *m, int *cuda_device);
const char *garage_ec_strerror(int code);
/* detail of the last GARAGE_EC_E_CUDA on this context (thread-unsafe snapshot; "" if none) */
const char *garage_ec_last_error(const garage_ec_ctx *ctx);
int garage_ec_abi_version(void);

/* ---- geometry helpers ------------------------------------------------------------------ */
uint32_t garage_ec_shard_len(uint32_t block_len, int k); /* ceil(block_len / k)            */
size_t garage_ec_stride_for(uint32_t shard_len);         /* shard_len rounded up to 128 B   */

/* ---- ENCODE -- call site: BlockManager::rpc_put_block, src/block/manager.rs:366-408,
 * right after DataBlock::from_buffer (manager.rs:376): the k data shards of each block go in,
 * the m parity shards come out; shard i is then sent to node i of the (k+m)-node set.
 *   data   : n * k * stride bytes, shard j of stripe s at (s*k + j) * stride
 *   parity : n * m * stride bytes, row  i of stripe s at (s*m + i) * stride                */
int garage_ec_encode(garage_ec_ctx *ctx, const uint8_t *data, uint8_t *parity,
                     const uint32_t *shard_len, size_t stride, size_t n_stripes, int mem_kind,
                     void *cuda_stream);

/* ---- RECONSTRUCT -- call sites: BlockManager::rpc_get_raw_block_internal,
 * src/block/manager.rs:276-339 (GET: any k of k+m shards arrived, rebuild the missing data
 * shards) and BlockResyncManager::resync_block fetch branch, src/block/resync.rs:460-500
 * (repair: rebuild this node's own shard from k survivors).
 *   shards  : n * (k+m) * stride bytes, shard i of stripe s at (s*(k+m) + i) * stride
 *   present : n * (k+m) bytes in {0,1}
 *   want    : NULL = rebuild every absent shard; else n*(k+m) bytes, only absent shards
 *             with want != 0 are rebuilt (GET wants data shards only; resync wants one)
 *   status  : n int32: 0 ok, GARAGE_EC_E_UNRECOVERABLE if < k present (stripe untouched)
 * Survivors used: the first k present shards in index order.  HOST calls return
 * GARAGE_EC_E_UNRECOVERABLE if any stripe was; DEVICE calls only fill status[].            */
int garage_ec_reconstruct(garage_ec_ctx *ctx, uint8_t *shards, const uint8_t *present,
                          const uint8_t *want, int32_t *status, const uint32_t *shard_len,
                          size_t stride, size_t n_stripes, int mem_kind, void *cuda_stream);

/* Gather form of the HOST-mode reconstruct for batching front-ends (SURVEY.md section 8 row f1): every
 * caller (a GET that lost shards, one of the 8 resync workers, src/block/resync.rs:43) owns its own
 * buffer -- stripes[s] points at the k+m shards of stripe s, `stride` apart -- and the batch is just the
 * list of those pointers: nobody copies shards into a contiguous staging array.  Pinned buffers from
 * garage_ec_host_alloc make the copies DMA-speed.  Same semantics as garage_ec_reconstruct(MEM_HOST). */
int garage_ec_reconstruct_stripes(garage_ec_ctx *ctx, uint8_t *const *stripes, const uint8_t *present,
                                  const uint8_t *want, int32_t *status, const uint32_t *shard_len,
                                  size_t stride, size_t n_stripes);

/* ---- VERIFY (scrub) -- call sites: DataBlock::verify via BlockManager::read_block,
 * src/block/manager.rs:554-609 / src/block/block.rs:69-83, driven by ScrubWorker::work,
 * src/block/repair.rs:438-490: recompute parity from the k data shards and compare with
 * the stored parity.  mismatch[s] bit i set iff parity row i differs.                      */
int garage_ec_verify(garage_ec_ctx *ctx, const uint8_t *shards, uint32_t *mismatch,
                     const uint32_t *shard_len, size_t stride, size_t n_stripes, int mem_kind,
                     void *cuda_stream);

/* ---- CORRECT (error-locating decode) -- call site: the DataBlock::verify failure on GET,
 * src/block/block.rs:69-83 (the block's content hash does not match although every shard passed its
 * own tag: a stale shard, a bad resync, bytes corrupted before they were tagged).  Finds and repairs
 * shards that are present but WRONG, from the parity alone (normative definition: DESIGN.md section 2).
 * Per stripe: e = number of absent shards, t = floor((m - e) / 2).
 *   e > m     status = GARAGE_EC_E_UNRECOVERABLE, stripe untouched;
 *   otherwise every byte column is decoded to the unique codeword that agrees with the received bytes
 *             at all present positions but at most t.  If every column decodes, the codeword is written
 *             into every absent shard and every present shard that differs from it (fixed[s*(k+m)+i] = 1
 *             for those), status = 0, output padding [shard_len, roundup16) written as zero.  If some
 *             column has no such codeword: status = GARAGE_EC_E_UNCORRECTABLE and NOTHING of the stripe
 *             is written (fixed stays 0) -- callers fall back to per-shard tags or a leave-one-out search.
 *   e = m     t = 0: a plain reconstruct, nothing is checked.
 * A column with more than t errors can still land within distance t of another codeword (probability
 * sum_{j<=t} C(k+m, j) 255^j / 256^m per column: ~0.14 % for RS(10,4), 2.3 % for RS(4,2)); the block's
 * content hash or the shard tags stay the final check.
 *   shards  : n * (k+m) * stride bytes, same layout / alignment / geometry rules as RECONSTRUCT
 *   present : n * (k+m) bytes in {0,1}, NULL = all present
 *   status  : n int32: 0, GARAGE_EC_E_UNRECOVERABLE or GARAGE_EC_E_UNCORRECTABLE
 *   fixed   : NULL or n * (k+m) bytes
 * HOST calls return GARAGE_EC_E_UNRECOVERABLE if any stripe was, else GARAGE_EC_E_UNCORRECTABLE if any
 * stripe was, else 0; they upload the present shards and download only the rebuilt or fixed ones.
 * DEVICE calls only fill status[] and never synchronise with the host (graph-capturable).
 * The matrix must be a generalized RS code with evaluation points 0..k+m-1 (both built-in kinds are; so is
 * garage_ec_create_with_matrix given a built-in matrix); for any other matrix this returns GARAGE_EC_E_INVALID. */
int garage_ec_correct(garage_ec_ctx *ctx, uint8_t *shards, const uint8_t *present, int32_t *status,
                      uint8_t *fixed, const uint32_t *shard_len, size_t stride, size_t n_stripes,
                      int mem_kind, void *cuda_stream);

/* ---- PER-SHARD INTEGRITY (SURVEY.md section 8 row f2) -- call sites: DataBlock::verify,
 * src/block/block.rs:69-83 (Plain => blake2sum(data) == hash) and read_block_from,
 * src/block/manager.rs:577-609.  A node stores 1/k of a block, so the whole-block hash cannot be
 * checked locally: every shard carries its own blake2sum (BLAKE2b-512 truncated to 32 bytes,
 * src/util/data.rs:130-138), computed here over [0, shard_len) of each shard.
 *   shards          : n_stripes * shards_per_stripe shards, `stride` apart (shard layout)
 *   shards_per_stripe: k (a data array), m (a parity array) or k+m
 *   sums_out        : 32 bytes per shard
 * garage_ec_check_sums compares with `expect` instead: bad_out[i] = 1 iff shard i differs.     */
int garage_ec_shard_sums(garage_ec_ctx *ctx, const uint8_t *shards, const uint32_t *shard_len,
                         size_t stride, size_t n_stripes, int shards_per_stripe, uint8_t *sums_out,
                         int mem_kind, void *cuda_stream);
int garage_ec_check_sums(garage_ec_ctx *ctx, const uint8_t *shards, const uint8_t *expect,
                         const uint32_t *shard_len, size_t stride, size_t n_stripes,
                         int shards_per_stripe, uint8_t *bad_out, int mem_kind, void *cuda_stream);
/* ---- SCRUB + REPAIR sweep (BASELINE config 5) -- ScrubWorker::work (src/block/repair.rs:438-490)
 * feeding resync (src/block/resync.rs:354-503) in one pass: blake2sum every shard, treat the ones
 * whose sum differs from `expect_sums` as erased, rebuild them in place from the first k intact
 * shards.  bad_out[s*(k+m)+i] = 1 iff shard i was corrupt; status[s] = 0 or
 * GARAGE_EC_E_UNRECOVERABLE (> m corrupt shards: reported, never fatal -- resync.rs:300-315).     */
int garage_ec_scrub_repair(garage_ec_ctx *ctx, uint8_t *shards, const uint8_t *expect_sums,
                           uint8_t *bad_out, int32_t *status, const uint32_t *shard_len,
                           size_t stride, size_t n_stripes, int mem_kind, void *cuda_stream);
/* host-side blake2sum of one buffer (the same function, for block hashes / small inputs)       */
void garage_ec_blake2sum(const uint8_t *data, size_t len, uint8_t out32[32]);
/* Which 32-byte tag the per-shard integrity calls of a context compute and compare
 * (garage_ec_shard_sums / _check_sums / _scrub_repair / _encode_blocks_with_sums):
 *   GARAGE_EC_SUM_BLAKE2 (default)  Garage's blake2sum of the shard (src/util/data.rs:130-138):
 *                     cryptographic, compute-bound on the GPU (~0.5 TB/s).
 *   GARAGE_EC_SUM_ADLER8  the shard cut in 8 segments of roundup16(ceil(len/8)) bytes, tag = the 8
 *                     little-endian zlib Adler-32 values of the segments (empty segment: 1).  Catches
 *                     bit rot, which is all scrub needs -- the block's content address stays its
 *                     blake2sum -- and streams at HBM speed (SURVEY.md section 8 row f2 allows a cheap
 *                     per-shard checksum).  The shard file header records which kind it carries.
 * garage_ec_shard_sum_host computes either tag on the CPU (nodes without a GPU, single shards).   */
#define GARAGE_EC_SUM_BLAKE2 0
#define GARAGE_EC_SUM_ADLER8 1
int garage_ec_set_sum_kind(garage_ec_ctx *ctx, int kind);
/* How HOST-mode calls of this context wait for the GPU: 0 (default) = cudaStreamSynchronize, the driver
 * spins on a CPU (lowest latency); 1 = block on an event, the waiting thread sleeps.  For callers that
 * keep several calls in flight from a small CPU budget -- the batching dispatchers in front of
 * rpc_put_block: three spinning waiters are three of the ~12 CPUs a host has per GPU.                   */
int garage_ec_set_wait_mode(garage_ec_ctx *ctx, int blocking);
int garage_ec_shard_sum_host(int kind, const uint8_t *data, size_t len, uint8_t out32[32]);

/* ---- BLOCK-LEVEL convenience (host memory only) -----------------------------------------
 * What rpc_put_block hands over is a contiguous block (bytes::Bytes), not shards.  These do
 * the framing (split + zero pad, src/api/s3/put.rs:583-617 block sizes) on the way to the
 * GPU so the Rust side needs no extra copy.
 *   blocks[s]     : block_len[s] bytes (host)
 *   parity_out    : n * m * stride bytes (host), row i of block s at (s*m + i) * stride.
 *                   The k data shards are just the slices block[j*L .. (j+1)*L) with
 *                   L = garage_ec_shard_len(block_len, k) (zero padded), so they never
 *                   cross PCIe back: Rust sends those slices of the original Bytes.
 *   stride        : >= garage_ec_shard_len(max block_len, k), multiple of 16               */
int garage_ec_encode_blocks(garage_ec_ctx *ctx, const uint8_t *const *blocks,
                            const uint32_t *block_len, size_t n_blocks, uint8_t *parity_out,
                            size_t stride);
/* same, and also returns the blake2sum of every shard (k data then m parity per block,
 * sums_out = n * (k+m) * 32 bytes), computed while the shards are on the device (row f2).   */
int garage_ec_encode_blocks_with_sums(garage_ec_ctx *ctx, const uint8_t *const *blocks,
                                      const uint32_t *block_len, size_t n_blocks,
                                      uint8_t *parity_out, uint8_t *sums_out, size_t stride);
/* inverse for GET: shards (host, shard layout) + present -> blocks_out[s] (block_len[s]
 * bytes each).  Runs reconstruct only for stripes with an absent data shard.               */
int garage_ec_decode_blocks(garage_ec_ctx *ctx, const uint8_t *shards, const uint8_t *present,
                            const uint32_t *block_len, size_t n_blocks, size_t stride,
                            uint8_t *const *blocks_out, int32_t *status);

/* ---- utilities used by the harness ------------------------------------------------------
 * device-side synthetic data (same splitmix64 counter stream as the oracle's
 * generator): fills dst[0..len) (device) with stream bytes at `offset`
 * (len, offset multiples of 8).                                                            */
int garage_ec_fill_random(garage_ec_ctx *ctx, uint8_t *dst_device, size_t len, uint64_t seed,
                          uint64_t offset, void *cuda_stream);
/* pinned host memory for block / shard buffers: the Rust side lands the HTTP body copy
 * (BytesBuf::take_exact, src/net/bytes_buf.rs:66-117) directly in such a buffer so the DMA
 * engines can read it.  Pageable memory is accepted everywhere, only slower.               */
int garage_ec_host_alloc(garage_ec_ctx *ctx, void **out, size_t bytes);
/* same, write-combined (cudaHostAllocWriteCombined): for buffers the CPU only WRITES sequentially and the
 * GPU reads (upload landing buffers) or the GPU writes and the CPU hands on without reading; CPU reads
 * from such memory are very slow.  The pages are not snooped during DMA.                              */
int garage_ec_host_alloc_wc(garage_ec_ctx *ctx, void **out, size_t bytes);
/* memcpy into a pinned buffer that the GPU reads next (the landing copy of a PUT body, BytesBuf::take_exact,
 * src/net/bytes_buf.rs:66-117; the survivors of a degraded GET).  Uses non-temporal stores so that the DMA
 * read finds the bytes in DRAM instead of snooping them out of the writing core's cache (7x faster upload
 * of freshly written data on the measured hosts).                                                          */
void garage_ec_copy_for_dma(void *dst_pinned, const void *src, size_t n);
void garage_ec_host_free(garage_ec_ctx *ctx, void *ptr);
/* NUMA placement.  On a multi-socket host each GPU hangs off one socket; garage_ec_host_alloc
 * places its pages on that socket's memory node (preferred-node policy + first touch from a CPU
 * of the node, both restored before returning), so DMA never crosses the inter-socket link.
 * garage_ec_numa_info reports the GPU's node and the node the last garage_ec_host_alloc of this
 * context landed on (-1 = unknown).  garage_ec_bind_thread pins the CALLING thread to the CPUs
 * of the GPU's node -- for the threads that fill those buffers (the batching workers in front of
 * rpc_put_block / the 8 resync workers, src/block/resync.rs:43; spawn_blocking threads,
 * src/block/block.rs:86): returns 0 if bound, 1 if nothing was changed (topology unknown or not
 * permitted).                                                                               */
int garage_ec_numa_info(const garage_ec_ctx *ctx, int *gpu_node, int *last_alloc_node);
int garage_ec_bind_thread(const garage_ec_ctx *ctx);

/* number of kernel launches issued by this context so far (bench.py's gpu_launches)        */
uint64_t garage_ec_launch_count(const garage_ec_ctx *ctx);
/* per-kernel CUDA-event timing of the RS kernels (encode / reconstruct / verify main
 * kernel, recorded on the stream they were launched on).  garage_ec_timing_read waits for
 * the recorded kernels, adds their durations to *total_ms / *launches and resets.          */
int garage_ec_set_timing(garage_ec_ctx *ctx, int enabled);
int garage_ec_timing_read(garage_ec_ctx *ctx, double *total_ms, uint64_t *launches);

/* test hook: the n_calls-th checked CUDA runtime call issued by this context from now on fails
 * (n_calls = 0: the next one; < 0: off).  Used by the fault-injection tests of the HOST-mode
 * ownership contract: after a failed call returns, nothing may still write the caller's buffers. */
int garage_ec_debug_fail_after(garage_ec_ctx *ctx, long n_calls);

#ifdef __cplusplus
}
#endif
#endif /* GARAGE_EC_H */
