// topk.cu — K10: per-row top-k of a factorised score matrix  score[r, i] = <A[r], B[i]> + row_bias[r] + col_bias[i],
// without materialising the n_rows x n_items scores.  sm_100a only.
//
// Precision: both operands are split into three bf16 pieces (x = x0 + x1 + x2 up to ~2^-24 |x|) by a staging pass, and the
// six products that matter are one bf16 GEMM over a 6x longer contraction:  A' = [a0 a0 a1 a0 a1 a2],  B' = [b0 b1 b0 b2 b1 b0].
// The dropped terms are <= ~2^-24 relative, so the fp32 accumulator sees an fp32-grade dot product.
//
// Staging (factor_split_kernel): A' and B' are written to the workspace already in the UMMA "K-major, no swizzle" core-matrix
// layout, one contiguous block per (tile, 64-element contraction chunk):  [chunk c = k/8 (8)][row (128 or 256)][8 bf16].
// A ring stage of the main kernel is therefore two TMA bulk copies (16 KB of A, 32 KB of B).
//
// Main kernel (factor_topk_kernel): one CTA per (128-row tile, item slice).  Warp 4 streams the ring, warp 5 issues
// tcgen05.mma (M = 128, N = 256, fp32 accumulators in TMEM, two buffers = all 512 columns so the MMAs of item tile j+1 run
// while the epilogue scans tile j), warps 0-3 are the epilogue: thread t owns row t (TMEM lane t).  Per score it adds the
// biases and compares with a per-row threshold held in a register; the scores of a 16-column chunk that beat it are queued
// in shared memory, and the warp's lanes then drain their queues together: a step along the row's exclusion list (walked
// forward, ids ascend) and an insertion into the row's k-entry min-heap (in shared memory when 128 * k entries fit next
// to the ring, else in the row's slot of the workspace).  Until k items have arrived the heap is a plain append buffer,
// heapified once.  Heap keys are 64-bit (order-preserving score bits << 32 | ~item), so one unsigned compare gives
// the order (score desc, item asc).  Items reach a slice in ascending id order, so a later item that ties the threshold
// always loses: the scan compares scores with a strict '>' — which also means a NaN score is never returned.
//
// Merge (factor_topk_merge_kernel): each slice leaves its k best keys sorted per row in the workspace; one thread per row
// merges the S sorted lists into the final k (score, item) pairs.  Empty slots (fewer than k eligible items) are key 0,
// which no real score produces (f2ord(-inf) = 0x007FFFFF), and come out as item -1, score -inf.
#include <math.h>

#include <algorithm>

#include "rbr_common.cuh"
#include "tc_ptx.cuh"

namespace rbr {

constexpr int FT_M = 128;                              // rows per tile (UMMA M, TMEM lanes)
constexpr int FT_N = 256;                              // items per tile (UMMA N)
constexpr int FT_KC = 64;                              // contraction elements per ring stage (4 UMMA K-steps)
constexpr int FT_A_BYTES = FT_M * FT_KC * 2;           // 16 KB
constexpr int FT_B_BYTES = FT_N * FT_KC * 2;           // 32 KB
constexpr int FT_STAGE_BYTES = FT_A_BYTES + FT_B_BYTES;
constexpr int FT_THREADS = 192;                        // warps 0-3 epilogue, 4 producer, 5 MMA issuer
constexpr int FT_PROD_WARP = 4, FT_MMA_WARP = 5;
constexpr int FT_SMEM_MAX = 232448;                    // 227 KB opt-in dynamic shared memory per CTA
constexpr int FT_MAX_SLICES = 16;
constexpr int FT_QUEUE_BYTES = FT_M * 16 * 8;          // per row: the candidate keys of one 16-column chunk
constexpr int64_t FT_PART_CAP = 96ll << 20;            // cap on the per-slice partial lists when choosing several slices
constexpr int FT_MAX_K = 256, FT_MAX_DIM = 512;

struct FtPlan {
    int64_t dimp;       // dim rounded up to 32 (6 * dimp is a whole number of 64-element chunks)
    int64_t nq;         // ring stages per item tile = 6 * dimp / 64
    int64_t rt, it;     // row tiles, item tiles
    int64_t S, tps;     // item slices, item tiles per slice
    int nst;            // ring stages
    int heap_smem;      // 1: per-row heaps in shared memory
    int smem;           // dynamic shared memory bytes
    int64_t off_b, off_part, total;   // workspace: A' | B' | partial top-k keys [n_rows][S][k]
};

static int ft_sm_count() {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
        n <= 0) {
        cudaGetLastError();
        return 148;                                     // B200
    }
    return n;
}

static bool ft_supported(int64_t n_rows, int64_t n_items, int64_t dim, int64_t k) {
    return n_rows >= 0 && n_items >= 1 && n_items < (1ll << 31) && dim >= 1 && dim <= FT_MAX_DIM && k >= 1 && k <= FT_MAX_K;
}

static FtPlan ft_plan(int64_t n_rows, int64_t n_items, int64_t dim, int64_t k, int sms) {
    FtPlan p;
    p.dimp = round_up(dim, 32);
    p.nq = 6 * p.dimp / FT_KC;
    p.rt = (n_rows + FT_M - 1) / FT_M;
    p.it = (n_items + FT_N - 1) / FT_N;
    // Slices: the CTA's cost is roughly its item tiles plus a share per slice that grows with k (filling, sorting and
    // writing its heaps, and the threshold starting over); the grid runs in waves of one CTA per SM.  Take the slice
    // count with the fewest wave-weighted tiles.  The share, in tiles, was fitted to timings at 20 000 x 12 000 on a
    // B200 (k = 10: 3 slices best, k = 100: 1-2).
    const double fill = 3.0 + (double)k / 16.0;
    int64_t best = 1;
    double best_cost = 1e300;
    const int64_t smax = p.it < FT_MAX_SLICES ? p.it : FT_MAX_SLICES;
    for (int64_t s = 1; s <= smax; ++s) {
        if (s > 1 && n_rows * s * k * 8 > FT_PART_CAP) break;
        const int64_t tps = (p.it + s - 1) / s;
        if ((p.it + tps - 1) / tps != s) continue;     // every slice must own at least one tile
        const int64_t waves = (p.rt * s + sms - 1) / sms;
        const double cost = (double)waves * ((double)tps + fill);
        if (cost < best_cost * 0.97) { best_cost = cost; best = s; }
    }
    p.S = best;
    p.tps = (p.it + p.S - 1) / p.S;
    const int64_t heap_bytes = (int64_t)FT_M * k * 8;
    const int64_t fixed = FT_QUEUE_BYTES + 1024;        // candidate queues, barriers + TMEM slot
    p.heap_smem = 0;
    p.nst = 4;
    for (int nst = 4; nst >= 2; --nst) {
        if (nst * FT_STAGE_BYTES + heap_bytes + fixed <= FT_SMEM_MAX) { p.nst = nst; p.heap_smem = 1; break; }
    }
    // >= 116 KB so that one CTA holds an SM: it allocates all 512 TMEM columns
    int64_t smem = p.nst * FT_STAGE_BYTES + (p.heap_smem ? heap_bytes : 0) + fixed;
    if (smem < 116 * 1024) smem = 116 * 1024;
    p.smem = (int)smem;
    const int64_t a_bytes = p.rt * p.nq * FT_A_BYTES;
    const int64_t b_bytes = p.it * p.nq * FT_B_BYTES;
    p.off_b = round_up(a_bytes, 1024);
    p.off_part = p.off_b + round_up(b_bytes, 1024);
    p.total = p.off_part + round_up(n_rows * p.S * k * 8, 1024);
    return p;
}

// ------------------------------------------------------------------------------------------------
// staging: X [n, dim] fp32 → three-piece bf16 operand in UMMA core-matrix blocks
// ------------------------------------------------------------------------------------------------
__global__ void factor_split_kernel(const float* __restrict__ X, int64_t n, int64_t dim, int64_t dimp, int64_t nq, int rows,
                                    int side, int64_t n_pad, __nv_bfloat16* __restrict__ out) {
    const int64_t chunks = 6 * dimp / 8;                // 8-element chunks of the split contraction per row
    const int64_t total = n_pad * chunks;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = idx / chunks, g = idx - r * chunks;
        const int64_t kk = g * 8;
        const int piece = (int)(kk / dimp);
        const int64_t d0 = kk - piece * dimp;
        // which split term of this operand each of the six contraction segments holds
        const int which = side == 0 ? (0x210100 >> (4 * piece)) & 0xF : (0x012010 >> (4 * piece)) & 0xF;
        __align__(16) __nv_bfloat16 v[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const float x = (r < n && d0 + e < dim) ? __ldg(X + r * dim + d0 + e) : 0.f;
            const __nv_bfloat16 h0 = __float2bfloat16_rn(x);
            const float r1 = x - __bfloat162float(h0);
            const __nv_bfloat16 h1 = __float2bfloat16_rn(r1);
            const __nv_bfloat16 h2 = __float2bfloat16_rn(r1 - __bfloat162float(h1));
            v[e] = which == 0 ? h0 : (which == 1 ? h1 : h2);
        }
        const int64_t tile = r / rows, rr = r - tile * rows, q = g / 8, c = g - q * 8;
        const int64_t off = (((tile * nq + q) * 8 + c) * rows + rr) * 8;
        *reinterpret_cast<uint4*>(out + off) = *reinterpret_cast<const uint4*>(v);
    }
}

// ------------------------------------------------------------------------------------------------
// per-row min-heap of 64-bit keys at h[0], h[hs], h[2 hs], ... (shared or global memory through a generic pointer)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void heap_sift_down(unsigned long long* h, int64_t hs, int n, int i, unsigned long long x) {
    while (true) {
        int c = 2 * i + 1;
        if (c >= n) break;
        unsigned long long cv = h[c * hs];
        if (c + 1 < n) {
            const unsigned long long c2 = h[(c + 1) * hs];
            if (c2 < cv) { cv = c2; ++c; }
        }
        if (cv >= x) break;
        h[i * hs] = cv;
        i = c;
    }
    h[i * hs] = x;
}
__device__ __forceinline__ void heap_make(unsigned long long* h, int64_t hs, int n) {
    for (int i = n / 2 - 1; i >= 0; --i) heap_sift_down(h, hs, n, i, h[i * hs]);
}
__device__ __forceinline__ float key_score(unsigned long long key) { return __uint_as_float(ord2f((uint32_t)(key >> 32))); }

// first position in idx[lo, hi) holding a value >= j
__device__ __forceinline__ int64_t lower_bound(const int64_t* __restrict__ idx, int64_t lo, int64_t hi, int64_t j) {
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(idx + mid) < j) lo = mid + 1; else hi = mid;
    }
    return lo;
}

struct FtArgs {
    const __nv_bfloat16* a_split;
    const __nv_bfloat16* b_split;
    const float* row_bias;
    const float* col_bias;
    const int64_t* excl_ptr;
    const int64_t* excl_idx;
    unsigned long long* part;      // [n_rows][S][k]
    int64_t n_rows, n_items, nq, it, S, tps;
    int k, nst, heap_smem;
};

__global__ void __launch_bounds__(FT_THREADS, 1) factor_topk_kernel(const FtArgs a) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const int warp = threadIdx.x >> 5;
    const int64_t rt = blockIdx.x, slice = blockIdx.y;
    const int64_t t0 = slice * a.tps;
    const int64_t t1 = min(a.it, t0 + a.tps);
    const int ntiles = (int)(t1 - t0);
    const int nq = (int)a.nq;
    const uint32_t sbase = smem_u32(smem);
    const uint32_t ring = sbase;
    unsigned long long* queue_s = reinterpret_cast<unsigned long long*>(smem + a.nst * FT_STAGE_BYTES);
    unsigned long long* heap_s = queue_s + FT_M * 16;
    const int heap_bytes = FT_QUEUE_BYTES + (a.heap_smem ? FT_M * a.k * 8 : 0);
    const uint32_t bars = sbase + a.nst * FT_STAGE_BYTES + heap_bytes;
    // barrier slots: full[nst], empty[nst], acc_full[2], acc_empty[2]; then the TMEM address slot
    const uint32_t bar_full = bars, bar_empty = bars + 8 * a.nst, bar_accf = bars + 16 * a.nst, bar_acce = bar_accf + 16;
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + a.nst * FT_STAGE_BYTES + heap_bytes + 16 * a.nst + 32);

    if (threadIdx.x == 0) {
        for (int i = 0; i < a.nst; ++i) { mbar_init(bar_full + 8 * i, 1); mbar_init(bar_empty + 8 * i, 1); }
        mbar_init(bar_accf, 1); mbar_init(bar_accf + 8, 1);
        mbar_init(bar_acce, FT_M); mbar_init(bar_acce + 8, FT_M);
        fence_barrier_init();
    }
    if (warp == FT_MMA_WARP) tmem_alloc(smem_u32((const void*)tmem_slot), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == FT_PROD_WARP) {
        // =========================== ring producer: two TMA bulk copies per stage ===========================
        if (elect_one()) {
            const uint8_t* asrc = reinterpret_cast<const uint8_t*>(a.a_split) + rt * a.nq * FT_A_BYTES;
            int stage = 0;
            uint32_t ph = 0;
            for (int g = 0; g < ntiles; ++g) {
                const uint8_t* bsrc = reinterpret_cast<const uint8_t*>(a.b_split) + (t0 + g) * a.nq * FT_B_BYTES;
                for (int q = 0; q < nq; ++q) {
                    mbar_wait(bar_empty + 8 * stage, ph ^ 1);
                    const uint32_t dst = ring + (uint32_t)(stage * FT_STAGE_BYTES);
                    mbar_expect_tx(bar_full + 8 * stage, (uint32_t)FT_STAGE_BYTES);
                    bulk_g2s(dst, asrc + (int64_t)q * FT_A_BYTES, FT_A_BYTES, bar_full + 8 * stage);
                    bulk_g2s(dst + FT_A_BYTES, bsrc + (int64_t)q * FT_B_BYTES, FT_B_BYTES, bar_full + 8 * stage);
                    if (++stage == a.nst) { stage = 0; ph ^= 1; }
                }
            }
        }
        __syncwarp();
    } else if (warp == FT_MMA_WARP) {
        // =========================== MMA issuer ===========================
        const bool leader = elect_one();
        const uint32_t idesc = umma_idesc(FT_M, FT_N);
        int stage = 0;
        uint32_t ph = 0;
        for (int g = 0; g < ntiles; ++g) {
            const int buf = g & 1;
            mbar_wait(bar_acce + 8 * buf, (uint32_t)(((g >> 1) & 1) ^ 1));     // epilogue drained this accumulator
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)(buf * FT_N);
            for (int q = 0; q < nq; ++q) {
                mbar_wait(bar_full + 8 * stage, ph);
                tc_fence_after();
                if (leader) {
                    const uint32_t sa = ring + (uint32_t)(stage * FT_STAGE_BYTES);
                    // A block [8 chunks][128 rows][16 B]: chunk stride 2048 B; B block [8][256][16 B]: chunk stride 4096 B;
                    // 8-row groups 128 B apart in both.  One K-step (16 elements) = two chunks.
                    const uint64_t ad = umma_desc(sa, FT_M * 16u, 128u);
                    const uint64_t bd = umma_desc(sa + FT_A_BYTES, FT_N * 16u, 128u);
#pragma unroll
                    for (int ks = 0; ks < FT_KC / 16; ++ks)
                        umma_bf16(d_tmem, ad + (uint64_t)(ks * 2 * FT_M), bd + (uint64_t)(ks * 2 * FT_N), idesc,
                                  (uint32_t)((q | ks) != 0));
                    umma_commit(bar_empty + 8 * stage);                          // frees the ring slot when the MMAs retire
                    if (q == nq - 1) umma_commit(bar_accf + 8 * buf);            // accumulator complete → epilogue
                }
                __syncwarp();
                if (++stage == a.nst) { stage = 0; ph ^= 1; }
            }
        }
    } else {
        // =========================== epilogue: thread t = row rt*128 + t = TMEM lane t ===========================
        const int t = threadIdx.x;
        const int64_t row = rt * FT_M + t;
        const bool valid = row < a.n_rows;
        const int k = a.k;
        const float rb = (valid && a.row_bias) ? __ldg(a.row_bias + row) : 0.f;
        // the row's exclusion list is walked forward with the ascending candidate ids: each entry is read once per slice
        int64_t ep = 0, ehi = 0, enext = INT64_MAX;
        if (valid && a.excl_ptr) {
            ehi = __ldg(a.excl_ptr + row + 1);
            ep = lower_bound(a.excl_idx, __ldg(a.excl_ptr + row), ehi, t0 * FT_N);
            if (ep < ehi) enext = __ldg(a.excl_idx + ep);
        }
        unsigned long long* part = a.part + (valid ? (row * a.S + slice) * k : 0);
        unsigned long long* hp = a.heap_smem ? heap_s + t : part;
        const int64_t hs = a.heap_smem ? FT_M : 1;
        unsigned long long* q = queue_s + t;
        int cnt = 0;
        unsigned long long root = 0ull;                     // the heap's smallest key once cnt == k
        float thr = valid ? -INFINITY : INFINITY;          // rows past n_rows take nothing
        const uint32_t lane_base = tmem_base + ((uint32_t)(warp * 32) << 16);
        for (int g = 0; g < ntiles; ++g) {
            const int buf = g & 1;
            mbar_wait(bar_accf + 8 * buf, (uint32_t)((g >> 1) & 1));
            tc_fence_after();
            const int64_t jt = (t0 + g) * FT_N;
            for (int ch = 0; ch < FT_N / 16; ++ch) {
                uint32_t v[16];
                tmem_ld16(lane_base + (uint32_t)(buf * FT_N + ch * 16), v);
                tmem_ld_wait();
                if (ch == FT_N / 16 - 1) {                 // the whole tile is read: release the accumulator
                    tc_fence_before();
                    mbar_arrive(bar_acce + 8 * buf);
                }
                const int64_t j0 = jt + ch * 16;
                // Pass 1: queue the chunk's candidates (a predicated store, no branch).  Handling a candidate on the spot
                // would serialise the warp once per column in which ANY of its 32 rows has one; draining the queues after
                // the chunk costs the longest queue of the warp instead.
                int nc = 0;
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const int64_t j = j0 + i;
                    const bool in = j < a.n_items;
                    float s = __uint_as_float(v[i]);
                    if (a.col_bias) s += in ? __ldg(a.col_bias + j) : 0.f;
                    s += rb;
                    s = s == 0.f ? 0.f : s;                      // -0 and +0 tie: one key, so the item id decides
                    const unsigned long long key =
                        ((unsigned long long)f2ord(__float_as_uint(s)) << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)j);
                    if (s > thr && in) q[(nc++) * FT_M] = key;
                }
                // Pass 2: in id order, against the threshold as it rises (a key compare: a later id that ties loses)
                for (int c = 0; c < nc; ++c) {
                    const unsigned long long key = q[c * FT_M];
                    if (cnt == k && key <= root) continue;
                    const int64_t j = (int64_t)(0xFFFFFFFFu - (uint32_t)key);
                    while (enext < j) enext = ++ep < ehi ? __ldg(a.excl_idx + ep) : INT64_MAX;
                    if (enext == j) continue;
                    if (cnt < k) {
                        hp[cnt * hs] = key;
                        if (++cnt < k) continue;
                        heap_make(hp, hs, k);
                    } else {
                        heap_sift_down(hp, hs, k, 0, key);
                    }
                    root = hp[0];
                    thr = key_score(root);
                }
            }
        }
        if (valid) {
            // heapsort: the min-heap leaves the keys in descending order
            if (cnt < k) heap_make(hp, hs, cnt);
            for (int end = cnt - 1; end > 0; --end) {
                const unsigned long long x = hp[end * hs];
                hp[end * hs] = hp[0];
                heap_sift_down(hp, hs, end, 0, x);
            }
            for (int i = 0; i < k; ++i) {
                const unsigned long long key = i < cnt ? hp[i * hs] : 0ull;
                if (a.heap_smem || i >= cnt) part[i] = key;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == FT_MMA_WARP) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// one thread per row: merge the S descending key lists of the row into the final k
__global__ void factor_topk_merge_kernel(const unsigned long long* __restrict__ part, int64_t n_rows, int S, int k,
                                         float* __restrict__ out_scores, int64_t* __restrict__ out_items) {
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n_rows) return;
    const unsigned long long* base = part + row * S * k;
    int pos[FT_MAX_SLICES];
    for (int s = 0; s < S; ++s) pos[s] = 0;
    for (int o = 0; o < k; ++o) {
        unsigned long long best = 0ull;
        int bs = -1;
        for (int s = 0; s < S; ++s) {
            if (pos[s] < k) {
                const unsigned long long v = __ldg(base + s * k + pos[s]);
                if (v > best) { best = v; bs = s; }
            }
        }
        if (bs >= 0) ++pos[bs];
        out_scores[row * k + o] = best ? key_score(best) : -INFINITY;
        out_items[row * k + o] = best ? (int64_t)(0xFFFFFFFFu - (uint32_t)(best & 0xFFFFFFFFull)) : -1;
    }
}

}  // namespace rbr

using namespace rbr;

extern "C" int64_t rbr_factor_topk_workspace_bytes(int64_t n_rows, int64_t n_items, int64_t dim, int64_t k) {
    if (!ft_supported(n_rows, n_items, dim, k)) {
        set_error("rbr_factor_topk: need 1 <= k <= %d, 1 <= dim <= %d, 1 <= n_items < 2^31 (got k=%lld dim=%lld n_items=%lld)",
                  FT_MAX_K, FT_MAX_DIM, (long long)k, (long long)dim, (long long)n_items);
        return RBR_EUNSUPPORTED;
    }
    return ft_plan(n_rows, n_items, dim, k, ft_sm_count()).total;
}

extern "C" int64_t rbr_factor_topk_slices(int64_t n_rows, int64_t n_items, int64_t dim, int64_t k) {
    if (!ft_supported(n_rows, n_items, dim, k)) {
        set_error("rbr_factor_topk_slices: shape outside the supported limits");
        return RBR_EUNSUPPORTED;
    }
    return ft_plan(n_rows, n_items, dim, k, ft_sm_count()).S;
}

extern "C" int rbr_factor_topk(const float* A, const float* row_bias, int64_t n_rows, const float* B, const float* col_bias,
                               int64_t n_items, int64_t dim, const int64_t* excl_ptr, const int64_t* excl_idx, int64_t k,
                               float* out_scores, int64_t* out_items, void* ws, int64_t ws_bytes, void* stream) {
    RBR_REQUIRE(ft_supported(n_rows, n_items, dim, k), RBR_EUNSUPPORTED,
                "rbr_factor_topk: need 1 <= k <= %d, 1 <= dim <= %d, 1 <= n_items < 2^31 (got k=%lld dim=%lld n_items=%lld)",
                FT_MAX_K, FT_MAX_DIM, (long long)k, (long long)dim, (long long)n_items);
    RBR_REQUIRE((excl_ptr == nullptr) == (excl_idx == nullptr), RBR_EINVAL,
                "rbr_factor_topk: excl_ptr and excl_idx must both be set or both be NULL");
    if (n_rows == 0) return RBR_OK;
    RBR_REQUIRE(A && B && out_scores && out_items && ws, RBR_EINVAL, "rbr_factor_topk: null pointer");
    const FtPlan p = ft_plan(n_rows, n_items, dim, k, ft_sm_count());
    RBR_REQUIRE(ws_bytes >= p.total, RBR_EWORKSPACE, "rbr_factor_topk: workspace %lld < %lld bytes", (long long)ws_bytes,
                (long long)p.total);
    cudaStream_t s = as_stream(stream);
    uint8_t* w = reinterpret_cast<uint8_t*>(ws);
    __nv_bfloat16* asp = reinterpret_cast<__nv_bfloat16*>(w);
    __nv_bfloat16* bsp = reinterpret_cast<__nv_bfloat16*>(w + p.off_b);
    unsigned long long* part = reinterpret_cast<unsigned long long*>(w + p.off_part);

    const int64_t a_chunks = p.rt * FT_M * (6 * p.dimp / 8), b_chunks = p.it * FT_N * (6 * p.dimp / 8);
    factor_split_kernel<<<(unsigned)std::min<int64_t>((a_chunks + 255) / 256, 65535), 256, 0, s>>>(
        A, n_rows, dim, p.dimp, p.nq, FT_M, 0, p.rt * FT_M, asp);
    RBR_LAUNCH_CHECK("factor_split_kernel(A)");
    factor_split_kernel<<<(unsigned)std::min<int64_t>((b_chunks + 255) / 256, 65535), 256, 0, s>>>(
        B, n_items, dim, p.dimp, p.nq, FT_N, 1, p.it * FT_N, bsp);
    RBR_LAUNCH_CHECK("factor_split_kernel(B)");

    RBR_CUDA(cudaFuncSetAttribute(factor_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, p.smem));
    FtArgs a;
    a.a_split = asp; a.b_split = bsp; a.row_bias = row_bias; a.col_bias = col_bias;
    a.excl_ptr = excl_ptr; a.excl_idx = excl_idx; a.part = part;
    a.n_rows = n_rows; a.n_items = n_items; a.nq = p.nq; a.it = p.it; a.S = p.S; a.tps = p.tps;
    a.k = (int)k; a.nst = p.nst; a.heap_smem = p.heap_smem;
    factor_topk_kernel<<<dim3((unsigned)p.rt, (unsigned)p.S), FT_THREADS, p.smem, s>>>(a);
    RBR_LAUNCH_CHECK("factor_topk_kernel");
    factor_topk_merge_kernel<<<(unsigned)((n_rows + 127) / 128), 128, 0, s>>>(part, n_rows, (int)p.S, (int)k, out_scores, out_items);
    RBR_LAUNCH_CHECK("factor_topk_merge_kernel");
    return RBR_OK;
}
