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

#include "factor_gemm.cuh"

namespace rbr {

constexpr int FT_QUEUE_BYTES = FT_M * 16 * 8;          // per row: the candidate keys of one 16-column chunk
constexpr int64_t FT_PART_CAP = 96ll << 20;            // cap on the per-slice partial lists when choosing several slices
constexpr int FT_MAX_K = 256;

struct FtPlan {
    FtGemm g;           // split operands: A' | B' at the start of the workspace
    int64_t S, tps;     // item slices, item tiles per slice
    int nst;            // ring stages
    int heap_smem;      // 1: per-row heaps in shared memory
    int smem;           // dynamic shared memory bytes
    int64_t off_part, total;   // workspace: A' | B' | partial top-k keys [n_rows][S][k]
};

static bool ft_supported(int64_t n_rows, int64_t n_items, int64_t dim, int64_t k) {
    return n_rows >= 0 && n_items >= 1 && n_items < (1ll << 31) && dim >= 1 && dim <= FT_MAX_DIM && k >= 1 && k <= FT_MAX_K;
}

static FtPlan ft_plan(int64_t n_rows, int64_t n_items, int64_t dim, int64_t k, int sms) {
    FtPlan p;
    p.g = ft_gemm_plan(n_rows, n_items, dim);
    // The per-slice share, in tiles (filling, sorting and writing the heaps, and the threshold starting over), was fitted
    // to timings at 20 000 x 12 000 on a B200 (k = 10: 3 slices best, k = 100: 1-2).
    p.S = ft_choose_slices(p.g, sms, 3.0 + (double)k / 16.0, n_rows * k * 8, FT_PART_CAP);
    p.tps = (p.g.it + p.S - 1) / p.S;
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
    p.off_part = p.g.end;
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
    // barrier slots: full[nst], empty[nst], acc_full[2], acc_empty[2]; then the TMEM address slot
    const FtBars bar = ft_bars(sbase + a.nst * FT_STAGE_BYTES + heap_bytes, a.nst);
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + a.nst * FT_STAGE_BYTES + heap_bytes + 16 * a.nst + 32);
    const uint32_t tmem_base = ft_setup(bar, a.nst, tmem_slot);

    if (warp == FT_PROD_WARP) {
        ft_produce(a.a_split, a.b_split, rt, t0, ntiles, nq, a.nst, ring, bar);
    } else if (warp == FT_MMA_WARP) {
        ft_mma(ntiles, nq, a.nst, ring, bar, tmem_base);
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
            mbar_wait(bar.accf + 8 * buf, (uint32_t)((g >> 1) & 1));
            tc_fence_after();
            const int64_t jt = (t0 + g) * FT_N;
            for (int ch = 0; ch < FT_N / 16; ++ch) {
                uint32_t v[16];
                tmem_ld16(lane_base + (uint32_t)(buf * FT_N + ch * 16), v);
                tmem_ld_wait();
                if (ch == FT_N / 16 - 1) {                 // the whole tile is read: release the accumulator
                    tc_fence_before();
                    mbar_arrive(bar.acce + 8 * buf);
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
                    const float s = ft_score(v[i], a.col_bias, j, in, rb);
                    const unsigned long long key = ft_key(s, j);
                    if (s > thr && in) q[(nc++) * FT_M] = key;
                }
                // Pass 2: in id order, against the threshold as it rises (a key compare: a later id that ties loses)
                for (int c = 0; c < nc; ++c) {
                    const unsigned long long key = q[c * FT_M];
                    if (cnt == k && key <= root) continue;
                    const int64_t j = key_item(key);
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
    ft_teardown(tmem_base);
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
        out_items[row * k + o] = best ? key_item(best) : -1;
    }
}

int ft_stage(const float* A, int64_t n_rows, const float* B, int64_t n_items, int64_t dim, const FtGemm& g, uint8_t* ws,
             cudaStream_t s) {
    const int64_t a_chunks = g.rt * FT_M * (6 * g.dimp / 8), b_chunks = g.it * FT_N * (6 * g.dimp / 8);
    factor_split_kernel<<<(unsigned)std::min<int64_t>((a_chunks + 255) / 256, 65535), 256, 0, s>>>(
        A, n_rows, dim, g.dimp, g.nq, FT_M, 0, g.rt * FT_M, reinterpret_cast<__nv_bfloat16*>(ws));
    RBR_LAUNCH_CHECK("factor_split_kernel(A)");
    factor_split_kernel<<<(unsigned)std::min<int64_t>((b_chunks + 255) / 256, 65535), 256, 0, s>>>(
        B, n_items, dim, g.dimp, g.nq, FT_N, 1, g.it * FT_N, reinterpret_cast<__nv_bfloat16*>(ws + g.off_b));
    RBR_LAUNCH_CHECK("factor_split_kernel(B)");
    return RBR_OK;
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
    __nv_bfloat16* bsp = reinterpret_cast<__nv_bfloat16*>(w + p.g.off_b);
    unsigned long long* part = reinterpret_cast<unsigned long long*>(w + p.off_part);

    const int rc = ft_stage(A, n_rows, B, n_items, dim, p.g, w, s);
    if (rc != RBR_OK) return rc;

    RBR_CUDA(cudaFuncSetAttribute(factor_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, p.smem));
    FtArgs a;
    a.a_split = asp; a.b_split = bsp; a.row_bias = row_bias; a.col_bias = col_bias;
    a.excl_ptr = excl_ptr; a.excl_idx = excl_idx; a.part = part;
    a.n_rows = n_rows; a.n_items = n_items; a.nq = p.g.nq; a.it = p.g.it; a.S = p.S; a.tps = p.tps;
    a.k = (int)k; a.nst = p.nst; a.heap_smem = p.heap_smem;
    factor_topk_kernel<<<dim3((unsigned)p.g.rt, (unsigned)p.S), FT_THREADS, p.smem, s>>>(a);
    RBR_LAUNCH_CHECK("factor_topk_kernel");
    factor_topk_merge_kernel<<<(unsigned)((n_rows + 127) / 128), 128, 0, s>>>(part, n_rows, (int)p.S, (int)k, out_scores, out_items);
    RBR_LAUNCH_CHECK("factor_topk_merge_kernel");
    return RBR_OK;
}
