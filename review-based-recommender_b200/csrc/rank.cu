// rank.cu — K11: exact full-catalogue rank of listed target items under a factorised score
//   score[r, i] = <A[r], B[i]> + row_bias[r] + col_bias[i],
// without materialising the n_rows x n_items scores.  sm_100a only.
//
// rank(r, t) = #{ eligible i : key(r, i) >= key(r, t) } with K10's key (score descending, then item id ascending), so the
// rank is the 1-based position t would take in K10's output for k = infinity.  Eligible = not in the row's exclusion list;
// NaN and -inf scores never count.  Both scans below use K10's staging kernel, ring producer, MMA issuer and score-to-key
// code (factor_gemm.cuh), so every score is bit-identical to the one K10 sees for the same (row, item).
//
// Capture scan (factor_rank_capture_kernel): one CTA per (128-row tile, item slice).  Thread t owns row t and walks the
// row's ascending target list forward with the column index, like K10's exclusion walk; each target's 64-bit key is written
// to the workspace (every target lies in exactly one slice).
//
// Count scan (factor_rank_count_kernel): same grid.  Thread t loads its row's target keys (at most max_targets), drops those
// whose score is NaN or -inf (rank -1), and sorts the rest descending in shared memory.  Every score whose key is >= the
// lowest target key, is not NaN / -inf and is not excluded (the exclusion list is walked forward as in K10) falls into bin
// b = #{target keys > key}: it counts toward the targets at sorted positions b .. m-1.  For one target per row that is a
// single compare.  After the scan the prefix sums of the bins are the slice's counts per target; they are added to the
// target's counter with integer atomics, so the result does not depend on the slice count or the order of the CTAs.
//
// Finish (factor_rank_finish_kernel): counter → int64 rank (-1 for NaN / -inf targets), key → fp32 score.
#include <math.h>

#include <algorithm>

#include "factor_gemm.cuh"

namespace rbr {

constexpr int FR_MAX_TARGETS = 64;                     // targets per row in one call (the caller splits longer rows)

struct FrPlan {
    FtGemm g;           // split operands: A' | B' at the start of the workspace
    int64_t S, tps;     // item slices, item tiles per slice
    int nst_cap, smem_cap;     // capture scan: ring stages, dynamic shared memory bytes
    int nst_cnt, smem_cnt;     // count scan
    int64_t off_key, off_acc, total;   // workspace: A' | B' | target keys [n_targets] | target counters [n_targets]
};

static bool fr_supported(int64_t n_rows, int64_t n_items, int64_t dim, int64_t n_targets, int64_t max_targets) {
    return n_rows >= 0 && n_items >= 1 && n_items < (1ll << 31) && dim >= 1 && dim <= FT_MAX_DIM && n_targets >= 0 &&
           max_targets >= 1 && max_targets <= FR_MAX_TARGETS;
}

static FrPlan fr_plan(int64_t n_rows, int64_t n_items, int64_t dim, int64_t n_targets, int64_t max_targets, int sms) {
    FrPlan p;
    p.g = ft_gemm_plan(n_rows, n_items, dim);
    // per slice: sorting the target keys, the prefix sums and the counter atomics — about one item tile's worth
    p.S = ft_choose_slices(p.g, sms, 1.0, 0, 0);
    p.tps = (p.g.it + p.S - 1) / p.S;
    const int64_t fixed = 1024;                                         // barriers + TMEM slot
    const int64_t tgt_bytes = (int64_t)FT_M * max_targets * (8 + 4);    // sorted target keys + bins, per row
    p.nst_cap = 4;
    p.nst_cnt = 2;
    for (int nst = 4; nst >= 2; --nst)
        if (nst * FT_STAGE_BYTES + tgt_bytes + fixed <= FT_SMEM_MAX) { p.nst_cnt = nst; break; }
    // >= 116 KB so that one CTA holds an SM: it allocates all 512 TMEM columns
    p.smem_cap = (int)std::max<int64_t>(p.nst_cap * FT_STAGE_BYTES + fixed, 116 * 1024);
    p.smem_cnt = (int)std::max<int64_t>(p.nst_cnt * FT_STAGE_BYTES + tgt_bytes + fixed, 116 * 1024);
    p.off_key = p.g.end;
    p.off_acc = p.off_key + round_up(n_targets * 8, 1024);
    p.total = p.off_acc + round_up(n_targets * 4, 1024);
    return p;
}

struct FrArgs {
    const __nv_bfloat16* a_split;
    const __nv_bfloat16* b_split;
    const float* row_bias;
    const float* col_bias;
    const int64_t* excl_ptr;
    const int64_t* excl_idx;
    const int64_t* tgt_ptr;
    const int64_t* tgt_idx;
    unsigned long long* tkey;      // [n_targets] keys from the capture scan
    unsigned int* acc;             // [n_targets] counts, summed over slices
    int64_t n_rows, n_items, nq, it, tps;
    int mt, nst;
};

// #{ j < m : tk[j] > key } for tk sorted descending (stride FT_M); top = the largest power of two <= m
__device__ __forceinline__ int fr_above(const unsigned long long* tk, int m, int top, unsigned long long key) {
    int b = 0;
    for (int st = top; st > 0; st >>= 1)
        if (b + st <= m && tk[(b + st - 1) * FT_M] > key) b += st;
    return b;
}

template <bool COUNT>
__device__ __forceinline__ void factor_rank_body(const FrArgs& a) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const int warp = threadIdx.x >> 5;
    const int64_t rt = blockIdx.x, slice = blockIdx.y;
    const int64_t t0 = slice * a.tps;
    const int64_t t1 = min(a.it, t0 + a.tps);
    const int ntiles = (int)(t1 - t0);
    const int nq = (int)a.nq;
    const uint32_t sbase = smem_u32(smem);
    const uint32_t ring = sbase;
    unsigned long long* keys_s = reinterpret_cast<unsigned long long*>(smem + a.nst * FT_STAGE_BYTES);
    unsigned int* bins_s = reinterpret_cast<unsigned int*>(keys_s + (COUNT ? FT_M * a.mt : 0));
    const int tgt_bytes = COUNT ? FT_M * a.mt * (8 + 4) : 0;
    const FtBars bar = ft_bars(sbase + a.nst * FT_STAGE_BYTES + tgt_bytes, a.nst);
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + a.nst * FT_STAGE_BYTES + tgt_bytes + 16 * a.nst + 32);
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
        const float rb = (valid && a.row_bias) ? __ldg(a.row_bias + row) : 0.f;
        // capture: the row's target list from the slice's first id on; count: its exclusion list.  Both walk forward with
        // the ascending column index, so each entry is read once per slice.
        int64_t lp = 0, lhi = 0, lnext = INT64_MAX;
        const int64_t* lidx = COUNT ? a.excl_idx : a.tgt_idx;
        const int64_t* lptr = COUNT ? a.excl_ptr : a.tgt_ptr;
        if (valid && lptr) {
            lhi = __ldg(lptr + row + 1);
            lp = lower_bound(lidx, __ldg(lptr + row), lhi, t0 * FT_N);
            if (lp < lhi) lnext = __ldg(lidx + lp);
        }
        unsigned long long* tk = keys_s + t;
        unsigned int* bins = bins_s + t;
        int m = 0, top = 0;
        int64_t g0 = 0, g1 = 0;                           // the row's targets handled by this call
        unsigned long long lowest = ~0ull;                // no real score reaches it: f2ord(x) = 0xFFFFFFFF only for a NaN
        if (COUNT && valid) {
            g0 = __ldg(a.tgt_ptr + row);
            g1 = min(__ldg(a.tgt_ptr + row + 1), g0 + a.mt);
            for (int64_t p = g0; p < g1; ++p) {           // insertion sort, descending; NaN / -inf targets are left out
                const unsigned long long key = a.tkey[p];
                if (!(key_score(key) > -INFINITY)) continue;
                int q = m++;
                for (; q > 0 && tk[(q - 1) * FT_M] < key; --q) tk[q * FT_M] = tk[(q - 1) * FT_M];
                tk[q * FT_M] = key;
            }
            for (int p = 0; p < m; ++p) bins[p * FT_M] = 0u;
            if (m) lowest = tk[(m - 1) * FT_M];
            top = m ? 1 << (31 - __clz(m)) : 0;
        }
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
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const int64_t j = j0 + i;
                    const bool in = j < a.n_items;
                    const float s = ft_score(v[i], a.col_bias, j, in, rb);
                    const unsigned long long key = ft_key(s, j);
                    const bool listed = j == lnext;
                    if (listed) lnext = ++lp < lhi ? __ldg(lidx + lp) : INT64_MAX;
                    if (COUNT) {
                        if (in && !listed && s > -INFINITY && key >= lowest) ++bins[fr_above(tk, m, top, key) * FT_M];
                    } else if (listed && in) {
                        a.tkey[lp - 1] = key;
                    }
                }
            }
        }
        if (COUNT && m) {
            unsigned int c = 0;
            for (int p = 0; p < m; ++p) { c += bins[p * FT_M]; bins[p * FT_M] = c; }
            for (int64_t p = g0; p < g1; ++p) {
                const unsigned long long key = a.tkey[p];
                if (!(key_score(key) > -INFINITY)) continue;
                const unsigned int n = bins[fr_above(tk, m, top, key) * FT_M];
                if (n) atomicAdd(a.acc + p, n);
            }
        }
    }
    ft_teardown(tmem_base);
}

__global__ void __launch_bounds__(FT_THREADS, 1) factor_rank_capture_kernel(const FrArgs a) { factor_rank_body<false>(a); }
__global__ void __launch_bounds__(FT_THREADS, 1) factor_rank_count_kernel(const FrArgs a) { factor_rank_body<true>(a); }

__global__ void factor_rank_finish_kernel(const unsigned long long* __restrict__ tkey, const unsigned int* __restrict__ acc,
                                          int64_t n, int64_t* __restrict__ out_ranks, float* __restrict__ out_scores) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float s = key_score(__ldg(tkey + i));
    const unsigned int c = __ldg(acc + i);
    out_scores[i] = s;
    out_ranks[i] = (s > -INFINITY && c > 0) ? (int64_t)c : -1;
}

}  // namespace rbr

using namespace rbr;

extern "C" int64_t rbr_factor_rank_workspace_bytes(int64_t n_rows, int64_t n_items, int64_t dim, int64_t n_targets,
                                                   int64_t max_targets) {
    if (!fr_supported(n_rows, n_items, dim, n_targets, max_targets)) {
        set_error("rbr_factor_rank: need 1 <= dim <= %d, 1 <= n_items < 2^31, 1 <= max_targets <= %d (got dim=%lld "
                  "n_items=%lld max_targets=%lld)", FT_MAX_DIM, FR_MAX_TARGETS, (long long)dim, (long long)n_items,
                  (long long)max_targets);
        return RBR_EUNSUPPORTED;
    }
    return fr_plan(n_rows, n_items, dim, n_targets, max_targets, ft_sm_count()).total;
}

extern "C" int rbr_factor_rank(const float* A, const float* row_bias, int64_t n_rows, const float* B, const float* col_bias,
                               int64_t n_items, int64_t dim, const int64_t* excl_ptr, const int64_t* excl_idx,
                               const int64_t* tgt_ptr, const int64_t* tgt_idx, int64_t n_targets, int64_t max_targets,
                               int64_t* out_ranks, float* out_scores, void* ws, int64_t ws_bytes, void* stream) {
    RBR_REQUIRE(fr_supported(n_rows, n_items, dim, n_targets, max_targets), RBR_EUNSUPPORTED,
                "rbr_factor_rank: need 1 <= dim <= %d, 1 <= n_items < 2^31, 1 <= max_targets <= %d (got dim=%lld "
                "n_items=%lld max_targets=%lld)", FT_MAX_DIM, FR_MAX_TARGETS, (long long)dim, (long long)n_items,
                (long long)max_targets);
    RBR_REQUIRE((excl_ptr == nullptr) == (excl_idx == nullptr), RBR_EINVAL,
                "rbr_factor_rank: excl_ptr and excl_idx must both be set or both be NULL");
    if (n_rows == 0 || n_targets == 0) return RBR_OK;
    RBR_REQUIRE(A && B && tgt_ptr && tgt_idx && out_ranks && out_scores && ws, RBR_EINVAL, "rbr_factor_rank: null pointer");
    const FrPlan p = fr_plan(n_rows, n_items, dim, n_targets, max_targets, ft_sm_count());
    RBR_REQUIRE(ws_bytes >= p.total, RBR_EWORKSPACE, "rbr_factor_rank: workspace %lld < %lld bytes", (long long)ws_bytes,
                (long long)p.total);
    cudaStream_t s = as_stream(stream);
    uint8_t* w = reinterpret_cast<uint8_t*>(ws);
    const int rc = ft_stage(A, n_rows, B, n_items, dim, p.g, w, s);
    if (rc != RBR_OK) return rc;
    RBR_CUDA(cudaMemsetAsync(w + p.off_key, 0, (size_t)(p.total - p.off_key), s));

    FrArgs a;
    a.a_split = reinterpret_cast<const __nv_bfloat16*>(w);
    a.b_split = reinterpret_cast<const __nv_bfloat16*>(w + p.g.off_b);
    a.row_bias = row_bias; a.col_bias = col_bias;
    a.excl_ptr = excl_ptr; a.excl_idx = excl_idx; a.tgt_ptr = tgt_ptr; a.tgt_idx = tgt_idx;
    a.tkey = reinterpret_cast<unsigned long long*>(w + p.off_key);
    a.acc = reinterpret_cast<unsigned int*>(w + p.off_acc);
    a.n_rows = n_rows; a.n_items = n_items; a.nq = p.g.nq; a.it = p.g.it; a.tps = p.tps;
    a.mt = (int)max_targets;
    const dim3 grid((unsigned)p.g.rt, (unsigned)p.S);
    a.nst = p.nst_cap;
    RBR_CUDA(cudaFuncSetAttribute(factor_rank_capture_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, p.smem_cap));
    factor_rank_capture_kernel<<<grid, FT_THREADS, p.smem_cap, s>>>(a);
    RBR_LAUNCH_CHECK("factor_rank_capture_kernel");
    a.nst = p.nst_cnt;
    RBR_CUDA(cudaFuncSetAttribute(factor_rank_count_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, p.smem_cnt));
    factor_rank_count_kernel<<<grid, FT_THREADS, p.smem_cnt, s>>>(a);
    RBR_LAUNCH_CHECK("factor_rank_count_kernel");
    factor_rank_finish_kernel<<<(unsigned)((n_targets + 255) / 256), 256, 0, s>>>(a.tkey, a.acc, n_targets, out_ranks, out_scores);
    RBR_LAUNCH_CHECK("factor_rank_finish_kernel");
    return RBR_OK;
}
