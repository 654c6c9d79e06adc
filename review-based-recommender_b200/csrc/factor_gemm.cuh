// factor_gemm.cuh — the score GEMM shared by K10 (topk.cu) and K11 (rank.cu):
//   score[r, i] = <A[r], B[i]> + row_bias[r] + col_bias[i]
// on a three-piece bf16 split of both operands (see topk.cu for the precision argument), tcgen05 M = 128, N = 256, two TMEM
// accumulators.  Both kernels run the same staging kernel, the same ring producer and MMA issuer and the same score-to-key
// code, so a score one of them sees is bit-identical to the score the other sees for the same (row, item).
#pragma once

#include <math.h>

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
constexpr int FT_MAX_DIM = 512;

// The operand half of a launch plan: split-operand geometry and workspace offsets of A' and B'.
struct FtGemm {
    int64_t dimp;       // dim rounded up to 32 (6 * dimp is a whole number of 64-element chunks)
    int64_t nq;         // ring stages per item tile = 6 * dimp / 64
    int64_t rt, it;     // row tiles, item tiles
    int64_t off_b;      // workspace offset of B' (A' starts at 0)
    int64_t end;        // first byte past B' (1024-aligned)
};

inline FtGemm ft_gemm_plan(int64_t n_rows, int64_t n_items, int64_t dim) {
    FtGemm g;
    g.dimp = round_up(dim, 32);
    g.nq = 6 * g.dimp / FT_KC;
    g.rt = (n_rows + FT_M - 1) / FT_M;
    g.it = (n_items + FT_N - 1) / FT_N;
    g.off_b = round_up(g.rt * g.nq * FT_A_BYTES, 1024);
    g.end = g.off_b + round_up(g.it * g.nq * FT_B_BYTES, 1024);
    return g;
}

inline int ft_sm_count() {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
        n <= 0) {
        cudaGetLastError();
        return 148;                                     // B200
    }
    return n;
}

// Item slices: the CTA's cost is roughly its item tiles plus `fill` tiles per slice (the per-slice fixed work); the grid
// runs in waves of one CTA per SM.  Take the slice count with the fewest wave-weighted tiles, among those whose per-slice
// buffers (part_bytes_per_slice each) stay under part_cap.
inline int64_t ft_choose_slices(const FtGemm& g, int sms, double fill, int64_t part_bytes_per_slice, int64_t part_cap) {
    int64_t best = 1;
    double best_cost = 1e300;
    const int64_t smax = g.it < FT_MAX_SLICES ? g.it : FT_MAX_SLICES;
    for (int64_t s = 1; s <= smax; ++s) {
        if (s > 1 && s * part_bytes_per_slice > part_cap) break;
        const int64_t tps = (g.it + s - 1) / s;
        if ((g.it + tps - 1) / tps != s) continue;     // every slice must own at least one tile
        const int64_t waves = (g.rt * s + sms - 1) / sms;
        const double cost = (double)waves * ((double)tps + fill);
        if (cost < best_cost * 0.97) { best_cost = cost; best = s; }
    }
    return best;
}

// Stages A [n_rows, dim] and B [n_items, dim] into A' (workspace offset 0) and B' (offset g.off_b): topk.cu.
int ft_stage(const float* A, int64_t n_rows, const float* B, int64_t n_items, int64_t dim, const FtGemm& g, uint8_t* ws,
             cudaStream_t s);

// first position in idx[lo, hi) holding a value >= j
__device__ __forceinline__ int64_t lower_bound(const int64_t* __restrict__ idx, int64_t lo, int64_t hi, int64_t j) {
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(idx + mid) < j) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// The score of (row, item j) from its raw fp32 accumulator bits, with the biases added in this order, and -0 folded into +0:
// -0 and +0 tie, so they must form one key and let the item id decide.
__device__ __forceinline__ float ft_score(uint32_t acc, const float* __restrict__ col_bias, int64_t j, bool in, float rb) {
    float s = __uint_as_float(acc);
    if (col_bias) s += in ? __ldg(col_bias + j) : 0.f;
    s += rb;
    return s == 0.f ? 0.f : s;
}
// 64-bit key: order-preserving score bits << 32 | ~item.  One unsigned compare orders by (score desc, item asc).
__device__ __forceinline__ unsigned long long ft_key(float s, int64_t j) {
    return ((unsigned long long)f2ord(__float_as_uint(s)) << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)j);
}
__device__ __forceinline__ float key_score(unsigned long long key) { return __uint_as_float(ord2f((uint32_t)(key >> 32))); }
__device__ __forceinline__ int64_t key_item(unsigned long long key) { return (int64_t)(0xFFFFFFFFu - (uint32_t)key); }

// Shared-memory barriers of the ring (full[nst], empty[nst]) and the accumulators (acc_full[2], acc_empty[2]) at `bars`.
struct FtBars {
    uint32_t full, empty, accf, acce;
};
__device__ __forceinline__ FtBars ft_bars(uint32_t bars, int nst) {
    FtBars b;
    b.full = bars; b.empty = bars + 8 * nst; b.accf = bars + 16 * nst; b.acce = b.accf + 16;
    return b;
}
// Initialises the barriers and allocates all 512 TMEM columns; every thread of the CTA calls it.  Returns the TMEM base.
__device__ __forceinline__ uint32_t ft_setup(const FtBars& b, int nst, volatile uint32_t* tmem_slot) {
    const int warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        for (int i = 0; i < nst; ++i) { mbar_init(b.full + 8 * i, 1); mbar_init(b.empty + 8 * i, 1); }
        mbar_init(b.accf, 1); mbar_init(b.accf + 8, 1);
        mbar_init(b.acce, FT_M); mbar_init(b.acce + 8, FT_M);
        fence_barrier_init();
    }
    if (warp == FT_MMA_WARP) tmem_alloc(smem_u32((const void*)tmem_slot), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    return *tmem_slot;
}
__device__ __forceinline__ void ft_teardown(uint32_t tmem_base) {
    tc_fence_before();
    __syncthreads();
    if ((threadIdx.x >> 5) == FT_MMA_WARP) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// Ring producer (warp FT_PROD_WARP): two TMA bulk copies per stage, for item tiles t0 .. t0 + ntiles - 1 of row tile rt.
__device__ __forceinline__ void ft_produce(const __nv_bfloat16* a_split, const __nv_bfloat16* b_split, int64_t rt, int64_t t0,
                                           int ntiles, int nq, int nst, uint32_t ring, const FtBars& b) {
    if (elect_one()) {
        const uint8_t* asrc = reinterpret_cast<const uint8_t*>(a_split) + rt * nq * FT_A_BYTES;
        int stage = 0;
        uint32_t ph = 0;
        for (int g = 0; g < ntiles; ++g) {
            const uint8_t* bsrc = reinterpret_cast<const uint8_t*>(b_split) + (t0 + g) * nq * FT_B_BYTES;
            for (int q = 0; q < nq; ++q) {
                mbar_wait(b.empty + 8 * stage, ph ^ 1);
                const uint32_t dst = ring + (uint32_t)(stage * FT_STAGE_BYTES);
                mbar_expect_tx(b.full + 8 * stage, (uint32_t)FT_STAGE_BYTES);
                bulk_g2s(dst, asrc + (int64_t)q * FT_A_BYTES, FT_A_BYTES, b.full + 8 * stage);
                bulk_g2s(dst + FT_A_BYTES, bsrc + (int64_t)q * FT_B_BYTES, FT_B_BYTES, b.full + 8 * stage);
                if (++stage == nst) { stage = 0; ph ^= 1; }
            }
        }
    }
    __syncwarp();
}

// MMA issuer (warp FT_MMA_WARP): item tile g accumulates into TMEM columns (g & 1) * 256 .. + 255.
__device__ __forceinline__ void ft_mma(int ntiles, int nq, int nst, uint32_t ring, const FtBars& b, uint32_t tmem_base) {
    const bool leader = elect_one();
    const uint32_t idesc = umma_idesc(FT_M, FT_N);
    int stage = 0;
    uint32_t ph = 0;
    for (int g = 0; g < ntiles; ++g) {
        const int buf = g & 1;
        mbar_wait(b.acce + 8 * buf, (uint32_t)(((g >> 1) & 1) ^ 1));       // epilogue drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(buf * FT_N);
        for (int q = 0; q < nq; ++q) {
            mbar_wait(b.full + 8 * stage, ph);
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
                umma_commit(b.empty + 8 * stage);                            // frees the ring slot when the MMAs retire
                if (q == nq - 1) umma_commit(b.accf + 8 * buf);              // accumulator complete → epilogue
            }
            __syncwarp();
            if (++stage == nst) { stage = 0; ph ^= 1; }
        }
    }
}

}  // namespace rbr
