// conv_bwd_tc.cu — K2c: backward of the fused conv → activation → max-over-time encoder as two tensor-core GEMMs over a
// token × filter-tap COEFFICIENT MATRIX.  sm_100a only (tcgen05 / TMEM / TMA).
//
// Replaces what autograd runs for the reverse of NgramFeat.forward (reference models/deepconn/layers.py:123-136) and of the
// embedding lookup (layers.py:23): max_pool1d backward, relu backward, aten::convolution_backward (dgrad + wgrad + bias
// grad), masked_fill backward and aten::embedding_dense_backward.
//
// After max-over-time one position per (doc n, filter h) carries gradient g[n,h] = feat_grad * act'(feat).  Define
//     C[v][h*k + j] = sum of g[n,h] over all (n, h) whose tap j reads token id v   (v = ids[n, argmax[n,h] + j - pad], unmasked)
// — every document side of a step accumulates into ONE matrix.  Both parameter gradients are then dense contractions of it:
//     table_grad[v, :]      += sum_hj C[v][hj] * W[hj, :]          [V x HJ] · [HJ x E]      (cmat_table_gemm_kernel)
//     weight_grad[hj, :]    += sum_v  C[v][hj] * x[v, :]           [HJ x V] · [V x E]       (cmat_weight_gemm_kernel)
// with x = the bf16 shadow table and W = the bf16-rounded conv weights, i.e. exactly the operands the forward multiplied.
// Against the arg-max-sparse CUDA-core kernels (conv_bwd.cu: one 600-byte row fetched per entry for EACH of the two
// gradients, a token sort, vector atomics into the 60 MB table gradient) the per-entry work drops to one 4-byte atomic and
// the row traffic to two passes over C: the DeepCoNN backward goes from ~0.45 ms to ~0.1 ms, NARRE's from 3.3 ms to < 1 ms.
//
// Precision: C is accumulated in fp32 (atomics), then split into bf16 hi + lo halves (C = hi + lo up to 2^-17 relative), so
// the tensor cores see the coefficient sums essentially exactly; products accumulate in fp32 in TMEM.
//
// Pipeline (all on the caller's stream):
//   cmat_scatter_kernel      per document side: C32[v][hj] += g (red.global.add.f32), bias_grad[h] += g
//   cmat_split_kernel        C32 → Chl = [hi | lo] bf16 (each C32 block is zero-filled by rbr_conv_bwd_cmat_begin before its scatter)
//   cmat_table_gemm_kernel   D[128 tokens x 160] = Chl[128 x 2HJp] · Wt2ᵀ   — A, B K-major SWIZZLE_128B via TMA, cta_group::1,
//                            2 CTAs/SM; epilogue adds the tile into table_grad (the padding row is skipped)
//   cmat_weight_gemm_kernel  D[128 hj x emb_pad] = sum over a slice of the vocabulary of Chlᵀ · x   — both operands MN-MAJOR
//                            (the contraction index, the token, is the row index of both TMA boxes), split-K over CTAs,
//                            epilogue = vector atomics into a [H][k][E] scratch, then transposed into weight_grad [H,E,k]
#include "rbr_common.cuh"
#include "tc_ptx.cuh"
#include "tma_util.cuh"

namespace rbr {

constexpr int CM_THREADS = 192;            // warp 0: TMA producer, warp 1: TMEM owner + MMA issuer, warps 2..5: epilogue
constexpr int CM_STAGES_T = 3;             // table GEMM ring (36 KB per stage, 2 CTAs per SM)
constexpr int CM_STAGES_W = 3;             // weight GEMM ring (up to 56 KB per stage, 1 CTA per SM)

struct CmatLayout {
    int64_t V, H, K, E, HJ, HJp, emb_pad, epad4;
    int64_t off_c32, off_chl, off_dw, total;
    // C32 is stored as n_chunks FILTER BLOCKS, block c = filters [c*hc, min(H, (c+1)*hc)) = columns [c*hc*K, ...) of the logical
    // [V][HJp] matrix, each block a contiguous [V][width] array (the last one also holds the zero padding columns up to HJp).
    // A block is sized to stay mostly L2-resident while the scatter's atomics land in it: a RED that misses L2 costs a DRAM
    // sector read + write-back at random addresses (44 G/s measured), one that hits is several times cheaper.  Blocking by
    // filter, not by token, means every (doc, filter) item belongs to exactly one block: the passes partition the items,
    // nothing is re-read.  Measured inside the graphed step (tools/timeline_step.py): DeepCoNN (64 MB) is fastest as ONE block
    // (939 us/step; 968 with two), NARRE (102 MB) with two (1567 us/step; 1584 with one, 1607 with three) — more passes cost
    // more in launches and stream joins than the extra L2 hits return, hence the 80 MB target.
    int64_t n_chunks, hc;
};
struct CmatChunk { int64_t h_lo, h_n, col_lo, width, base; };      // base = float offset of the block inside C32
static CmatLayout cmat_layout(int64_t vocab, int64_t emb, int64_t filters, int64_t ksize) {
    CmatLayout l;
    l.V = vocab; l.H = filters; l.K = ksize; l.E = emb;
    l.HJ = filters * ksize;
    l.HJp = cmat_hjp(filters, ksize);
    l.emb_pad = rbr_emb_pad(emb);
    l.epad4 = round_up(emb, 4);
    int64_t off = 0;
    l.off_c32 = off; off += round_up(vocab * l.HJp * 4, 1024);
    l.off_chl = off; off += round_up(vocab * 2 * l.HJp * 2, 1024);
    l.off_dw = off; off += round_up(l.HJ * l.epad4 * 4, 1024);
    l.total = off;
    int64_t want = (vocab * l.HJp * 4 + (80ll << 20) - 1) / (80ll << 20);
    want = std::max<int64_t>(1, std::min<int64_t>(want, 16));
    l.hc = round_up((filters + want - 1) / want, 4);                            // block widths stay float4-aligned
    l.n_chunks = (filters + l.hc - 1) / l.hc;
    return l;
}
static CmatChunk cmat_chunk(const CmatLayout& l, int64_t c) {
    CmatChunk k;
    k.h_lo = c * l.hc;
    k.h_n = std::min(l.H, k.h_lo + l.hc) - k.h_lo;
    k.col_lo = k.h_lo * l.K;
    k.width = (c == l.n_chunks - 1) ? l.HJp - k.col_lo : l.hc * l.K;
    k.base = l.V * k.col_lo;
    return k;
}

// ------------------------------------------------------------------------------------------------------------------
// scatter: one thread per (doc, filter) item, IT items in flight per thread.
// The chain per item is two dependent memory round trips — {feat, feat_grad, arg-max} → {the k token ids (and mask bytes)
// under the window} → k fire-and-forget REDs — and nearly every load misses L2 (the operands of a whole step stream through
// it), so the kernel is bound by how many of those loads are in flight: the inputs of an item are fetched together, the tap
// loop is unrolled (KT = k, or 0 = runtime loop) so its k id / mask loads issue back to back, and the SM is kept full
// (2048 threads x IT items).
template <int KT, int IT>
__global__ void __launch_bounds__(256, IT > 2 ? 6 : 8) cmat_scatter_kernel(const IdView ids, const uint8_t* __restrict__ mask, int64_t n_docs, int L, int H,
                                                              int K, int pad, int64_t v_lo, int64_t v_hi, const float* __restrict__ feat,
                                                              const int32_t* __restrict__ argmax, const float* __restrict__ feat_grad,
                                                              int feat_ld, int act, float* __restrict__ c32, int HJp,
                                                              float* __restrict__ bias_grad) {
    // H = filters of this block (feat / argmax / feat_grad / bias_grad already point at its first filter), c32 = the block,
    // HJp = its row pitch
    extern __shared__ float bsum[];            // [H] CTA-partial bias gradient
    for (int i = threadIdx.x; i < H; i += blockDim.x) bsum[i] = 0.f;
    __syncthreads();
    constexpr int KU = KT > 0 ? KT : 1;        // unrolled taps per pass of the tap loop
    const int taps = KT > 0 ? KT : K;
    const uint32_t total = (uint32_t)(n_docs * H);                 // < 2^31 (checked by the caller): 32-bit index arithmetic
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t q0 = blockIdx.x * blockDim.x + threadIdx.x; q0 < total; q0 += IT * stride) {
        uint32_t n[IT];
        int h[IT], ts[IT];
        float g[IT];
#pragma unroll
        for (int u = 0; u < IT; ++u) {
            const uint32_t q = q0 + u * stride;
            g[u] = 0.f;
            n[u] = 0; h[u] = 0; ts[u] = 0;
            if (q < total && q >= q0) {
                n[u] = q / (uint32_t)H;
                h[u] = (int)(q - n[u] * (uint32_t)H);
                const int64_t o = (int64_t)n[u] * feat_ld + h[u];
                const float y = __ldg(feat + o), gr = __ldg(feat_grad + o);
                ts[u] = __ldg(argmax + o) - pad;
                g[u] = gr * act_grad_from_out(act, y);
            }
        }
#pragma unroll
        for (int u = 0; u < IT; ++u)
            if (g[u] != 0.f && bias_grad) atomicAdd(bsum + h[u], g[u]);
        for (int j0 = 0; j0 < taps; j0 += KU) {
            int row[IT][KU];                   // C row of tap j0 + jj of item u, or -1 (rows are < 2^31: cmat_shape_ok)
#pragma unroll
            for (int u = 0; u < IT; ++u)
#pragma unroll
                for (int jj = 0; jj < KU; ++jj) {
                    const int t = ts[u] + j0 + jj;
                    row[u][jj] = -1;
                    if (g[u] != 0.f && t >= 0 && t < L) {
                        const int64_t i = (int64_t)n[u] * L + t;
                        const int64_t id = ld_id(ids, i);
                        if (ld_mask(ids, mask, i, id) && id >= v_lo && id < v_hi) row[u][jj] = (int)id;
                    }
                }
#pragma unroll
            for (int u = 0; u < IT; ++u)
#pragma unroll
                for (int jj = 0; jj < KU; ++jj)
                    if (row[u][jj] >= 0)
                        atomicAdd(c32 + (int64_t)row[u][jj] * HJp + h[u] * K + j0 + jj, g[u]);      // no return value: RED.E.ADD.F32
        }
    }
    __syncthreads();
    if (bias_grad)
        for (int i = threadIdx.x; i < H; i += blockDim.x) {
            const float v = bsum[i];
            if (v != 0.f) atomicAdd(bias_grad + i, v);
        }
}

// The same scatter, specialised until the item loop is ~60 straight-line instructions (the generic kernel above executes ~220
// per item: index divisions, IdView / mask / range branches, a CAS loop per bias partial — it was issue-bound at 60 us for
// NARRE's 6.1 M items with every load hitting L2).  Here the grid size makes the thread count a multiple of H, so a thread keeps
// ONE filter h for its whole life (bias partial in a register, documents advance by a constant, no division in the loop); all
// indices are 32-bit; window positions are clamped instead of branched around; id width and mask source are template arguments.
template <int KT, int IT, int I32, int MM>       // I32: id width 0 = int64, 1 = int32, 2 = uint16;       // MM: 0 = no mask, 1 = mask bytes, 2 = mask is (id != 0)
__global__ void __launch_bounds__(256, 8) cmat_scatter_fast_kernel(const void* __restrict__ ids_raw, const uint8_t* __restrict__ mask, int n_docs,
                                                                   int L, int H, int pad, int v_lo, int v_hi, const float* __restrict__ feat,
                                                                   const int32_t* __restrict__ argmax, const float* __restrict__ feat_grad,
                                                                   int feat_ld, int act, float* __restrict__ c32, int HJp,
                                                                   float* __restrict__ bias_grad) {
    extern __shared__ float bsum[];            // [H] CTA-partial bias gradient
    for (int i = threadIdx.x; i < H; i += blockDim.x) bsum[i] = 0.f;
    __syncthreads();
    const uint32_t gthreads = gridDim.x * blockDim.x;               // a multiple of H (host)
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    const int h = (int)(q % (uint32_t)H);
    const int dn = (int)(gthreads / (uint32_t)H);                   // documents per grid-wide step
    const int hk = h * KT;
    const uint32_t v_span = (uint32_t)(v_hi - v_lo);
    const bool relu = act == RBR_ACT_RELU;
    float bacc = 0.f;
    for (int n0 = (int)(q / (uint32_t)H); n0 < n_docs; n0 += IT * dn) {
        int nn[IT], ts[IT];
        float g[IT];
#pragma unroll
        for (int u = 0; u < IT; ++u) {
            const int n = n0 + u * dn;
            nn[u] = n < n_docs ? n : n_docs - 1;
            const int o = nn[u] * feat_ld + h;
            // streamed once: evict-first, so that they do not push the coefficient block the atomics land in out of L2
            const float y = __ldcs(feat + o), gr = __ldcs(feat_grad + o);
            ts[u] = __ldcs(argmax + o) - pad;
            const float d = relu ? (y > 0.f ? 1.f : 0.f) : (1.f - y * y);
            g[u] = n < n_docs ? gr * d : 0.f;
        }
        int row[IT][KT];
#pragma unroll
        for (int u = 0; u < IT; ++u)
#pragma unroll
            for (int j = 0; j < KT; ++j) {
                const int t = ts[u] + j;
                const int tc = min(max(t, 0), L - 1);
                const int i = nn[u] * L + tc;
                int id;
                if (I32 == 2) id = (int)__ldg(reinterpret_cast<const uint16_t*>(ids_raw) + i);
                else if (I32 == 1) id = __ldg(reinterpret_cast<const int32_t*>(ids_raw) + i);
                else {
                    const int64_t w = __ldg(reinterpret_cast<const int64_t*>(ids_raw) + i);
                    id = (w >= 0 && w < 0x7fffffffll) ? (int)w : -1;
                }
                bool ok = (t == tc) && g[u] != 0.f && (uint32_t)(id - v_lo) < v_span;
                if (MM == 1) ok = ok && __ldg(mask + i) != 0;
                if (MM == 2) ok = ok && id != 0;
                row[u][j] = ok ? id : -1;
            }
#pragma unroll
        for (int u = 0; u < IT; ++u) {
            bacc += g[u];
#pragma unroll
            for (int j = 0; j < KT; ++j)
                if (row[u][j] >= 0) atomicAdd(c32 + ((uint32_t)row[u][j] * (uint32_t)HJp + (uint32_t)(hk + j)), g[u]);
        }
    }
    if (bias_grad) {
        if (bacc != 0.f) atomicAdd(bsum + h, bacc);
        __syncthreads();
        for (int i = threadIdx.x; i < H; i += blockDim.x) {
            const float v = bsum[i];
            if (v != 0.f) atomicAdd(bias_grad + i, v);
        }
    }
}

// One filter block of C32 ([rows][width] fp32) → its columns of Chl = [hi | lo] bf16 ([rows][2 HJp]).  One thread per 4 columns.
__global__ void __launch_bounds__(256) cmat_split_kernel(const float4* __restrict__ blk, int64_t rows, int width, int col_lo, int HJp,
                                                         __nv_bfloat16* __restrict__ chl) {
    const int q4 = width >> 2;
    const int64_t total = rows * q4;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += stride) {
        const int64_t r = q / q4;
        const int c = col_lo + (int)(q - r * q4) * 4;
        const float4 v = __ldcs(blk + q);                          // dead after this read
        const __nv_bfloat162 h01 = __floats2bfloat162_rn(v.x, v.y), h23 = __floats2bfloat162_rn(v.z, v.w);
        const float2 f01 = __bfloat1622float2(h01), f23 = __bfloat1622float2(h23);
        const __nv_bfloat162 l01 = __floats2bfloat162_rn(v.x - f01.x, v.y - f01.y), l23 = __floats2bfloat162_rn(v.z - f23.x, v.w - f23.y);
        uint2 hi, lo;
        hi.x = *reinterpret_cast<const uint32_t*>(&h01); hi.y = *reinterpret_cast<const uint32_t*>(&h23);
        lo.x = *reinterpret_cast<const uint32_t*>(&l01); lo.y = *reinterpret_cast<const uint32_t*>(&l23);
        __nv_bfloat16* row = chl + r * (2 * (int64_t)HJp);
        *reinterpret_cast<uint2*>(row + c) = hi;
        *reinterpret_cast<uint2*>(row + HJp + c) = lo;
    }
}

// MN-major SWIZZLE_128B operand (cute::UMMA make_umma_desc<Major::MN>, LayoutType::B128: ((8,n),(8,k)):((1,LBO),(8,SBO)) in
// 16-byte units): 64 contiguous MN elements (128 B) per K row, 8 K rows = one 1024-byte swizzle atom, the next 8 K rows SBO
// bytes further, the next 64 MN elements LBO bytes further.  Exactly what TMA writes for a box of [K rows][64 MN columns].
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t addr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((addr >> 4) & 0x3FFFu) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) | ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) |
           (1ull << 46) | (2ull << 61);
}
// instruction descriptor with both operands MN-major (bits 15, 16)
__device__ __forceinline__ uint32_t umma_idesc_mn(int M, int N) { return umma_idesc(M, N) | (1u << 15) | (1u << 16); }

// ------------------------------------------------------------------------------------------------------------------
// table gradient: D[128 tokens x NT] = Chl[128 x 2HJp] · Wt2[NT x 2HJp]ᵀ
// ------------------------------------------------------------------------------------------------------------------
struct TableGemmArgs {
    int64_t vocab;
    int E, NT, nkb;            // nkb = 2 * HJp / 64
    int64_t padding_idx;
    float* table_grad;         // [vocab][E]
    int overwrite;             // 1: table_grad = tile (every row and column of the gradient is written, padding row = 0); 0: +=
};

__global__ void __launch_bounds__(CM_THREADS, 2)
cmat_table_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const TableGemmArgs a) {
    extern __shared__ uint8_t smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t sbase = (raw + 1023u) & ~1023u;
    uint8_t* smem = smem_raw + (sbase - raw);
    const int b_bytes = a.NT * 128;
    const int stage_bytes = 16384 + b_bytes;
    const uint32_t bars = sbase + CM_STAGES_T * stage_bytes;            // full[S], empty[S], acc_full
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + CM_STAGES_T * stage_bytes + 8 * (2 * CM_STAGES_T + 1));
    const int m0 = (int)blockIdx.x * 128, n0 = blockIdx.y * a.NT;

    if (threadIdx.x == 0) {
        for (int i = 0; i < CM_STAGES_T; ++i) { mbar_init(bars + 8 * i, 1); mbar_init(bars + 8 * (CM_STAGES_T + i), 1); }
        mbar_init(bars + 16 * CM_STAGES_T, 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(smem_u32((const void*)tmem_slot), 256);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (elect_one()) {
            tma_prefetch_desc(&tmA);
            tma_prefetch_desc(&tmB);
            int stage = 0;
            uint32_t ph = 0;
            for (int kb = 0; kb < a.nkb; ++kb) {
                mbar_wait(bars + 8 * (CM_STAGES_T + stage), ph ^ 1);
                const uint32_t fb = bars + 8 * stage;
                mbar_expect_tx(fb, (uint32_t)stage_bytes);
                const uint32_t dst = sbase + stage * stage_bytes;
                tma_load_2d(dst, &tmA, kb * 64, m0, fb);
                tma_load_2d(dst + 16384, &tmB, kb * 64, n0, fb);
                if (++stage == CM_STAGES_T) { stage = 0; ph ^= 1; }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        const uint32_t idesc = umma_idesc(128, a.NT);
        int stage = 0;
        uint32_t ph = 0;
        for (int kb = 0; kb < a.nkb; ++kb) {
            mbar_wait(bars + 8 * stage, ph);
            tc_fence_after();
            if (elect_one()) {
                const uint32_t sa = sbase + stage * stage_bytes;
                const uint64_t ad = umma_desc_sw128(sa), bd = umma_desc_sw128(sa + 16384);
#pragma unroll
                for (int ks = 0; ks < 4; ++ks)
                    umma_bf16(tmem_base, ad + (uint64_t)(ks * 2), bd + (uint64_t)(ks * 2), idesc, (uint32_t)((kb | ks) != 0));
                umma_commit(bars + 8 * (CM_STAGES_T + stage));
                if (kb == a.nkb - 1) umma_commit(bars + 16 * CM_STAGES_T);
            }
            __syncwarp();
            if (++stage == CM_STAGES_T) { stage = 0; ph ^= 1; }
        }
    } else {
        const int quad = warp & 3;                                   // TMEM lane quadrant this warp may read
        const int64_t row = (int64_t)m0 + quad * 32 + lane;
        const bool in_range = row < a.vocab;
        const bool pad_row = row == a.padding_idx;
        const bool live = in_range && (a.overwrite || !pad_row);
        const float keep = pad_row ? 0.f : 1.f;                      // overwrite mode writes the padding row as zeros
        float* dst_row = a.table_grad + row * a.E;
        mbar_wait(bars + 16 * CM_STAGES_T, 0);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16);
        for (int c0 = 0; c0 < a.NT; c0 += 16) {
            uint32_t v[16];
            tmem_ld16(taddr + (uint32_t)c0, v);
            tmem_ld_wait();
            if (live) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int col = n0 + c0 + q * 4;
                    if (col + 3 < a.E) {
                        float4* p = reinterpret_cast<float4*>(dst_row + col);
                        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (!a.overwrite) o = *p;
                        o.x += keep * __uint_as_float(v[4 * q]); o.y += keep * __uint_as_float(v[4 * q + 1]);
                        o.z += keep * __uint_as_float(v[4 * q + 2]); o.w += keep * __uint_as_float(v[4 * q + 3]);
                        __stcs(p, o);                                   // streamed: keep Chl (read again by the weight GEMM) in L2 instead
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, 256);
}

// ------------------------------------------------------------------------------------------------------------------
// weight gradient: D[128 hj x emb_pad] = sum over this CTA's token blocks of Chl[tokens, m0:m0+128]ᵀ · x[tokens, :]
// ------------------------------------------------------------------------------------------------------------------
struct WeightGemmArgs {
    int64_t vocab;
    int E, epad4, HJ, HJp, nch;     // nch = emb_pad / 64 (N chunks of 64 columns)
    int n_tb, ksplit;               // token blocks of 64 rows; CTAs per M tile
    float* dw_hke;                  // [HJ][epad4] fp32 scratch (+=)
};

__global__ void __launch_bounds__(CM_THREADS, 1)
cmat_weight_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmX, const WeightGemmArgs a) {
    extern __shared__ uint8_t smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t sbase = (raw + 1023u) & ~1023u;
    uint8_t* smem = smem_raw + (sbase - raw);
    const int stage_bytes = (2 + a.nch) * 8192;
    const uint32_t bars = sbase + CM_STAGES_W * stage_bytes;
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + CM_STAGES_W * stage_bytes + 8 * (2 * CM_STAGES_W + 1));
    const int m0 = blockIdx.x * 128;
    const int split = blockIdx.y;
    const int n_mine = (a.n_tb - split + a.ksplit - 1) / a.ksplit;      // token blocks split, split + ksplit, ...
    const uint32_t tmem_cols = a.nch * 64 <= 256 ? 256u : 512u;

    if (threadIdx.x == 0) {
        for (int i = 0; i < CM_STAGES_W; ++i) { mbar_init(bars + 8 * i, 1); mbar_init(bars + 8 * (CM_STAGES_W + i), 1); }
        mbar_init(bars + 16 * CM_STAGES_W, 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(smem_u32((const void*)tmem_slot), tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (n_mine > 0) {
        if (warp == 0) {
            if (elect_one()) {
                tma_prefetch_desc(&tmA);
                tma_prefetch_desc(&tmX);
                int stage = 0;
                uint32_t ph = 0;
                for (int i = 0; i < n_mine; ++i) {
                    const int row = (split + i * a.ksplit) * 64;
                    mbar_wait(bars + 8 * (CM_STAGES_W + stage), ph ^ 1);
                    const uint32_t fb = bars + 8 * stage;
                    mbar_expect_tx(fb, (uint32_t)stage_bytes);
                    const uint32_t dst = sbase + stage * stage_bytes;
                    tma_load_2d(dst, &tmA, m0, row, fb);
                    tma_load_2d(dst + 8192, &tmA, m0 + 64, row, fb);
                    for (int c = 0; c < a.nch; ++c) tma_load_2d(dst + 16384 + c * 8192, &tmX, c * 64, row, fb);
                    if (++stage == CM_STAGES_W) { stage = 0; ph ^= 1; }
                }
            }
            __syncwarp();
        } else if (warp == 1) {
            // N is issued in groups of <= 4 chunks (UMMA N <= 256)
            const int g0 = a.nch <= 4 ? a.nch : (a.nch + 1) / 2, g1 = a.nch - g0;
            const uint32_t idesc0 = umma_idesc_mn(128, g0 * 64), idesc1 = g1 ? umma_idesc_mn(128, g1 * 64) : 0u;
            int stage = 0;
            uint32_t ph = 0;
            for (int i = 0; i < n_mine; ++i) {
                mbar_wait(bars + 8 * stage, ph);
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t sa = sbase + stage * stage_bytes, sb = sa + 16384;
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {                 // 16 token rows (K) per MMA = 2048 bytes of every chunk
                        const uint64_t ad = umma_desc_mn_sw128(sa + ks * 2048, 8192, 1024);
                        umma_bf16(tmem_base, ad, umma_desc_mn_sw128(sb + ks * 2048, 8192, 1024), idesc0, (uint32_t)((i | ks) != 0));
                        if (g1)
                            umma_bf16(tmem_base + (uint32_t)(g0 * 64), ad, umma_desc_mn_sw128(sb + g0 * 8192 + ks * 2048, 8192, 1024), idesc1,
                                      (uint32_t)((i | ks) != 0));
                    }
                    umma_commit(bars + 8 * (CM_STAGES_W + stage));
                    if (i == n_mine - 1) umma_commit(bars + 16 * CM_STAGES_W);
                }
                __syncwarp();
                if (++stage == CM_STAGES_W) { stage = 0; ph ^= 1; }
            }
        } else {
            const int quad = warp & 3;
            const int gm = m0 + quad * 32 + lane;                    // column of [hi | lo]
            const int hj = gm >= a.HJp ? gm - a.HJp : gm;            // hi and lo halves add into the same row
            const bool live = hj < a.HJ;
            float* dst_row = a.dw_hke + (int64_t)hj * a.epad4;
            mbar_wait(bars + 16 * CM_STAGES_W, 0);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16);
            for (int c0 = 0; c0 < a.nch * 64; c0 += 16) {
                uint32_t v[16];
                tmem_ld16(taddr + (uint32_t)c0, v);
                tmem_ld_wait();
                if (live) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int col = c0 + q * 4;
                        if (col + 3 < a.E)
                            atomicAdd(reinterpret_cast<float4*>(dst_row + col),
                                      make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]), __uint_as_float(v[4 * q + 2]),
                                                  __uint_as_float(v[4 * q + 3])));
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, tmem_cols);
}

// weight_grad[h][e][j] += dw_hke[h][j][e];  dw_hke re-zeroed
__global__ void cmat_unpack_kernel(float* __restrict__ dw_hke, int H, int E, int K, int epad4, float* __restrict__ wgrad) {
    const int64_t total = (int64_t)H * K * epad4;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += stride) {
        const int e = (int)(q % epad4);
        const int hj = (int)(q / epad4);
        const float v = dw_hke[q];
        if (v != 0.f) {
            dw_hke[q] = 0.f;
            if (e < E) atomicAdd(wgrad + ((int64_t)(hj / K) * E + e) * K + (hj % K), v);
        }
    }
}

// Dynamic shared memory of the two GEMMs of rbr_conv_bwd_cmat_finish (rings + barriers + TMEM slot + 1024-byte alignment slack),
// and the most each may take.  cmat_shape_ok declines a shape that exceeds either, so "supported" means "finish will run": the
// weight GEMM's ring grows with the embedding width (emb_pad 512 needs 240 KB) and such shapes go to the sparse backward instead.
constexpr int CM_SMEM_T_MAX = 116 * 1024;  // two table-GEMM CTAs per SM
constexpr int CM_SMEM_W_MAX = 227 * 1024;
struct CmatSmem { int table, weight; };
static CmatSmem cmat_smem(int64_t emb) {
    int64_t NT, tiles;
    cmat_ntile(emb, &NT, &tiles);
    const int64_t nch = rbr_emb_pad(emb) / 64;
    CmatSmem s;
    s.table = CM_STAGES_T * (16384 + (int)NT * 128) + 8 * (2 * CM_STAGES_T + 1) + 16 + 1024;
    s.weight = CM_STAGES_W * (2 + (int)nch) * 8192 + 8 * (2 * CM_STAGES_W + 1) + 16 + 1024;
    return s;
}

static bool cmat_shape_ok(int64_t vocab, int64_t emb, int64_t filters, int64_t ksize) {
    if (vocab < 1 || vocab >= (1ll << 31) || emb < 4 || emb % 4 != 0 || emb > 512 || filters < 1 || ksize < 1 || ksize > 8) return false;
    if (filters > 1024) return false;
    const CmatSmem sm = cmat_smem(emb);
    if (sm.table > CM_SMEM_T_MAX || sm.weight > CM_SMEM_W_MAX) return false;
    const int64_t hjp = cmat_hjp(filters, ksize);
    if (hjp > 4096) return false;
    return vocab * hjp * 4 <= (3ll << 30);          // coefficient matrix up to 3 GiB (fp32) + the same again in bf16
}

}  // namespace rbr

using namespace rbr;

extern "C" int rbr_conv_bwd_cmat_supported(int64_t vocab, int64_t emb, int64_t filters, int64_t ksize) {
    return cmat_shape_ok(vocab, emb, filters, ksize) && tensor_map_encoder() != nullptr ? 1 : 0;
}

extern "C" int64_t rbr_conv_bwd_cmat_workspace_bytes(int64_t vocab, int64_t emb, int64_t filters, int64_t ksize) {
    if (!cmat_shape_ok(vocab, emb, filters, ksize)) return 0;
    return cmat_layout(vocab, emb, filters, ksize).total;
}

extern "C" int rbr_conv_bwd_cmat_chunks(int64_t vocab, int64_t emb, int64_t filters, int64_t ksize) {
    if (!cmat_shape_ok(vocab, emb, filters, ksize)) return 0;
    return (int)cmat_layout(vocab, emb, filters, ksize).n_chunks;
}

extern "C" int rbr_conv_bwd_cmat_begin(int chunk, int64_t vocab, int64_t emb, int64_t filters, int64_t ksize, void* ws, int64_t ws_bytes,
                                       void* stream) {
    RBR_REQUIRE(ws, RBR_EINVAL, "conv_bwd_cmat_begin: null pointer");
    RBR_REQUIRE(cmat_shape_ok(vocab, emb, filters, ksize), RBR_EUNSUPPORTED, "conv_bwd_cmat: shape outside the dense tensor-core backward");
    const CmatLayout l = cmat_layout(vocab, emb, filters, ksize);
    RBR_REQUIRE(ws_bytes >= l.total, RBR_EWORKSPACE, "conv_bwd_cmat_begin: workspace too small");
    RBR_REQUIRE(chunk >= -1 && chunk < l.n_chunks, RBR_EINVAL, "conv_bwd_cmat_begin: bad chunk");
    float* c32 = reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + l.off_c32);
    if (chunk < 0) {
        RBR_CUDA(cudaMemsetAsync(c32, 0, (size_t)(vocab * l.HJp * 4), as_stream(stream)));
    } else {
        const CmatChunk k = cmat_chunk(l, chunk);
        RBR_CUDA(cudaMemsetAsync(c32 + k.base, 0, (size_t)(vocab * k.width * 4), as_stream(stream)));
    }
    return RBR_OK;
}

// one filter block of one document side
static int cmat_scatter_block(const CmatLayout& l, const CmatChunk& k, const void* ids_raw, const uint8_t* mask, int64_t n_docs, int64_t doc_len,
                              int64_t pad, int activation, const float* feat, const int32_t* argmax, const float* feat_grad, int64_t feat_ld,
                              float* bias_grad, float* c32, int flags, void* stream) {
    const int64_t vocab = l.V, ksize = l.K, filters = k.h_n;
    feat += k.h_lo; argmax += k.h_lo; feat_grad += k.h_lo;
    if (bias_grad) bias_grad += k.h_lo;
    float* c32p = c32 + k.base;
    const int pitch = (int)k.width;
    const int64_t total = n_docs * filters;
    RBR_REQUIRE(total < (1ll << 31) - (1ll << 24), RBR_EUNSUPPORTED, "conv_bwd_cmat_scatter: n_docs * filters must stay below 2^31");
    // fast path: 32-bit indices everywhere, k in {1, 3, 5}, and a grid whose thread count is a multiple of the block's filters
    {
        int64_t g = filters, r = 256;
        while (r) { const int64_t t = g % r; g = r; r = t; }            // g = gcd(filters, 256)
        const int64_t m = filters / g;                                  // grid must be a multiple of m
        const bool small = n_docs * std::max(feat_ld, doc_len) < (1ll << 31) - 1 && vocab < (1ll << 31) - 1 && vocab * k.width < (1ll << 32) &&
                           filters * ksize < (1 << 20);
        if (small && m <= 148 * 8 && (ksize == 1 || ksize == 3 || ksize == 5)) {
            constexpr int IT = 2;
            int64_t blocks = (total + 256 * IT - 1) / (256 * IT);
            if (blocks > 148 * 8) blocks = 148 * 8;
            blocks = std::max<int64_t>(m, blocks / m * m);
            const int mm = mask ? 1 : ((flags & RBR_MASK_FROM_IDS) ? 2 : 0);
            const int i32 = (flags & RBR_IDS_U16) ? 2 : ((flags & RBR_IDS_I32) ? 1 : 0);
#define RBR_SF(KT, I32, MM)                                                                                                              \
    cmat_scatter_fast_kernel<KT, IT, I32, MM><<<(unsigned)blocks, 256, (size_t)filters * 4, as_stream(stream)>>>(                        \
        ids_raw, mask, (int)n_docs, (int)doc_len, (int)filters, (int)pad, 0, (int)vocab, feat, argmax, feat_grad, (int)feat_ld,          \
        activation, c32p, pitch, bias_grad)
#define RBR_SF_K(I32, MM)                                                                     \
    do {                                                                                      \
        if (ksize == 1) RBR_SF(1, I32, MM); else if (ksize == 3) RBR_SF(3, I32, MM); else RBR_SF(5, I32, MM); \
    } while (0)
            if (i32 == 2)      { if (mm == 0) RBR_SF_K(2, 0); else if (mm == 1) RBR_SF_K(2, 1); else RBR_SF_K(2, 2); }
            else if (i32 == 1) { if (mm == 0) RBR_SF_K(1, 0); else if (mm == 1) RBR_SF_K(1, 1); else RBR_SF_K(1, 2); }
            else               { if (mm == 0) RBR_SF_K(0, 0); else if (mm == 1) RBR_SF_K(0, 1); else RBR_SF_K(0, 2); }
#undef RBR_SF_K
#undef RBR_SF
            RBR_LAUNCH_CHECK("cmat_scatter_fast_kernel");
            return RBR_OK;
        }
    }
    int64_t blocks = (total + 256 * 2 - 1) / (256 * 2);
    if (blocks > 148 * 8) blocks = 148 * 8;
#define RBR_SCATTER(KT)                                                                                                                      \
    cmat_scatter_kernel<KT, 2><<<(unsigned)blocks, 256, (size_t)filters * 4, as_stream(stream)>>>(                                           \
        id_view(ids_raw, flags), mask, n_docs, (int)doc_len, (int)filters, (int)ksize, (int)pad, 0, vocab, feat, argmax, feat_grad, (int)feat_ld, \
        activation, c32p, pitch, bias_grad)
    switch (ksize) {
        case 1: RBR_SCATTER(1); break;
        case 3: RBR_SCATTER(3); break;
        case 5: RBR_SCATTER(5); break;
        default: RBR_SCATTER(0); break;
    }
#undef RBR_SCATTER
    RBR_LAUNCH_CHECK("cmat_scatter_kernel");
    return RBR_OK;
}

extern "C" int rbr_conv_bwd_cmat_scatter(const void* ids_raw, const uint8_t* mask, int64_t n_docs, int64_t doc_len, int64_t vocab,
                                         int64_t emb, int64_t filters, int64_t ksize, int64_t pad, int activation, const float* feat,
                                         const int32_t* argmax, const float* feat_grad, int64_t feat_ld, float* bias_grad, int chunk,
                                         void* ws, int64_t ws_bytes, int flags, void* stream) {
    RBR_REQUIRE(ids_raw && feat && argmax && feat_grad && ws, RBR_EINVAL, "conv_bwd_cmat_scatter: null pointer");
    RBR_REQUIRE(cmat_shape_ok(vocab, emb, filters, ksize), RBR_EUNSUPPORTED, "conv_bwd_cmat: shape outside the dense tensor-core backward");
    RBR_REQUIRE(n_docs >= 0 && doc_len > 0 && pad >= 0 && feat_ld >= filters, RBR_EINVAL, "conv_bwd_cmat_scatter: bad sizes");
    const CmatLayout l = cmat_layout(vocab, emb, filters, ksize);
    RBR_REQUIRE(ws_bytes >= l.total, RBR_EWORKSPACE, "conv_bwd_cmat_scatter: workspace too small");
    RBR_REQUIRE(chunk >= -1 && chunk < l.n_chunks, RBR_EINVAL, "conv_bwd_cmat_scatter: bad chunk");
    if (n_docs == 0) return RBR_OK;
    float* c32 = reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + l.off_c32);
    for (int64_t c = (chunk < 0 ? 0 : chunk); c < (chunk < 0 ? l.n_chunks : chunk + 1); ++c) {
        const int rc = cmat_scatter_block(l, cmat_chunk(l, c), ids_raw, mask, n_docs, doc_len, pad, activation, feat, argmax, feat_grad, feat_ld,
                                          bias_grad, c32, flags, stream);
        if (rc != RBR_OK) return rc;
    }
    return RBR_OK;
}

extern "C" int rbr_conv_bwd_cmat_finish(int what, int chunk, const void* shadow_bf16, const void* packed,
                                        int64_t vocab, int64_t emb, int64_t filters, int64_t ksize, int64_t padding_idx, float* table_grad,
                                        float* weight_grad, void* ws, int64_t ws_bytes, void* stream) {
    RBR_REQUIRE(ws && packed, RBR_EINVAL, "conv_bwd_cmat_finish: null pointer");
    RBR_REQUIRE(cmat_shape_ok(vocab, emb, filters, ksize), RBR_EUNSUPPORTED, "conv_bwd_cmat: shape outside the dense tensor-core backward");
    RBR_REQUIRE((what & ~15) == 0 && (what & 7) != 0, RBR_EINVAL,
                "conv_bwd_cmat_finish: `what` is a mask of 1 (split), 2 (table), 4 (weight), 8 (table: overwrite instead of +=)");
    const CmatLayout l = cmat_layout(vocab, emb, filters, ksize);
    RBR_REQUIRE(ws_bytes >= l.total, RBR_EWORKSPACE, "conv_bwd_cmat_finish: workspace too small");
    const PackLayout pl = pack_layout(emb, filters, ksize);
    cudaStream_t s = as_stream(stream);
    char* base = reinterpret_cast<char*>(ws);
    float* c32 = reinterpret_cast<float*>(base + l.off_c32);
    __nv_bfloat16* chl = reinterpret_cast<__nv_bfloat16*>(base + l.off_chl);
    float* dw = reinterpret_cast<float*>(base + l.off_dw);
    if (what & 1) {
        RBR_REQUIRE(chunk >= -1 && chunk < l.n_chunks, RBR_EINVAL, "conv_bwd_cmat_finish: bad chunk");
        for (int64_t c = (chunk < 0 ? 0 : chunk); c < (chunk < 0 ? l.n_chunks : chunk + 1); ++c) {
            const CmatChunk k = cmat_chunk(l, c);
            const int64_t total = vocab * (k.width / 4);
            int64_t blocks = (total + 255) / 256;
            if (blocks > 148 * 16) blocks = 148 * 16;
            cmat_split_kernel<<<(unsigned)blocks, 256, 0, s>>>(reinterpret_cast<const float4*>(c32 + k.base), vocab, (int)k.width, (int)k.col_lo,
                                                               (int)l.HJp, chl);
            RBR_LAUNCH_CHECK("cmat_split_kernel");
        }
    }
    if (what & 2) {
        RBR_REQUIRE(table_grad, RBR_EINVAL, "conv_bwd_cmat_finish: table part needs table_grad");
        RBR_REQUIRE((uintptr_t)table_grad % 16 == 0, RBR_EINVAL, "conv_bwd_cmat_finish: table_grad must be 16-byte aligned");
        CUtensorMap tmA, tmB;
        RBR_REQUIRE(make_tmap_bf16_2d(&tmA, chl, (uint64_t)(2 * l.HJp), (uint64_t)vocab, (uint64_t)(2 * l.HJp), 64, 128) &&
                        make_tmap_bf16_2d(&tmB, reinterpret_cast<const char*>(packed) + pl.off_wt2, (uint64_t)(2 * l.HJp),
                                          (uint64_t)(pl.NT * pl.n_tiles), (uint64_t)(2 * l.HJp), 64, (uint32_t)pl.NT),
                    RBR_ECUDA, "conv_bwd_cmat_finish: cuTensorMapEncodeTiled failed");
        TableGemmArgs a{};
        a.vocab = vocab; a.E = (int)emb; a.NT = (int)pl.NT; a.nkb = (int)(2 * l.HJp / 64); a.padding_idx = padding_idx;
        a.table_grad = table_grad;
        a.overwrite = (what & 8) ? 1 : 0;
        const int smem = cmat_smem(emb).table;
        static bool attr = false;
        if (!attr) {
            RBR_CUDA(cudaFuncSetAttribute(cmat_table_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CM_SMEM_T_MAX));
            attr = true;
        }
        RBR_REQUIRE(smem <= CM_SMEM_T_MAX, RBR_EUNSUPPORTED, "conv_bwd_cmat_finish: shared memory");
        dim3 grid((unsigned)((vocab + 127) / 128), (unsigned)pl.n_tiles);
        cmat_table_gemm_kernel<<<grid, CM_THREADS, smem, s>>>(tmA, tmB, a);
        RBR_LAUNCH_CHECK("cmat_table_gemm_kernel");
    }
    if (what & 4) {
        RBR_REQUIRE(weight_grad && shadow_bf16, RBR_EINVAL, "conv_bwd_cmat_finish: weight part needs weight_grad and the bf16 shadow table");
        CUtensorMap tmA, tmX;
        RBR_REQUIRE(make_tmap_bf16_2d(&tmA, chl, (uint64_t)(2 * l.HJp), (uint64_t)vocab, (uint64_t)(2 * l.HJp), 64, 64) &&
                        make_tmap_bf16_2d(&tmX, shadow_bf16, (uint64_t)l.emb_pad, (uint64_t)vocab, (uint64_t)l.emb_pad, 64, 64),
                    RBR_ECUDA, "conv_bwd_cmat_finish: cuTensorMapEncodeTiled failed");
        WeightGemmArgs a{};
        a.vocab = vocab; a.E = (int)emb; a.epad4 = (int)l.epad4; a.HJ = (int)l.HJ; a.HJp = (int)l.HJp; a.nch = (int)(l.emb_pad / 64);
        a.n_tb = (int)((vocab + 63) / 64);
        const int m_tiles = (int)(2 * l.HJp / 128);
        static int sms = 0;
        if (!sms) {
            int dev = 0;
            RBR_CUDA(cudaGetDevice(&dev));
            RBR_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        }
        a.ksplit = sms / m_tiles < 1 ? 1 : sms / m_tiles;
        if (a.ksplit > a.n_tb) a.ksplit = a.n_tb;
        a.dw_hke = dw;
        const int smem = cmat_smem(emb).weight;
        static bool attr = false;
        if (!attr) {
            RBR_CUDA(cudaFuncSetAttribute(cmat_weight_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CM_SMEM_W_MAX));
            attr = true;
        }
        RBR_REQUIRE(smem <= CM_SMEM_W_MAX, RBR_EUNSUPPORTED, "conv_bwd_cmat_finish: shared memory");
        dim3 grid((unsigned)m_tiles, (unsigned)a.ksplit);
        cmat_weight_gemm_kernel<<<grid, CM_THREADS, smem, s>>>(tmA, tmX, a);
        RBR_LAUNCH_CHECK("cmat_weight_gemm_kernel");
        const int64_t tot = l.HJ * l.epad4;
        int blocks = (int)((tot + 255) / 256);
        if (blocks > 148 * 4) blocks = 148 * 4;
        cmat_unpack_kernel<<<blocks, 256, 0, s>>>(dw, (int)filters, (int)emb, (int)ksize, (int)l.epad4, weight_grad);
        RBR_LAUNCH_CHECK("cmat_unpack_kernel");
    }
    return RBR_OK;
}
