// attn_tc.cu — K3 on tensor cores: NARRE review-level attention for BOTH sides in one launch, forward and backward.
//
// Replaces LinearAttention.forward (reference models/narre/narre.py:40-64) and its autograd reverse:
//     e      = ebd_vals(other_id)                                    [B,R,A]     (narre.py:53)
//     logit  = relu(feat@W_rv + e@W_id + b_1) @ h + b_2              [B,R]       (narre.py:55)
//     score  = exp(logit) / (sum_R exp(logit) + 1e-8)                            (narre.py:58; no mask, no max-shift)
//     out    = sum_R score * feat                                    [B,H]       (narre.py:60)
// attn.cu gives each sample to one warp (serial FMA chains: 0.08 of the HBM roofline).  Here a CTA owns a TILE of samples
// (80 review rows) and the three contractions — feat@W_rv, e@W_id and, in the backward, dHid@W_rvᵀ, featᵀ@dHid, eᵀ@dHid,
// dHid@W_idᵀ — run on the tensor cores as warp-level mma.sync.m16n8k8 TF32 in the 3xTF32 scheme
//     x = hi + lo (hi = x with the low 13 mantissa bits cleared, lo = x - hi exactly),   a·b ≈ hi_a·hi_b + lo_a·hi_b + hi_a·lo_b
// whose dropped term is 2^-22 relative: fp32-grade results (the 1e-5 parity bar holds in both conv precision modes), with
// fp32 accumulation.  Weights are split once per CTA into shared memory; the softmax, the weighted pool and all reductions of
// the parameter gradients stay in registers / shared memory.  blockIdx.y = side (user / item): one launch for both.
#include "rbr_common.cuh"

namespace rbr {

constexpr int AT_MAXW = 6;         // m-tiles (16 review rows each) per sample tile; two warps per m-tile → <= 384 threads

// ---- mma.sync m16n8k8 TF32 ------------------------------------------------------------------------------------------
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void split_hi_lo(float x, uint32_t& hi, uint32_t& lo) {
    hi = __float_as_uint(x) & 0xFFFFE000u;            // tf32 keeps 10 mantissa bits: clear the 13 the tensor core would drop
    lo = __float_as_uint(x - __uint_as_float(hi));    // exact; its own low bits are dropped by the hardware (2^-22 relative)
}
// D += A·B in 3xTF32 for one 16x8 tile, A given as fp32 fragment values (split here), B as pre-split hi / lo
__device__ __forceinline__ void mma_3x(float (&d)[4], const uint32_t (&ahi)[4], const uint32_t (&alo)[4], uint32_t bh0, uint32_t bh1,
                                       uint32_t bl0, uint32_t bl1) {
    mma_tf32(d, alo, bh0, bh1);
    mma_tf32(d, ahi, bl0, bl1);
    mma_tf32(d, ahi, bh0, bh1);
}

// Shared-memory layout of a B operand [K rows][N columns], N a multiple of 32 processed in groups of 4 n-tiles: column n of
// a group is stored at (n % 8) * 4 + n / 8, so that the four values a lane needs for n-tiles 0..3 (columns g, g+8, g+16, g+24)
// are one 16-byte load; row pitch 40 floats per 32 columns keeps the quarter-warp phases conflict-free.
__host__ __device__ constexpr int b_pitch(int n_cols) { return (n_cols / 32) * 40; }
__device__ __forceinline__ int b_index(int k, int n, int pitch) { return k * pitch + (n >> 5) * 40 + (n & 7) * 4 + ((n & 31) >> 3); }

struct AttnSide {
    const float* feat;          // [B, R, H]
    const int64_t* other_id;    // [B, R]
    const float *W_rv, *W_id, *h, *b1, *b2, *ebd;
    int64_t n_ids, padding_idx;
    float* out;                 // [B, H]
    float* scores;              // [B, R]
    // backward
    const float *out_grad, *scores_grad;
    float *feat_grad, *W_rv_grad, *W_id_grad, *h_grad, *b1_grad, *b2_grad, *ebd_grad;
};
struct AttnArgs {
    AttnSide side[2];
    int n_sides;
    int64_t B;
    int R, H, A;
    int TS, rows, NW;           // samples per tile, TS * R, warps (= m-tiles of 16 rows)
    int Hp8, PF, PE;            // H rounded up to 8; pitches of the feature / id-embedding tiles
};

struct AttnSmem {
    int wrv_hi, wrv_lo, wid_hi, wid_lo, wrvT_hi, wrvT_lo, widT_hi, widT_lo;   // B operands (bwd: plus the transposed ones)
    int F, E, L, S, GO, DHa, DHb, red;
    int total;
};
__host__ __device__ inline AttnSmem attn_tc_smem(const AttnArgs& a, bool bwd) {
    AttnSmem s;
    int off = 0;
    const int pa = b_pitch(32);                       // A <= 32 columns → one group
    s.wrv_hi = off; off += a.Hp8 * pa;
    s.wrv_lo = off; off += a.Hp8 * pa;
    s.wid_hi = off; off += 32 * pa;
    s.wid_lo = off; off += 32 * pa;
    const int hcols = (a.Hp8 + 31) / 32 * 32;         // W_rvᵀ as a B operand: K = A rows, N = H columns in groups of 32
    s.wrvT_hi = off; if (bwd) off += 32 * b_pitch(hcols);
    s.wrvT_lo = off; if (bwd) off += 32 * b_pitch(hcols);
    s.widT_hi = off; if (bwd) off += 32 * pa;
    s.widT_lo = off; if (bwd) off += 32 * pa;
    s.F = off; off += (a.NW * 16) * a.PF;
    s.E = off; off += (a.NW * 16) * a.PE;
    s.L = off; off += 2 * a.NW * 16;                  // logit partials of the two column halves / d logits per row
    s.S = off; off += a.NW * 16;                      // scores per row
    s.GO = off; if (bwd) off += a.TS * a.PF;          // out_grad rows of the tile's samples
    s.DHa = off; if (bwd) off += (a.NW * 16) * 36;    // d hid as an A operand (row-major, pitch 36)
    s.DHb = off; if (bwd) off += (a.NW * 16) * pa;    // d hid as a B operand (K = rows, permuted columns)
    s.red = off; off += 4 * 32 + 8;                   // cross-warp reductions of dh, db1 (+ db2)
    s.total = off;
    return s;
}

// pick this warp's two n-tiles (half nh of the 32 attention columns) out of a 4-n-tile B-fragment load
__device__ __forceinline__ float sel0(const float4& v, int nh) { return nh ? v.z : v.x; }
__device__ __forceinline__ float sel1(const float4& v, int nh) { return nh ? v.w : v.y; }

// hid accumulators of this warp: m-tile rows m0..m0+15, n-tiles 2nh and 2nh+1 (16 of the 32 attention units) = F·W_rv + E·W_id
__device__ __forceinline__ void attn_hidden_mma(const float* Fs, int PF, const float* Es, int PE, const float* wrv_hi, const float* wrv_lo,
                                                const float* wid_hi, const float* wid_lo, int Hp8, int m0, int nh, int lane,
                                                float (&acc)[2][4]) {
    const int g = lane >> 2, t = lane & 3;
    constexpr int pa = b_pitch(32);
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[nt][i] = 0.f;
    const float* fa = Fs + (m0 + g) * PF + t;
    const float* bh = wrv_hi + t * pa + g * 4;
    const float* bl = wrv_lo + t * pa + g * 4;
    for (int k0 = 0; k0 < Hp8; k0 += 8, fa += 8, bh += 8 * pa, bl += 8 * pa) {
        uint32_t ahi[4], alo[4];
        split_hi_lo(fa[0], ahi[0], alo[0]);
        split_hi_lo(fa[8 * PF], ahi[1], alo[1]);
        split_hi_lo(fa[4], ahi[2], alo[2]);
        split_hi_lo(fa[8 * PF + 4], ahi[3], alo[3]);
        const float4 bh0 = *reinterpret_cast<const float4*>(bh), bh1 = *reinterpret_cast<const float4*>(bh + 4 * pa);
        const float4 bl0 = *reinterpret_cast<const float4*>(bl), bl1 = *reinterpret_cast<const float4*>(bl + 4 * pa);
        mma_3x(acc[0], ahi, alo, __float_as_uint(sel0(bh0, nh)), __float_as_uint(sel0(bh1, nh)), __float_as_uint(sel0(bl0, nh)),
               __float_as_uint(sel0(bl1, nh)));
        mma_3x(acc[1], ahi, alo, __float_as_uint(sel1(bh0, nh)), __float_as_uint(sel1(bh1, nh)), __float_as_uint(sel1(bl0, nh)),
               __float_as_uint(sel1(bl1, nh)));
    }
    const float* ea = Es + (m0 + g) * PE + t;
    const float* ih = wid_hi + t * pa + g * 4;
    const float* il = wid_lo + t * pa + g * 4;
#pragma unroll
    for (int k0 = 0; k0 < 32; k0 += 8) {
        uint32_t ahi[4], alo[4];
        split_hi_lo(ea[k0], ahi[0], alo[0]);
        split_hi_lo(ea[k0 + 8 * PE], ahi[1], alo[1]);
        split_hi_lo(ea[k0 + 4], ahi[2], alo[2]);
        split_hi_lo(ea[k0 + 8 * PE + 4], ahi[3], alo[3]);
        const float4 bh0 = *reinterpret_cast<const float4*>(ih + k0 * pa), bh1 = *reinterpret_cast<const float4*>(ih + (k0 + 4) * pa);
        const float4 bl0 = *reinterpret_cast<const float4*>(il + k0 * pa), bl1 = *reinterpret_cast<const float4*>(il + (k0 + 4) * pa);
        mma_3x(acc[0], ahi, alo, __float_as_uint(sel0(bh0, nh)), __float_as_uint(sel0(bh1, nh)), __float_as_uint(sel0(bl0, nh)),
               __float_as_uint(sel0(bl1, nh)));
        mma_3x(acc[1], ahi, alo, __float_as_uint(sel1(bh0, nh)), __float_as_uint(sel1(bh1, nh)), __float_as_uint(sel1(bl0, nh)),
               __float_as_uint(sel1(bl1, nh)));
    }
}

// split a [K][N] weight (N <= 32 columns, zero padded to 32; rows >= K_real zero) into the permuted hi / lo B layout
__device__ __forceinline__ void stage_b_operand(float* hi, float* lo, const float* __restrict__ w, int k_real, int k_pad, int n_real,
                                                int ld, bool transpose) {
    const int pa = b_pitch(32);
    for (int i = threadIdx.x; i < k_pad * 32; i += blockDim.x) {
        const int k = i >> 5, n = i & 31;
        float v = 0.f;
        if (k < k_real && n < n_real) v = transpose ? w[n * ld + k] : w[k * ld + n];
        uint32_t h_, l_;
        split_hi_lo(v, h_, l_);
        const int idx = b_index(k, n, pa);
        hi[idx] = __uint_as_float(h_);
        lo[idx] = __uint_as_float(l_);
    }
}

// async global → shared copies (LDGSTS): a thread issues all its copies of a tile back to back — with one CTA of 5 warps per
// SM a load-then-store loop exposes a full memory round trip per iteration
__device__ __forceinline__ void cp_async_f32(float* dst_smem, const float* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_f32x2(float* dst_smem, const float* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_f32x4(float* dst_smem, const float* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all_() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// rows [0, n_rows) x columns [0, H) of a row-major fp32 matrix (row pitch H) → shared tile of pitch PF, rows n_rows..rows_pad
// and columns H..PF zero-filled.  One warp per row (no index divisions), lanes across the columns.
__device__ __forceinline__ void stage_rows_async(float* tile, int PF, int rows_pad, const float* __restrict__ src, int n_rows, int H) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const bool pair = (H & 1) == 0 && (reinterpret_cast<uintptr_t>(src) & 7) == 0;
    for (int r = warp; r < rows_pad; r += nw) {
        float* dst = tile + r * PF;
        if (r < n_rows) {
            const float* s_ = src + (int64_t)r * H;
            if (pair) {
                for (int c = lane * 2; c < H; c += 64) cp_async_f32x2(dst + c, s_ + c);
            } else {
                for (int c = lane; c < H; c += 32) cp_async_f32(dst + c, s_ + c);
            }
            for (int c = H + lane; c < PF; c += 32) dst[c] = 0.f;
        } else {
            for (int c = lane; c < PF; c += 32) dst[c] = 0.f;
        }
    }
}

// feature rows + gathered id-embedding rows of one tile → shared memory (zero padded rows / columns); the caller waits
// (cp_async_wait_all_ + __syncthreads) before reading
__device__ __forceinline__ void attn_stage_tile(const AttnArgs& a, const AttnSide& sd, int64_t b0, int n_s, float* Fs, float* Es,
                                                bool count_oob) {
    const int rows_pad = a.NW * 16;
    const int rows_live = n_s * a.R;
    stage_rows_async(Fs, a.PF, rows_pad, sd.feat + b0 * a.R * a.H, rows_live, a.H);
    const bool v4 = (a.A & 3) == 0;
    for (int i = threadIdx.x; i < rows_pad * 8; i += blockDim.x) {            // 8 chunks of 4 attention columns per row
        const int r = i >> 3, c = (i & 7) * 4;
        float* dst = Es + r * a.PE + c;
        bool copied = false;
        if (r < rows_live) {
            const int64_t id = __ldg(sd.other_id + b0 * a.R + r);
            const bool ok = id >= 0 && id < sd.n_ids;
            if (!ok && c == 0 && count_oob) note_oob();
            if (ok && c < a.A) {
                const float* src = sd.ebd + id * a.A + c;
                if (v4) {
                    cp_async_f32x4(dst, src);
                    copied = true;
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) dst[j] = c + j < a.A ? __ldg(src + j) : 0.f;
                    copied = true;
                }
            }
        }
        if (!copied) *reinterpret_cast<float4*>(dst) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

__global__ void __launch_bounds__(2 * AT_MAXW * 32) narre_attn_tc_fwd_kernel(const AttnArgs a) {
    extern __shared__ __align__(16) float smem[];
    const AttnSide& sd = a.side[blockIdx.y];
    const AttnSmem L = attn_tc_smem(a, false);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
    const int mt = warp >> 1, nh = warp & 1;            // two warps per m-tile of 16 review rows: attention units 16nh .. 16nh+15
    stage_b_operand(smem + L.wrv_hi, smem + L.wrv_lo, sd.W_rv, a.H, a.Hp8, a.A, a.A, false);
    stage_b_operand(smem + L.wid_hi, smem + L.wid_lo, sd.W_id, a.A, 32, a.A, a.A, false);
    float* Fs = smem + L.F;
    float* Es = smem + L.E;
    float* Ls = smem + L.L;                              // [2][rows_pad]: logit partials of the two column halves
    float* Ss = smem + L.S;
    const int rows_pad = a.NW * 16;
    const float b2v = __ldg(sd.b2);
    // this lane's 4 attention units: columns (2nh + nt) * 8 + 2t, +1
    float b1v[2][2], hv[2][2];
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int c = (2 * nh + nt) * 8 + 2 * t + j;
            b1v[nt][j] = c < a.A ? __ldg(sd.b1 + c) : 0.f;
            hv[nt][j] = c < a.A ? __ldg(sd.h + c) : 0.f;
        }
    const int64_t n_tiles = (a.B + a.TS - 1) / a.TS;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t b0 = tile * a.TS;
        const int n_s = (int)min((int64_t)a.TS, a.B - b0);
        __syncthreads();                                   // previous tile's readers are done with Fs / Ss
        attn_stage_tile(a, sd, b0, n_s, Fs, Es, true);
        cp_async_wait_all_();
        __syncthreads();
        {
            float acc[2][4];
            attn_hidden_mma(Fs, a.PF, Es, a.PE, smem + L.wrv_hi, smem + L.wrv_lo, smem + L.wid_hi, smem + L.wid_lo, a.Hp8, mt * 16, nh, lane, acc);
            float p0 = 0.f, p1 = 0.f;                      // logit partials of rows g and g + 8 over this warp's 16 units
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
                p0 = fmaf(fmaxf(acc[nt][0] + b1v[nt][0], 0.f), hv[nt][0], p0);
                p0 = fmaf(fmaxf(acc[nt][1] + b1v[nt][1], 0.f), hv[nt][1], p0);
                p1 = fmaf(fmaxf(acc[nt][2] + b1v[nt][0], 0.f), hv[nt][0], p1);
                p1 = fmaf(fmaxf(acc[nt][3] + b1v[nt][1], 0.f), hv[nt][1], p1);
            }
            p0 += __shfl_xor_sync(0xffffffffu, p0, 1); p0 += __shfl_xor_sync(0xffffffffu, p0, 2);
            p1 += __shfl_xor_sync(0xffffffffu, p1, 1); p1 += __shfl_xor_sync(0xffffffffu, p1, 2);
            if (t == 0) { Ls[nh * rows_pad + mt * 16 + g] = p0; Ls[nh * rows_pad + mt * 16 + g + 8] = p1; }
        }
        __syncthreads();
        // softmax over the R reviews of a sample (max-shifted, the reference's +1e-8 rescaled: finite where it overflows)
        if (threadIdx.x < n_s) {
            const int s = threadIdx.x;
            float m = -INFINITY;
            for (int r = 0; r < a.R; ++r) {
                const float lg = Ls[s * a.R + r] + Ls[rows_pad + s * a.R + r] + b2v;
                Ls[s * a.R + r] = lg;
                m = fmaxf(m, lg);
            }
            float sum = 0.f;
            for (int r = 0; r < a.R; ++r) { const float e = expf(Ls[s * a.R + r] - m); Ss[s * a.R + r] = e; sum += e; }
            const float inv = 1.f / (sum + 1e-8f * expf(-m));
            for (int r = 0; r < a.R; ++r) {
                const float sc = Ss[s * a.R + r] * inv;
                Ss[s * a.R + r] = sc;
                sd.scores[(b0 + s) * a.R + r] = sc;
            }
        }
        __syncthreads();
        // out[s, :] = sum_r score[s, r] * feat[s, r, :]      (one warp per sample, lanes across the features)
        for (int s = warp; s < n_s; s += (int)(blockDim.x >> 5)) {
            const float* fr = Fs + s * a.R * a.PF;
            const float* sc = Ss + s * a.R;
            for (int hcol = lane; hcol < a.H; hcol += 32) {
                float acc = 0.f;
                for (int r = 0; r < a.R; ++r) acc = fmaf(sc[r], fr[r * a.PF + hcol], acc);
                sd.out[(b0 + s) * a.H + hcol] = acc;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(2 * AT_MAXW * 32) narre_attn_tc_bwd_kernel(const AttnArgs a) {
    extern __shared__ __align__(16) float smem[];
    const AttnSide& sd = a.side[blockIdx.y];
    const AttnSmem L = attn_tc_smem(a, true);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
    const int mt = warp >> 1, nh = warp & 1, n_warps = (int)(blockDim.x >> 5);
    constexpr int pa = b_pitch(32);
    const int hcols = (a.Hp8 + 31) / 32 * 32, pht = b_pitch(hcols), n_hgroups = hcols / 32;
    stage_b_operand(smem + L.wrv_hi, smem + L.wrv_lo, sd.W_rv, a.H, a.Hp8, a.A, a.A, false);
    stage_b_operand(smem + L.wid_hi, smem + L.wid_lo, sd.W_id, a.A, 32, a.A, a.A, false);
    stage_b_operand(smem + L.widT_hi, smem + L.widT_lo, sd.W_id, a.A, 32, a.A, a.A, true);        // [k = a][n = a2] = W_id[a2][a]
    // W_rvᵀ as a B operand [k = a (32 rows)][n = h (hcols columns)]
    for (int k = warp; k < 32; k += n_warps)
        for (int n = lane; n < hcols; n += 32) {
            const float v = (k < a.A && n < a.H) ? __ldg(sd.W_rv + n * a.A + k) : 0.f;
            uint32_t h_, l_;
            split_hi_lo(v, h_, l_);
            const int idx = b_index(k, n, pht);
            smem[L.wrvT_hi + idx] = __uint_as_float(h_);
            smem[L.wrvT_lo + idx] = __uint_as_float(l_);
        }
    float* Fs = smem + L.F;
    float* Es = smem + L.E;
    float* Ls = smem + L.L;
    float* Ss = smem + L.S;
    float* GO = smem + L.GO;
    float* DHa = smem + L.DHa;
    float* DHb = smem + L.DHb;
    float* red = smem + L.red;
    float b1v[2][2], hv[2][2];
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int c = (2 * nh + nt) * 8 + 2 * t + j;
            b1v[nt][j] = c < a.A ? __ldg(sd.b1 + c) : 0.f;
            hv[nt][j] = c < a.A ? __ldg(sd.h + c) : 0.f;
        }
    // persistent partial parameter gradients of this thread
    float dh_p[2][2], db1_p[2][2], db2_p = 0.f;
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) { dh_p[nt][0] = dh_p[nt][1] = db1_p[nt][0] = db1_p[nt][1] = 0.f; }
    // dW_rv: tasks (m-tile of 16 feature rows h, column half) shared round-robin by the warps; dW_id: 2 m-tiles x 2 halves
    const int n_hm = (a.Hp8 + 15) / 16, n_tasks = 2 * n_hm;
    constexpr int MAX_WT = 4;
    float dwrv[MAX_WT][2][4];
    float dwid[2][4];
#pragma unroll
    for (int i = 0; i < MAX_WT; ++i)
#pragma unroll
        for (int nt = 0; nt < 2; ++nt)
#pragma unroll
            for (int j = 0; j < 4; ++j) dwrv[i][nt][j] = 0.f;
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
        for (int j = 0; j < 4; ++j) dwid[nt][j] = 0.f;
    const int rows_pad = a.NW * 16;

    const int64_t n_tiles = (a.B + a.TS - 1) / a.TS;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t b0 = tile * a.TS;
        const int n_s = (int)min((int64_t)a.TS, a.B - b0);
        const int rows_live = n_s * a.R;
        __syncthreads();
        attn_stage_tile(a, sd, b0, n_s, Fs, Es, false);
        stage_rows_async(GO, a.PF, a.TS, sd.out_grad + b0 * a.H, n_s, a.H);
        for (int i = threadIdx.x; i < rows_pad; i += blockDim.x) Ss[i] = i < rows_live ? __ldg(sd.scores + b0 * a.R + i) : 0.f;
        cp_async_wait_all_();
        __syncthreads();
        // ds[row] = out_grad[s] · feat[row] (+ scores_grad[row])
        for (int r = warp; r < rows_live; r += n_warps) {
            const float* go = GO + (r / a.R) * a.PF;
            const float* fr = Fs + r * a.PF;
            float p = 0.f;
            for (int c = lane; c < a.H; c += 32) p = fmaf(go[c], fr[c], p);
            p = warp_sum(p);
            if (lane == 0) Ls[r] = p + (sd.scores_grad ? __ldg(sd.scores_grad + b0 * a.R + r) : 0.f);
        }
        __syncthreads();
        // d logit[r] = score[r] * (ds[r] - sum_r' score[r'] ds[r'])
        if (threadIdx.x < n_s) {
            const int s = threadIdx.x;
            float dot = 0.f;
            for (int r = 0; r < a.R; ++r) dot = fmaf(Ls[s * a.R + r], Ss[s * a.R + r], dot);
            for (int r = 0; r < a.R; ++r) {
                const float dl = Ss[s * a.R + r] * (Ls[s * a.R + r] - dot);
                Ls[s * a.R + r] = dl;
                db2_p += dl;
            }
        } else if (threadIdx.x < a.TS) {
            for (int r = 0; r < a.R; ++r) Ls[threadIdx.x * a.R + r] = 0.f;
        }
        for (int i = a.TS * a.R + threadIdx.x; i < rows_pad; i += blockDim.x) Ls[i] = 0.f;
        __syncthreads();
        // recompute hid; d hid = (hid > 0) * dl[row] * h[a]  → DHa (A operand) and DHb (B operand); dh, db1 partials
        {
            float acc[2][4];
            const int m0 = mt * 16;
            attn_hidden_mma(Fs, a.PF, Es, a.PE, smem + L.wrv_hi, smem + L.wrv_lo, smem + L.wid_hi, smem + L.wid_lo, a.Hp8, m0, nh, lane, acc);
            const float dl0 = Ls[m0 + g], dl1 = Ls[m0 + g + 8];
#pragma unroll
            for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const int c = (2 * nh + nt) * 8 + 2 * t + j;
                    const float h0 = fmaxf(acc[nt][j] + b1v[nt][j], 0.f), h1 = fmaxf(acc[nt][2 + j] + b1v[nt][j], 0.f);
                    dh_p[nt][j] = fmaf(dl0, h0, fmaf(dl1, h1, dh_p[nt][j]));
                    const float d0 = h0 > 0.f ? dl0 * hv[nt][j] : 0.f, d1 = h1 > 0.f ? dl1 * hv[nt][j] : 0.f;
                    db1_p[nt][j] += d0 + d1;
                    DHa[(m0 + g) * 36 + c] = d0;
                    DHa[(m0 + g + 8) * 36 + c] = d1;
                    DHb[b_index(m0 + g, c, pa)] = d0;
                    DHb[b_index(m0 + g + 8, c, pa)] = d1;
                }
        }
        __syncthreads();
        // ---- d feat[rows, H] = score[row] * out_grad[s] + DH · W_rvᵀ      (M = the m-tile's 16 rows, N = H: the two warps of an
        //      m-tile take alternate groups of 32 columns, K = A)
        {
            const int m0 = mt * 16;
            uint32_t ahi[4][4], alo[4][4];
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
                const float* da = DHa + (m0 + g) * 36 + ks * 8 + t;
                split_hi_lo(da[0], ahi[ks][0], alo[ks][0]);
                split_hi_lo(da[8 * 36], ahi[ks][1], alo[ks][1]);
                split_hi_lo(da[4], ahi[ks][2], alo[ks][2]);
                split_hi_lo(da[8 * 36 + 4], ahi[ks][3], alo[ks][3]);
            }
            const int r0 = m0 + g, r1 = m0 + g + 8;
            const float sc0 = Ss[r0], sc1 = Ss[r1];
            const float* go0 = GO + (r0 / a.R) * a.PF;
            const float* go1 = GO + (r1 / a.R) * a.PF;
            float* dst0 = sd.feat_grad + (b0 * a.R + r0) * a.H;
            float* dst1 = sd.feat_grad + (b0 * a.R + r1) * a.H;
            for (int hg = nh; hg < n_hgroups; hg += 2) {
                float acc[4][4];
#pragma unroll
                for (int nt = 0; nt < 4; ++nt)
#pragma unroll
                    for (int i = 0; i < 4; ++i) acc[nt][i] = 0.f;
                const float* bb = smem + L.wrvT_hi + t * pht + hg * 40 + g * 4;
                const float* bl = smem + L.wrvT_lo + t * pht + hg * 40 + g * 4;
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
                    const float4 bh0 = *reinterpret_cast<const float4*>(bb + ks * 8 * pht), bh1 = *reinterpret_cast<const float4*>(bb + (ks * 8 + 4) * pht);
                    const float4 bl0 = *reinterpret_cast<const float4*>(bl + ks * 8 * pht), bl1 = *reinterpret_cast<const float4*>(bl + (ks * 8 + 4) * pht);
                    mma_3x(acc[0], ahi[ks], alo[ks], __float_as_uint(bh0.x), __float_as_uint(bh1.x), __float_as_uint(bl0.x), __float_as_uint(bl1.x));
                    mma_3x(acc[1], ahi[ks], alo[ks], __float_as_uint(bh0.y), __float_as_uint(bh1.y), __float_as_uint(bl0.y), __float_as_uint(bl1.y));
                    mma_3x(acc[2], ahi[ks], alo[ks], __float_as_uint(bh0.z), __float_as_uint(bh1.z), __float_as_uint(bl0.z), __float_as_uint(bl1.z));
                    mma_3x(acc[3], ahi[ks], alo[ks], __float_as_uint(bh0.w), __float_as_uint(bh1.w), __float_as_uint(bl0.w), __float_as_uint(bl1.w));
                }
#pragma unroll
                for (int nt = 0; nt < 4; ++nt) {
                    const int c = hg * 32 + nt * 8 + 2 * t;
                    if (c < a.H) {                                    // H even or odd: the pair is written element-wise
                        if (r0 < rows_live) {
                            dst0[c] = fmaf(sc0, go0[c], acc[nt][0]);
                            if (c + 1 < a.H) dst0[c + 1] = fmaf(sc0, go0[c + 1], acc[nt][1]);
                        }
                        if (r1 < rows_live) {
                            dst1[c] = fmaf(sc1, go1[c], acc[nt][2]);
                            if (c + 1 < a.H) dst1[c + 1] = fmaf(sc1, go1[c + 1], acc[nt][3]);
                        }
                    }
                }
            }
            // ---- d e[rows, A] = DH · W_idᵀ  (this warp's 16 columns) → id-embedding rows (atomics; padding row skipped)
            float acc[2][4];
#pragma unroll
            for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                for (int i = 0; i < 4; ++i) acc[nt][i] = 0.f;
            const float* bb = smem + L.widT_hi + t * pa + g * 4;
            const float* bl = smem + L.widT_lo + t * pa + g * 4;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
                const float4 bh0 = *reinterpret_cast<const float4*>(bb + ks * 8 * pa), bh1 = *reinterpret_cast<const float4*>(bb + (ks * 8 + 4) * pa);
                const float4 bl0 = *reinterpret_cast<const float4*>(bl + ks * 8 * pa), bl1 = *reinterpret_cast<const float4*>(bl + (ks * 8 + 4) * pa);
                mma_3x(acc[0], ahi[ks], alo[ks], __float_as_uint(sel0(bh0, nh)), __float_as_uint(sel0(bh1, nh)), __float_as_uint(sel0(bl0, nh)),
                       __float_as_uint(sel0(bl1, nh)));
                mma_3x(acc[1], ahi[ks], alo[ks], __float_as_uint(sel1(bh0, nh)), __float_as_uint(sel1(bh1, nh)), __float_as_uint(sel1(bl0, nh)),
                       __float_as_uint(sel1(bl1, nh)));
            }
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int r = half ? r1 : r0;
                if (r < rows_live) {
                    const int64_t id = __ldg(sd.other_id + b0 * a.R + r);
                    if (id >= 0 && id < sd.n_ids && id != sd.padding_idx) {
#pragma unroll
                        for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                            for (int j = 0; j < 2; ++j) {
                                const int c = (2 * nh + nt) * 8 + 2 * t + j;
                                const float v = acc[nt][half * 2 + j];
                                if (c < a.A && v != 0.f) atomicAdd(sd.ebd_grad + id * a.A + c, v);
                            }
                    }
                }
            }
        }
        // ---- dW_rv[h, a] += featᵀ · DH   (M = h, N = A, K = rows);  dW_id[a2, a] += eᵀ · DH
        {
#pragma unroll
            for (int sl = 0; sl < MAX_WT; ++sl) {                     // static slot index: dwrv stays in registers
                const int task = warp + sl * n_warps;
                if (task >= n_tasks) break;
                const int m0 = (task >> 1) * 16, th = task & 1;
                const bool in0 = m0 + g < a.Hp8, in1 = m0 + g + 8 < a.Hp8;
                const float* fa = Fs + t * a.PF + m0 + g;
                const float* db = DHb + t * pa + g * 4;
                for (int k0 = 0; k0 < rows_pad; k0 += 8, fa += 8 * a.PF, db += 8 * pa) {
                    // A[m = h][k = row] = F[row][h]   (transposed read of the feature tile)
                    uint32_t ahi[4], alo[4];
                    split_hi_lo(in0 ? fa[0] : 0.f, ahi[0], alo[0]);
                    split_hi_lo(in1 ? fa[8] : 0.f, ahi[1], alo[1]);
                    split_hi_lo(in0 ? fa[4 * a.PF] : 0.f, ahi[2], alo[2]);
                    split_hi_lo(in1 ? fa[4 * a.PF + 8] : 0.f, ahi[3], alo[3]);
                    const float4 b0v = *reinterpret_cast<const float4*>(db);
                    const float4 b1w = *reinterpret_cast<const float4*>(db + 4 * pa);
                    uint32_t bh0[2], bl0[2], bh1[2], bl1[2];
                    split_hi_lo(sel0(b0v, th), bh0[0], bl0[0]); split_hi_lo(sel1(b0v, th), bh0[1], bl0[1]);
                    split_hi_lo(sel0(b1w, th), bh1[0], bl1[0]); split_hi_lo(sel1(b1w, th), bh1[1], bl1[1]);
#pragma unroll
                    for (int nt = 0; nt < 2; ++nt) mma_3x(dwrv[sl][nt], ahi, alo, bh0[nt], bh1[nt], bl0[nt], bl1[nt]);
                }
            }
            if (warp < 4) {                                           // dW_id: m-tile = warp >> 1 (a2 rows), column half = warp & 1
                const int m0 = (warp >> 1) * 16, th = warp & 1;
                const float* ea = Es + t * a.PE + m0 + g;
                const float* db = DHb + t * pa + g * 4;
                for (int k0 = 0; k0 < rows_pad; k0 += 8, ea += 8 * a.PE, db += 8 * pa) {
                    uint32_t ahi[4], alo[4];
                    split_hi_lo(ea[0], ahi[0], alo[0]);
                    split_hi_lo(ea[8], ahi[1], alo[1]);
                    split_hi_lo(ea[4 * a.PE], ahi[2], alo[2]);
                    split_hi_lo(ea[4 * a.PE + 8], ahi[3], alo[3]);
                    const float4 b0v = *reinterpret_cast<const float4*>(db);
                    const float4 b1w = *reinterpret_cast<const float4*>(db + 4 * pa);
                    uint32_t bh0[2], bl0[2], bh1[2], bl1[2];
                    split_hi_lo(sel0(b0v, th), bh0[0], bl0[0]); split_hi_lo(sel1(b0v, th), bh0[1], bl0[1]);
                    split_hi_lo(sel0(b1w, th), bh1[0], bl1[0]); split_hi_lo(sel1(b1w, th), bh1[1], bl1[1]);
#pragma unroll
                    for (int nt = 0; nt < 2; ++nt) mma_3x(dwid[nt], ahi, alo, bh0[nt], bh1[nt], bl0[nt], bl1[nt]);
                }
            }
        }
    }
    // ---- flush the CTA's partial parameter gradients
    {
#pragma unroll
        for (int sl = 0; sl < MAX_WT; ++sl) {
            const int task = warp + sl * n_warps;
            if (task >= n_tasks) break;
            const int hm = task >> 1, th = task & 1;
#pragma unroll
            for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int hrow = hm * 16 + g + (j >> 1) * 8, c = (2 * th + nt) * 8 + 2 * t + (j & 1);
                    const float v = dwrv[sl][nt][j];
                    if (hrow < a.H && c < a.A && v != 0.f) atomicAdd(sd.W_rv_grad + hrow * a.A + c, v);
                }
        }
        if (warp < 4) {
            const int th = warp & 1;
#pragma unroll
            for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int arow = (warp >> 1) * 16 + g + (j >> 1) * 8, c = (2 * th + nt) * 8 + 2 * t + (j & 1);
                    const float v = dwid[nt][j];
                    if (arow < a.A && c < a.A && v != 0.f) atomicAdd(sd.W_id_grad + arow * a.A + c, v);
                }
        }
    }
    // dh / db1: reduce over the 8 row groups g (lanes with equal t), then over warps through shared memory
    __syncthreads();
    for (int i = threadIdx.x; i < 64; i += blockDim.x) red[i] = 0.f;
    if (threadIdx.x == 0) red[64] = 0.f;
    __syncthreads();
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            float vh = dh_p[nt][j], vb = db1_p[nt][j];
#pragma unroll
            for (int o = 4; o < 32; o <<= 1) { vh += __shfl_xor_sync(0xffffffffu, vh, o); vb += __shfl_xor_sync(0xffffffffu, vb, o); }
            if (g == 0) {
                const int c = (2 * nh + nt) * 8 + 2 * t + j;
                atomicAdd(red + c, vh);
                atomicAdd(red + 32 + c, vb);
            }
        }
    if (db2_p != 0.f) atomicAdd(red + 64, db2_p);
    __syncthreads();
    if (threadIdx.x < a.A) {
        if (red[threadIdx.x] != 0.f) atomicAdd(sd.h_grad + threadIdx.x, red[threadIdx.x]);
        if (red[32 + threadIdx.x] != 0.f) atomicAdd(sd.b1_grad + threadIdx.x, red[32 + threadIdx.x]);
    }
    if (threadIdx.x == 0 && red[64] != 0.f) atomicAdd(sd.b2_grad, red[64]);
}

static bool attn_tc_plan(int64_t B, int R, int H, int A, bool bwd, AttnArgs* a, size_t* smem_bytes) {
    if (A < 1 || A > 32 || R < 1 || R > 64 || H < 1 || H > 512) return false;
    a->B = B; a->R = R; a->H = H; a->A = A;
    a->Hp8 = (H + 7) & ~7;
    // samples per tile: as many as keep the tile within 80..128 review rows and 8 warps
    int ts = 80 / R;
    if (ts < 1) ts = 1;
    while ((ts * R + 15) / 16 > AT_MAXW) --ts;
    if (ts < 1) return false;
    a->TS = ts;
    a->rows = ts * R;
    a->NW = (a->rows + 15) / 16;
    // feature-tile pitch ≡ 4 (mod 32): conflict-free A-fragment reads (rows g, columns t)
    int pf = a->Hp8;
    while (pf % 32 != 4) ++pf;
    a->PF = pf;
    a->PE = 36;
    // dW_rv m-tiles per warp must fit the register budget
    if (((a->Hp8 + 15) / 16 + a->NW - 1) / a->NW > 4) return false;
    *smem_bytes = (size_t)attn_tc_smem(*a, bwd).total * 4;
    // forward: a smaller tile that lets TWO CTAs share an SM hides one CTA's tile load behind the other's math
    // (R = 10, H = 150: 6 samples / 107 KB instead of 8 / 122 KB — 89.9 -> 74.4 us; the backward does not fit twice either way)
    if (!bwd && *smem_bytes > 112 * 1024) {
        for (int t2 = ts - 1; t2 >= 1 && t2 * R >= 48; --t2) {
            AttnArgs b = *a;
            b.TS = t2; b.rows = t2 * R; b.NW = (b.rows + 15) / 16;
            if (((b.Hp8 + 15) / 16 + b.NW - 1) / b.NW > 4) break;
            const size_t sm = (size_t)attn_tc_smem(b, bwd).total * 4;
            if (sm <= 112 * 1024) { *a = b; *smem_bytes = sm; break; }
        }
    }
    return *smem_bytes <= 227 * 1024;
}

}  // namespace rbr

using namespace rbr;

static int attn_fill_side(AttnSide& s, const float* feat, const int64_t* other_id, const float* W_rv, const float* W_id, const float* h,
                          const float* b1, const float* b2, const float* ebd, int64_t n_ids) {
    s.feat = feat; s.other_id = other_id; s.W_rv = W_rv; s.W_id = W_id; s.h = h; s.b1 = b1; s.b2 = b2; s.ebd = ebd; s.n_ids = n_ids;
    return (feat && other_id && W_rv && W_id && h && b1 && b2 && ebd) ? RBR_OK : RBR_EINVAL;
}

extern "C" int rbr_narre_attn_pair_supported(int64_t reviews, int64_t hidden, int64_t att) {
    AttnArgs a{};
    size_t smem = 0;
    return attn_tc_plan(1, (int)reviews, (int)hidden, (int)att, true, &a, &smem) ? 1 : 0;
}

// Both sides' forward in one launch.  Arrays of 2 pointers per argument (side 0 = user reviews, side 1 = item reviews);
// n_sides may be 1.  Returns RBR_EUNSUPPORTED (no message) when the shape is outside this kernel: the caller falls back to K3.
extern "C" int rbr_narre_attn_pair_fwd(int n_sides, const float* const* feat, const int64_t* const* other_id, int64_t batch,
                                       int64_t reviews, int64_t hidden, int64_t att, const float* const* W_rv, const float* const* W_id,
                                       const float* const* h, const float* const* b_1, const float* const* b_2,
                                       const float* const* ebd_vals, const int64_t* n_ids, float* const* out, float* const* scores,
                                       void* stream) {
    RBR_REQUIRE(n_sides == 1 || n_sides == 2, RBR_EINVAL, "rbr_narre_attn_pair_fwd: n_sides must be 1 or 2");
    AttnArgs a{};
    size_t smem = 0;
    if (!attn_tc_plan(batch, (int)reviews, (int)hidden, (int)att, false, &a, &smem)) return RBR_EUNSUPPORTED;
    a.n_sides = n_sides;
    for (int s = 0; s < n_sides; ++s) {
        RBR_REQUIRE(attn_fill_side(a.side[s], feat[s], other_id[s], W_rv[s], W_id[s], h[s], b_1[s], b_2[s], ebd_vals[s], n_ids[s]) == RBR_OK &&
                        out[s] && scores[s],
                    RBR_EINVAL, "rbr_narre_attn_pair_fwd: null pointer");
        a.side[s].out = out[s]; a.side[s].scores = scores[s];
    }
    if (batch == 0) return RBR_OK;
    static bool attr = false;
    if (!attr) {
        RBR_CUDA(cudaFuncSetAttribute(narre_attn_tc_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        attr = true;
    }
    const int64_t n_tiles = (batch + a.TS - 1) / a.TS;
    const int64_t per_side = (2 * 148) / n_sides / (smem > 112 * 1024 ? 2 : 1);   // persistent CTAs: all co-resident
    int64_t gx = n_tiles < per_side ? n_tiles : per_side;
    dim3 grid((unsigned)gx, (unsigned)n_sides);
    narre_attn_tc_fwd_kernel<<<grid, 2 * a.NW * 32, smem, as_stream(stream)>>>(a);
    RBR_LAUNCH_CHECK("narre_attn_tc_fwd_kernel");
    return RBR_OK;
}

extern "C" int rbr_narre_attn_pair_bwd(int n_sides, const float* const* feat, const int64_t* const* other_id, int64_t batch,
                                       int64_t reviews, int64_t hidden, int64_t att, const float* const* W_rv, const float* const* W_id,
                                       const float* const* h, const float* const* b_1, const float* const* b_2,
                                       const float* const* ebd_vals, const int64_t* n_ids, const int64_t* padding_idx,
                                       const float* const* scores, const float* const* out_grad, const float* const* scores_grad,
                                       float* const* feat_grad, float* const* W_rv_grad, float* const* W_id_grad, float* const* h_grad,
                                       float* const* b_1_grad, float* const* b_2_grad, float* const* ebd_vals_grad, void* stream) {
    RBR_REQUIRE(n_sides == 1 || n_sides == 2, RBR_EINVAL, "rbr_narre_attn_pair_bwd: n_sides must be 1 or 2");
    AttnArgs a{};
    size_t smem = 0;
    if (!attn_tc_plan(batch, (int)reviews, (int)hidden, (int)att, true, &a, &smem)) return RBR_EUNSUPPORTED;
    a.n_sides = n_sides;
    for (int s = 0; s < n_sides; ++s) {
        RBR_REQUIRE(attn_fill_side(a.side[s], feat[s], other_id[s], W_rv[s], W_id[s], h[s], b_1[s], b_2[s], ebd_vals[s], n_ids[s]) == RBR_OK &&
                        scores[s] && out_grad[s] && feat_grad[s] && W_rv_grad[s] && W_id_grad[s] && h_grad[s] && b_1_grad[s] &&
                        b_2_grad[s] && ebd_vals_grad[s],
                    RBR_EINVAL, "rbr_narre_attn_pair_bwd: null pointer");
        AttnSide& sd = a.side[s];
        sd.padding_idx = padding_idx[s];
        sd.scores = const_cast<float*>(scores[s]);
        sd.out_grad = out_grad[s];
        sd.scores_grad = scores_grad ? scores_grad[s] : nullptr;
        sd.feat_grad = feat_grad[s]; sd.W_rv_grad = W_rv_grad[s]; sd.W_id_grad = W_id_grad[s]; sd.h_grad = h_grad[s];
        sd.b1_grad = b_1_grad[s]; sd.b2_grad = b_2_grad[s]; sd.ebd_grad = ebd_vals_grad[s];
    }
    if (batch == 0) return RBR_OK;
    static bool attr = false;
    if (!attr) {
        RBR_CUDA(cudaFuncSetAttribute(narre_attn_tc_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        attr = true;
    }
    const int64_t n_tiles = (batch + a.TS - 1) / a.TS;
    const int64_t per_side = 148 / n_sides;                           // one CTA per SM (232 registers per thread), all co-resident
    int64_t gx = n_tiles < per_side ? n_tiles : per_side;
    dim3 grid((unsigned)gx, (unsigned)n_sides);
    narre_attn_tc_bwd_kernel<<<grid, 2 * a.NW * 32, smem, as_stream(stream)>>>(a);
    RBR_LAUNCH_CHECK("narre_attn_tc_bwd_kernel");
    return RBR_OK;
}

RBR_DEFINE_OOB_ACCESSOR(attn_tc)
