// head.cu — K4: fused LastFeat (user + item) + FM interaction + MSE loss, forward and backward.
//
// Replaces, per mini-batch, LastFeat.forward x2 (reference models/deepconn/layers.py:156-165: text_feat @ W + b +
// ebd(id)), FM.forward (layers.py:188-209: relu(u*i) → dropout → @h + user_bias(id) + item_bias(id) + g_bias) and
// nn.MSELoss (trainer/train_deepconn_pp.py:140,164) — about ten cuBLAS/elementwise launches in the reference.
// Latency/HBM-bound: ~1 KB per sample.  One warp per sample; lane = latent dimension.
#include "rbr_common.cuh"

namespace rbr {

constexpr int HD_KQ = 4;          // latent dim <= 128
constexpr int HD_WARPS = 8;
constexpr int HD_BS = 32;         // samples per CTA iteration in the backward

__device__ __forceinline__ float keep_scale(float p, uint64_t seed, int64_t b, int K, int kk) {
    if (p <= 0.f) return 1.f;
    return hash_uniform(seed, (uint64_t)b * (uint64_t)K + (uint64_t)kk) >= p ? 1.f / (1.f - p) : 0.f;
}

// smem weight copy with row stride K+1 (conflict-free both for lane=k and for lane=h access)
__device__ __forceinline__ void stage_weight(float* dst, const float* __restrict__ src, int H, int K) {
    for (int i = threadIdx.x; i < H * K; i += blockDim.x) dst[(i / K) * (K + 1) + (i % K)] = src[i];
}

__global__ void __launch_bounds__(HD_WARPS * 32) head_fwd_kernel(
    const float* __restrict__ u_text, const float* __restrict__ i_text, const int64_t* __restrict__ u_id,
    const int64_t* __restrict__ i_id, int64_t B, int H, int K, const float* __restrict__ Wu, const float* __restrict__ bu,
    const float* __restrict__ ebd_u, const float* __restrict__ Wi, const float* __restrict__ bi, const float* __restrict__ ebd_i,
    const float* __restrict__ fm_h, const float* __restrict__ user_bias, const float* __restrict__ item_bias,
    const float* __restrict__ g_bias, int64_t users, int64_t items, float drop_p, uint64_t drop_seed,
    const uint64_t* __restrict__ drop_seed_dev, float* __restrict__ pred, float* __restrict__ u_lat, float* __restrict__ i_lat,
    const float* __restrict__ ratings, float grad_scale, float* __restrict__ loss_sum, float* __restrict__ pred_grad) {
    if (drop_seed_dev) drop_seed += *drop_seed_dev;          // device-resident step counter (CUDA-graph replay varies the mask)
    extern __shared__ __align__(16) float smem[];
    float* Wu_s = smem;
    float* Wi_s = smem + H * (K + 1);
    float* xrow = Wi_s + H * (K + 1);                 // [HD_WARPS][2][H] text rows of the warp's current sample
    stage_weight(Wu_s, Wu, H, K);
    stage_weight(Wi_s, Wi, H, K);
    __syncthreads();
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    float* xu = xrow + (wib * 2) * H;
    float* xi = xu + H;
    const float gb = g_bias[0];
    float loss_acc = 0.f;
    for (int64_t b = (int64_t)blockIdx.x * HD_WARPS + wib; b < B; b += (int64_t)gridDim.x * HD_WARPS) {
        for (int h = lane; h < H; h += 32) { xu[h] = u_text[b * H + h]; xi[h] = i_text[b * H + h]; }
        __syncwarp();
        int64_t uid = u_id[b], iid = i_id[b];
        const bool u_ok = uid >= 0 && uid < users, i_ok = iid >= 0 && iid < items;
        if (lane == 0 && (!u_ok || !i_ok)) note_oob();
        float part = 0.f;
#pragma unroll
        for (int q = 0; q < HD_KQ; ++q) {
            const int kk = lane + 32 * q;
            if (kk < K) {
                float su = 0.f, si = 0.f;
                for (int h = 0; h < H; ++h) {
                    su = fmaf(xu[h], Wu_s[h * (K + 1) + kk], su);
                    si = fmaf(xi[h], Wi_s[h * (K + 1) + kk], si);
                }
                // reference order: (text @ W + b) + ebd  (layers.py:163)
                const float ul = (su + bu[kk]) + (u_ok ? ebd_u[uid * K + kk] : 0.f);
                const float il = (si + bi[kk]) + (i_ok ? ebd_i[iid * K + kk] : 0.f);
                u_lat[b * K + kk] = ul;
                i_lat[b * K + kk] = il;
                const float fm = fmaxf(ul * il, 0.f) * keep_scale(drop_p, drop_seed, b, K, kk);
                part = fmaf(fm, fm_h[kk], part);
            }
        }
        part = warp_sum(part);
        if (lane == 0) {
            const float p = part + (u_ok ? user_bias[uid] : 0.f) + (i_ok ? item_bias[iid] : 0.f) + gb;
            pred[b] = p;
            if (ratings) {
                const float d = p - ratings[b];
                loss_acc = fmaf(d, d, loss_acc);
                if (pred_grad) pred_grad[b] = 2.f * d * grad_scale;
            }
        }
        __syncwarp();
    }
    if (ratings && loss_sum && lane == 0 && loss_acc != 0.f) atomicAdd(loss_sum, loss_acc * grad_scale);
}

__global__ void __launch_bounds__(HD_WARPS * 32) head_bwd_kernel(
    const float* __restrict__ u_text, const float* __restrict__ i_text, const int64_t* __restrict__ u_id,
    const int64_t* __restrict__ i_id, int64_t B, int H, int K, const float* __restrict__ Wu, const float* __restrict__ Wi,
    const float* __restrict__ fm_h, const float* __restrict__ u_lat, const float* __restrict__ i_lat, float drop_p,
    uint64_t drop_seed, const uint64_t* __restrict__ drop_seed_dev, int64_t pad_eu, int64_t pad_ei, int64_t pad_bu, int64_t pad_bi,
    int64_t users, int64_t items, const float* __restrict__ pred_grad,
    float* __restrict__ u_text_grad, float* __restrict__ i_text_grad, float* __restrict__ Wu_grad, float* __restrict__ bu_grad,
    float* __restrict__ ebd_u_grad, float* __restrict__ Wi_grad, float* __restrict__ bi_grad, float* __restrict__ ebd_i_grad,
    float* __restrict__ fm_h_grad, float* __restrict__ user_bias_grad, float* __restrict__ item_bias_grad,
    float* __restrict__ g_bias_grad) {
    if (drop_seed_dev) drop_seed += *drop_seed_dev;
    extern __shared__ __align__(16) float smem[];
    const int KS = K + 1;
    float* Wu_s = smem;                          // [H][K+1]
    float* Wi_s = Wu_s + H * KS;
    float* dWu_s = Wi_s + H * KS;                // [H][K]   CTA-partial weight grads (owner-exclusive updates)
    float* dWi_s = dWu_s + H * K;
    float* xu_s = dWi_s + H * K;                 // [HD_BS][H]
    float* xi_s = xu_s + HD_BS * H;
    float* du_s = xi_s + HD_BS * H;              // [HD_BS][K]
    float* di_s = du_s + HD_BS * K;
    stage_weight(Wu_s, Wu, H, K);
    stage_weight(Wi_s, Wi, H, K);
    for (int i = threadIdx.x; i < 2 * H * K; i += blockDim.x) dWu_s[i] = 0.f;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    float dbu[HD_KQ], dbi[HD_KQ], dfh[HD_KQ];
#pragma unroll
    for (int q = 0; q < HD_KQ; ++q) dbu[q] = dbi[q] = dfh[q] = 0.f;
    float dgb = 0.f;
    __syncthreads();

    for (int64_t b0 = (int64_t)blockIdx.x * HD_BS; b0 < B; b0 += (int64_t)gridDim.x * HD_BS) {
        const int nb = (int)min((int64_t)HD_BS, B - b0);
        // ---- phase 1: per-sample latent gradients (one warp per sample, HD_BS/HD_WARPS samples per warp)
        for (int s = wib; s < HD_BS; s += HD_WARPS) {
            const int64_t b = b0 + s;
            if (s < nb) {
                for (int h = lane; h < H; h += 32) { xu_s[s * H + h] = u_text[b * H + h]; xi_s[s * H + h] = i_text[b * H + h]; }
                const float gp = pred_grad[b];
                const int64_t uid = u_id[b], iid = i_id[b];
                const bool u_ok = uid >= 0 && uid < users, i_ok = iid >= 0 && iid < items;
                const bool u_row = u_ok && uid != pad_eu, i_row = i_ok && iid != pad_ei;        // LastFeat.ebd padding rows
                const bool ub_row = u_ok && uid != pad_bu, ib_row = i_ok && iid != pad_bi;      // FM.user_bias / item_bias padding rows
#pragma unroll
                for (int q = 0; q < HD_KQ; ++q) {
                    const int kk = lane + 32 * q;
                    if (kk < K) {
                        const float ul = u_lat[b * K + kk], il = i_lat[b * K + kk];
                        const float prod = ul * il;
                        const float ks = keep_scale(drop_p, drop_seed, b, K, kk);
                        const float dfm = (prod > 0.f) ? gp * fm_h[kk] * ks : 0.f;
                        const float du = dfm * il, di = dfm * ul;
                        du_s[s * K + kk] = du;
                        di_s[s * K + kk] = di;
                        dbu[q] += du; dbi[q] += di;
                        dfh[q] = fmaf(fmaxf(prod, 0.f) * ks, gp, dfh[q]);
                        if (u_row && du != 0.f) atomicAdd(ebd_u_grad + uid * K + kk, du);
                        if (i_row && di != 0.f) atomicAdd(ebd_i_grad + iid * K + kk, di);
                    }
                }
                if (lane == 0) {
                    dgb += gp;
                    if (ub_row) atomicAdd(user_bias_grad + uid, gp);
                    if (ib_row) atomicAdd(item_bias_grad + iid, gp);
                }
            } else {
                for (int h = lane; h < H; h += 32) { xu_s[s * H + h] = 0.f; xi_s[s * H + h] = 0.f; }
                for (int kk = lane; kk < K; kk += 32) { du_s[s * K + kk] = 0.f; di_s[s * K + kk] = 0.f; }
            }
        }
        __syncthreads();
        // ---- phase 2a: text-feature gradients  d_text[b,h] = sum_k d_lat[b,k] * W[h,k]
        for (int o = threadIdx.x; o < nb * H; o += blockDim.x) {
            const int s = o / H, h = o - s * H;
            float au = 0.f, ai = 0.f;
            for (int kk = 0; kk < K; ++kk) {
                au = fmaf(du_s[s * K + kk], Wu_s[h * KS + kk], au);
                ai = fmaf(di_s[s * K + kk], Wi_s[h * KS + kk], ai);
            }
            u_text_grad[(b0 + s) * H + h] = au;
            i_text_grad[(b0 + s) * H + h] = ai;
        }
        // ---- phase 2b: weight gradients  dW[h,k] += sum_b text[b,h] * d_lat[b,k]   (thread owns (h,k))
        for (int o = threadIdx.x; o < H * K; o += blockDim.x) {
            const int h = o / K, kk = o - h * K;
            float au = 0.f, ai = 0.f;
#pragma unroll 8
            for (int s = 0; s < HD_BS; ++s) {
                au = fmaf(xu_s[s * H + h], du_s[s * K + kk], au);
                ai = fmaf(xi_s[s * H + h], di_s[s * K + kk], ai);
            }
            dWu_s[o] += au;
            dWi_s[o] += ai;
        }
        __syncthreads();
    }
    // ---- flush CTA partials
    for (int o = threadIdx.x; o < H * K; o += blockDim.x) {
        if (dWu_s[o] != 0.f) atomicAdd(Wu_grad + o, dWu_s[o]);
        if (dWi_s[o] != 0.f) atomicAdd(Wi_grad + o, dWi_s[o]);
    }
#pragma unroll
    for (int q = 0; q < HD_KQ; ++q) {
        const int kk = lane + 32 * q;
        if (kk < K) {
            if (dbu[q] != 0.f) atomicAdd(bu_grad + kk, dbu[q]);
            if (dbi[q] != 0.f) atomicAdd(bi_grad + kk, dbi[q]);
            if (dfh[q] != 0.f) atomicAdd(fm_h_grad + kk, dfh[q]);
        }
    }
    if (lane == 0 && dgb != 0.f) atomicAdd(g_bias_grad, dgb);
}

// ------------------------------------------------------------------------------------------------------------------
// Register-tiled versions (latent % 4 == 0, hidden % 4 == 0, 16-byte aligned operands): a CTA owns HD2_TS consecutive
// samples, a warp 4 of them, a lane one latent column (forward, weight gradient) or one text column (text gradient).  Every
// shared-memory operand is read once per 4 FMAs (float4 over the contraction index, broadcast across the warp), which takes
// the kernels from ~3 to ~1.5 instructions per FMA — they were bound by instruction latency with 2 warps per scheduler, not by
// memory (ncu: issue active 26 %, DRAM 2 %).  The accumulation order of every sum is that of the kernels above: same bits.
// ------------------------------------------------------------------------------------------------------------------
// NW warps per CTA, 4 samples per warp: a CTA tile is 4 NW consecutive samples.  Text rows sit in shared memory with a row
// stride of Hp = round_up(H, 4) floats (pad columns and weight rows H .. Hp-1 are zero), so hidden need not be a multiple of 4.
__device__ __forceinline__ void stage_f4(float* dst, const float* __restrict__ src, int n_floats) {
    const float4* s4 = reinterpret_cast<const float4*>(src);
    float4* d4 = reinterpret_cast<float4*>(dst);
    for (int i = threadIdx.x; i < (n_floats >> 2); i += blockDim.x) d4[i] = __ldg(s4 + i);
}
// [rows][H] global → [rows_total][Hp] shared, zero-filling the pad columns and the rows >= rows
__device__ __forceinline__ void stage_rows(float* dst, const float* __restrict__ src, int rows, int rows_total, int H, int Hp, bool vec) {
    if (vec && H == Hp) {
        stage_f4(dst, src, rows * H);
        for (int i = rows * H + threadIdx.x; i < rows_total * H; i += blockDim.x) dst[i] = 0.f;
    } else {
        const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
        for (int r = w; r < rows_total; r += nw)
            for (int c = lane; c < Hp; c += 32) dst[r * Hp + c] = (r < rows && c < H) ? __ldg(src + r * H + c) : 0.f;
    }
}

template <int NW>
__global__ void __launch_bounds__(NW * 32) head_fwd2_kernel(
    const float* __restrict__ u_text, const float* __restrict__ i_text, const int64_t* __restrict__ u_id,
    const int64_t* __restrict__ i_id, int64_t B, int H, int K, const float* __restrict__ Wu, const float* __restrict__ bu,
    const float* __restrict__ ebd_u, const float* __restrict__ Wi, const float* __restrict__ bi, const float* __restrict__ ebd_i,
    const float* __restrict__ fm_h, const float* __restrict__ user_bias, const float* __restrict__ item_bias,
    const float* __restrict__ g_bias, int64_t users, int64_t items, float drop_p, uint64_t drop_seed,
    const uint64_t* __restrict__ drop_seed_dev, float* __restrict__ pred, float* __restrict__ u_lat, float* __restrict__ i_lat,
    const float* __restrict__ ratings, float grad_scale, float* __restrict__ loss_sum, float* __restrict__ pred_grad, int vec) {
    constexpr int TS = 4 * NW;
    if (drop_seed_dev) drop_seed += *drop_seed_dev;
    extern __shared__ __align__(16) float smem[];
    const int Hp = (H + 3) & ~3;
    float* Wu_s = smem;                                // [Hp][K]
    float* Wi_s = Wu_s + Hp * K;
    float* xu_s = Wi_s + Hp * K;                       // [TS][Hp]
    float* xi_s = xu_s + TS * Hp;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    stage_rows(Wu_s, Wu, H, Hp, K, K, vec != 0);
    stage_rows(Wi_s, Wi, H, Hp, K, K, vec != 0);
    const float gb = g_bias[0];
    float loss_acc = 0.f;
    for (int64_t b0 = (int64_t)blockIdx.x * TS; b0 < B; b0 += (int64_t)gridDim.x * TS) {
        const int nb = (int)min((int64_t)TS, B - b0);
        __syncthreads();                               // previous tile consumed
        stage_rows(xu_s, u_text + b0 * H, nb, TS, H, Hp, vec != 0);
        stage_rows(xi_s, i_text + b0 * H, nb, TS, H, Hp, vec != 0);
        // this warp's 4 samples: ids, then (lane = latent column) the embedding rows of the first 32 columns — fetched while the
        // tile is staged and multiplied, not after
        int64_t uid[4], iid[4];
        bool u_ok[4], i_ok[4];
        float eu0[4], ei0[4];
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            const int64_t b = b0 + wib * 4 + s;
            uid[s] = iid[s] = 0;
            u_ok[s] = i_ok[s] = false;
            if (b < B) {
                uid[s] = u_id[b]; iid[s] = i_id[b];
                u_ok[s] = uid[s] >= 0 && uid[s] < users;
                i_ok[s] = iid[s] >= 0 && iid[s] < items;
                if (lane == 0 && (!u_ok[s] || !i_ok[s])) note_oob();
            }
        }
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            eu0[s] = (u_ok[s] && lane < K) ? ebd_u[uid[s] * K + lane] : 0.f;
            ei0[s] = (i_ok[s] && lane < K) ? ebd_i[iid[s] * K + lane] : 0.f;
        }
        __syncthreads();
        float part[4] = {0.f, 0.f, 0.f, 0.f};         // per-lane partial of each sample's FM sum (columns lane, lane + 32, ...)
        for (int k0 = 0; k0 < K; k0 += 32) {
            const int kk = k0 + lane;
            const int kc = kk < K ? kk : K - 1;        // clamped column for the loads; results of kk >= K are dropped
            float su[4] = {0.f, 0.f, 0.f, 0.f}, si[4] = {0.f, 0.f, 0.f, 0.f};
            const float* xu_w = xu_s + (wib * 4) * Hp;
            const float* xi_w = xi_s + (wib * 4) * Hp;
            for (int h = 0; h < Hp; h += 4) {
                float wu[4], wi[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) { wu[j] = Wu_s[(h + j) * K + kc]; wi[j] = Wi_s[(h + j) * K + kc]; }
#pragma unroll
                for (int s = 0; s < 4; ++s) {
                    const float4 a = *reinterpret_cast<const float4*>(xu_w + s * Hp + h);
                    const float4 c = *reinterpret_cast<const float4*>(xi_w + s * Hp + h);
                    su[s] = fmaf(a.x, wu[0], su[s]); su[s] = fmaf(a.y, wu[1], su[s]); su[s] = fmaf(a.z, wu[2], su[s]); su[s] = fmaf(a.w, wu[3], su[s]);
                    si[s] = fmaf(c.x, wi[0], si[s]); si[s] = fmaf(c.y, wi[1], si[s]); si[s] = fmaf(c.z, wi[2], si[s]); si[s] = fmaf(c.w, wi[3], si[s]);
                }
            }
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                const int64_t b = b0 + wib * 4 + s;
                if (b < B && kk < K) {
                    const float eu = k0 == 0 ? eu0[s] : (u_ok[s] ? ebd_u[uid[s] * K + kk] : 0.f);
                    const float ei = k0 == 0 ? ei0[s] : (i_ok[s] ? ebd_i[iid[s] * K + kk] : 0.f);
                    // reference order: (text @ W + b) + ebd  (layers.py:163)
                    const float ul = (su[s] + bu[kk]) + eu;
                    const float il = (si[s] + bi[kk]) + ei;
                    u_lat[b * K + kk] = ul;
                    i_lat[b * K + kk] = il;
                    const float fm = fmaxf(ul * il, 0.f) * keep_scale(drop_p, drop_seed, b, K, kk);
                    part[s] = fmaf(fm, fm_h[kk], part[s]);
                }
            }
        }
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            const int64_t b = b0 + wib * 4 + s;
            const float tot = warp_sum(part[s]);
            if (lane == 0 && b < B) {
                const float pv = tot + (u_ok[s] ? user_bias[uid[s]] : 0.f) + (i_ok[s] ? item_bias[iid[s]] : 0.f) + gb;
                pred[b] = pv;
                if (ratings) {
                    const float d = pv - ratings[b];
                    loss_acc = fmaf(d, d, loss_acc);
                    if (pred_grad) pred_grad[b] = 2.f * d * grad_scale;
                }
            }
        }
    }
    if (ratings && loss_sum && lane == 0 && loss_acc != 0.f) atomicAdd(loss_sum, loss_acc * grad_scale);
}

template <int NW>
__global__ void __launch_bounds__(NW * 32) head_bwd2_kernel(
    const float* __restrict__ u_text, const float* __restrict__ i_text, const int64_t* __restrict__ u_id,
    const int64_t* __restrict__ i_id, int64_t B, int H, int K, const float* __restrict__ Wu, const float* __restrict__ Wi,
    const float* __restrict__ fm_h, const float* __restrict__ u_lat, const float* __restrict__ i_lat, float drop_p,
    uint64_t drop_seed, const uint64_t* __restrict__ drop_seed_dev, int64_t pad_eu, int64_t pad_ei, int64_t pad_bu, int64_t pad_bi,
    int64_t users, int64_t items, const float* __restrict__ pred_grad,
    float* __restrict__ u_text_grad, float* __restrict__ i_text_grad, float* __restrict__ Wu_grad, float* __restrict__ bu_grad,
    float* __restrict__ ebd_u_grad, float* __restrict__ Wi_grad, float* __restrict__ bi_grad, float* __restrict__ ebd_i_grad,
    float* __restrict__ fm_h_grad, float* __restrict__ user_bias_grad, float* __restrict__ item_bias_grad,
    float* __restrict__ g_bias_grad, int vec) {
    constexpr int TS = 4 * NW;
    if (drop_seed_dev) drop_seed += *drop_seed_dev;
    extern __shared__ __align__(16) float smem[];
    const int KS = K + 1;                        // padded weight rows: conflict-free for lane = text column
    const int Hp = (H + 3) & ~3;
    float* Wu_s = smem;                          // [H][K+1]
    float* Wi_s = Wu_s + H * KS;
    float* xu_s = Wi_s + H * KS;                 // [TS][Hp]
    xu_s += (4 - ((2 * H * KS) & 3)) & 3;        // keep the float4 views below 16-byte aligned
    float* xi_s = xu_s + TS * Hp;
    float* du_s = xi_s + TS * Hp;                // [TS][K]
    float* di_s = du_s + TS * K;
    stage_weight(Wu_s, Wu, H, K);
    stage_weight(Wi_s, Wi, H, K);
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    float dbu[HD_KQ], dbi[HD_KQ], dfh[HD_KQ];
#pragma unroll
    for (int q = 0; q < HD_KQ; ++q) dbu[q] = dbi[q] = dfh[q] = 0.f;
    float dgb = 0.f;

    for (int64_t b0 = (int64_t)blockIdx.x * TS; b0 < B; b0 += (int64_t)gridDim.x * TS) {
        const int nb = (int)min((int64_t)TS, B - b0);
        __syncthreads();
        stage_rows(xu_s, u_text + b0 * H, nb, TS, H, Hp, vec != 0);
        stage_rows(xi_s, i_text + b0 * H, nb, TS, H, Hp, vec != 0);
        // ---- phase 1: per-sample latent gradients (warp = 4 samples, lane = latent column)
#pragma unroll
        for (int ss = 0; ss < 4; ++ss) {
            const int s = wib * 4 + ss;
            const int64_t b = b0 + s;
            if (s < nb) {
                const float gp = pred_grad[b];
                const int64_t uid = u_id[b], iid = i_id[b];
                const bool u_ok = uid >= 0 && uid < users, i_ok = iid >= 0 && iid < items;
                const bool u_row = u_ok && uid != pad_eu, i_row = i_ok && iid != pad_ei;        // LastFeat.ebd padding rows
                const bool ub_row = u_ok && uid != pad_bu, ib_row = i_ok && iid != pad_bi;      // FM.user_bias / item_bias padding rows
#pragma unroll
                for (int q = 0; q < HD_KQ; ++q) {
                    const int kk = lane + 32 * q;
                    if (kk < K) {
                        const float ul = u_lat[b * K + kk], il = i_lat[b * K + kk];
                        const float prod = ul * il;
                        const float ks = keep_scale(drop_p, drop_seed, b, K, kk);
                        const float dfm = (prod > 0.f) ? gp * fm_h[kk] * ks : 0.f;
                        const float du = dfm * il, di = dfm * ul;
                        du_s[s * K + kk] = du;
                        di_s[s * K + kk] = di;
                        dbu[q] += du; dbi[q] += di;
                        dfh[q] = fmaf(fmaxf(prod, 0.f) * ks, gp, dfh[q]);
                        if (u_row && du != 0.f) atomicAdd(ebd_u_grad + uid * K + kk, du);
                        if (i_row && di != 0.f) atomicAdd(ebd_i_grad + iid * K + kk, di);
                    }
                }
                if (lane == 0) {
                    dgb += gp;
                    if (ub_row) atomicAdd(user_bias_grad + uid, gp);
                    if (ib_row) atomicAdd(item_bias_grad + iid, gp);
                }
            } else {
                for (int kk = lane; kk < K; kk += 32) { du_s[s * K + kk] = 0.f; di_s[s * K + kk] = 0.f; }
            }
        }
        __syncthreads();
        // ---- phase 2a: text-feature gradients  d_text[b,h] = sum_k d_lat[b,k] * W[h,k]   (warp = its 4 samples, lane = text column)
        for (int h0 = 0; h0 < H; h0 += 32) {
            const int h = h0 + lane;
            const int hc = h < H ? h : H - 1;
            float au[4] = {0.f, 0.f, 0.f, 0.f}, ai[4] = {0.f, 0.f, 0.f, 0.f};
            const float* wu = Wu_s + hc * KS;
            const float* wi = Wi_s + hc * KS;
            for (int kk = 0; kk < K; kk += 4) {
                const float w0 = wu[kk], w1 = wu[kk + 1], w2 = wu[kk + 2], w3 = wu[kk + 3];
                const float v0 = wi[kk], v1 = wi[kk + 1], v2 = wi[kk + 2], v3 = wi[kk + 3];
#pragma unroll
                for (int ss = 0; ss < 4; ++ss) {
                    const float4 a = *reinterpret_cast<const float4*>(du_s + (wib * 4 + ss) * K + kk);
                    const float4 c = *reinterpret_cast<const float4*>(di_s + (wib * 4 + ss) * K + kk);
                    au[ss] = fmaf(a.x, w0, au[ss]); au[ss] = fmaf(a.y, w1, au[ss]); au[ss] = fmaf(a.z, w2, au[ss]); au[ss] = fmaf(a.w, w3, au[ss]);
                    ai[ss] = fmaf(c.x, v0, ai[ss]); ai[ss] = fmaf(c.y, v1, ai[ss]); ai[ss] = fmaf(c.z, v2, ai[ss]); ai[ss] = fmaf(c.w, v3, ai[ss]);
                }
            }
            if (h < H) {
#pragma unroll
                for (int ss = 0; ss < 4; ++ss) {
                    const int s = wib * 4 + ss;
                    if (s < nb) {
                        u_text_grad[(b0 + s) * H + h] = au[ss];
                        i_text_grad[(b0 + s) * H + h] = ai[ss];
                    }
                }
            }
        }
        // ---- phase 2b: weight gradients  dW[h,k] += sum_b text[b,h] * d_lat[b,k]   (lane = latent column, warp walks groups of 4 text
        //      columns; the tile's partial goes straight to the global gradient)
        for (int k0 = 0; k0 < K; k0 += 32) {
            const int kk = k0 + lane;
            const int kc = kk < K ? kk : K - 1;
            for (int hg = wib; hg < (Hp >> 2); hg += NW) {
                const int h = hg * 4;
                float au[4] = {0.f, 0.f, 0.f, 0.f}, ai[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 8
                for (int s = 0; s < TS; ++s) {
                    const float4 a = *reinterpret_cast<const float4*>(xu_s + s * Hp + h);
                    const float4 c = *reinterpret_cast<const float4*>(xi_s + s * Hp + h);
                    const float du = du_s[s * K + kc], di = di_s[s * K + kc];
                    au[0] = fmaf(a.x, du, au[0]); au[1] = fmaf(a.y, du, au[1]); au[2] = fmaf(a.z, du, au[2]); au[3] = fmaf(a.w, du, au[3]);
                    ai[0] = fmaf(c.x, di, ai[0]); ai[1] = fmaf(c.y, di, ai[1]); ai[2] = fmaf(c.z, di, ai[2]); ai[3] = fmaf(c.w, di, ai[3]);
                }
                if (kk < K) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        if (h + j < H) {
                            if (au[j] != 0.f) atomicAdd(Wu_grad + (h + j) * K + kk, au[j]);
                            if (ai[j] != 0.f) atomicAdd(Wi_grad + (h + j) * K + kk, ai[j]);
                        }
                    }
                }
            }
        }
    }
    // ---- flush per-thread partials
#pragma unroll
    for (int q = 0; q < HD_KQ; ++q) {
        const int kk = lane + 32 * q;
        if (kk < K) {
            if (dbu[q] != 0.f) atomicAdd(bu_grad + kk, dbu[q]);
            if (dbi[q] != 0.f) atomicAdd(bi_grad + kk, dbi[q]);
            if (dfh[q] != 0.f) atomicAdd(fm_h_grad + kk, dfh[q]);
        }
    }
    if (lane == 0 && dgb != 0.f) atomicAdd(g_bias_grad, dgb);
}

// test / debug aid: the keep-scale both kernels apply, keep[b,k] in {0, 1/(1-p)}
__global__ void head_dropout_mask_kernel(int64_t B, int K, float drop_p, uint64_t drop_seed, const uint64_t* __restrict__ drop_seed_dev,
                                         float* __restrict__ keep) {
    if (drop_seed_dev) drop_seed += *drop_seed_dev;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < B * K; q += stride)
        keep[q] = keep_scale(drop_p, drop_seed, q / K, K, (int)(q % K));
}

}  // namespace rbr

using namespace rbr;

extern "C" int rbr_head_dropout_mask(int64_t batch, int64_t latent, float drop_p, uint64_t drop_seed, const uint64_t* drop_seed_dev,
                                     float* keep, void* stream) {
    RBR_REQUIRE(keep && batch >= 0 && latent > 0, RBR_EINVAL, "rbr_head_dropout_mask: bad arguments");
    RBR_REQUIRE(drop_p >= 0.f && drop_p < 1.f, RBR_EINVAL, "rbr_head_dropout_mask: dropout p must be in [0,1)");
    if (batch == 0) return RBR_OK;
    int64_t blocks = (batch * latent + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    head_dropout_mask_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(batch, (int)latent, drop_p, drop_seed, drop_seed_dev, keep);
    RBR_LAUNCH_CHECK("head_dropout_mask_kernel");
    return RBR_OK;
}

extern "C" int rbr_head_fwd(const float* u_text, const float* i_text, const int64_t* u_id, const int64_t* i_id, int64_t batch,
                            int64_t hidden, int64_t latent, const float* Wu, const float* bu, const float* ebd_u,
                            const float* Wi, const float* bi, const float* ebd_i, const float* fm_h, const float* user_bias,
                            const float* item_bias, const float* g_bias, int64_t users, int64_t items, float drop_p,
                            uint64_t drop_seed, const uint64_t* drop_seed_dev, float* pred, float* u_lat, float* i_lat,
                            const float* ratings, float grad_scale, float* loss_sum, float* pred_grad, void* stream) {
    RBR_REQUIRE(u_text && i_text && u_id && i_id && Wu && bu && ebd_u && Wi && bi && ebd_i && fm_h && user_bias && item_bias &&
                    g_bias && pred && u_lat && i_lat,
                RBR_EINVAL, "rbr_head_fwd: null pointer");
    RBR_REQUIRE(batch >= 0 && hidden > 0 && latent > 0 && latent <= 32 * HD_KQ, RBR_EUNSUPPORTED,
                "rbr_head_fwd: latent_dim must be in [1,%d]", 32 * HD_KQ);
    RBR_REQUIRE(drop_p >= 0.f && drop_p < 1.f, RBR_EINVAL, "rbr_head_fwd: dropout p must be in [0,1)");
    if (batch == 0) return RBR_OK;
    const int H = (int)hidden, K = (int)latent;
    {   // register-tiled kernel (latent % 4 == 0: float4 views of the latent gradients; everything else is padded in shared memory)
        const int Hp = (H + 3) & ~3;
        const bool small = batch <= 32 * 148 * 2;                      // few tiles: 16-sample CTAs fill the SMs twice over
        const int ts = small ? 16 : 32;
        const size_t smem2 = ((size_t)2 * Hp * K + (size_t)2 * ts * Hp) * 4;
        const bool aligned = (((uintptr_t)u_text | (uintptr_t)i_text | (uintptr_t)Wu | (uintptr_t)Wi) & 15) == 0;
        if (K % 4 == 0 && smem2 <= 200 * 1024) {
            static bool attr2 = false;
            if (!attr2) {
                RBR_CUDA(cudaFuncSetAttribute(head_fwd2_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
                RBR_CUDA(cudaFuncSetAttribute(head_fwd2_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
                attr2 = true;
            }
            int64_t blocks = (batch + ts - 1) / ts;
            if (blocks > 148 * 4) blocks = 148 * 4;
            auto kern = small ? head_fwd2_kernel<4> : head_fwd2_kernel<8>;
            kern<<<(unsigned)blocks, ts * 8, smem2, as_stream(stream)>>>(
                u_text, i_text, u_id, i_id, batch, H, K, Wu, bu, ebd_u, Wi, bi, ebd_i, fm_h, user_bias, item_bias, g_bias, users, items,
                drop_p, drop_seed, drop_seed_dev, pred, u_lat, i_lat, ratings, grad_scale, loss_sum, pred_grad, aligned ? 1 : 0);
            RBR_LAUNCH_CHECK("head_fwd2_kernel");
            return RBR_OK;
        }
    }
    const size_t smem = ((size_t)2 * H * (K + 1) + (size_t)HD_WARPS * 2 * H) * 4;
    RBR_REQUIRE(smem <= 200 * 1024, RBR_EUNSUPPORTED, "rbr_head_fwd: hidden*latent too large for shared memory");
    RBR_CUDA(cudaFuncSetAttribute(head_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t blocks = (batch + HD_WARPS - 1) / HD_WARPS;
    if (blocks > 148 * 2) blocks = 148 * 2;
    head_fwd_kernel<<<(unsigned)blocks, HD_WARPS * 32, smem, as_stream(stream)>>>(
        u_text, i_text, u_id, i_id, batch, H, K, Wu, bu, ebd_u, Wi, bi, ebd_i, fm_h, user_bias, item_bias, g_bias, users, items,
        drop_p, drop_seed, drop_seed_dev, pred, u_lat, i_lat, ratings, grad_scale, loss_sum, pred_grad);
    RBR_LAUNCH_CHECK("head_fwd_kernel");
    return RBR_OK;
}

extern "C" int rbr_head_bwd(const float* u_text, const float* i_text, const int64_t* u_id, const int64_t* i_id, int64_t batch,
                            int64_t hidden, int64_t latent, const float* Wu, const float* Wi, const float* fm_h,
                            const float* u_lat, const float* i_lat, float drop_p, uint64_t drop_seed,
                            const uint64_t* drop_seed_dev, int64_t ebd_u_padding_idx, int64_t ebd_i_padding_idx,
                            int64_t user_bias_padding_idx, int64_t item_bias_padding_idx, int64_t users, int64_t items, const float* pred_grad, float* u_text_grad, float* i_text_grad, float* Wu_grad, float* bu_grad,
                            float* ebd_u_grad, float* Wi_grad, float* bi_grad, float* ebd_i_grad, float* fm_h_grad,
                            float* user_bias_grad, float* item_bias_grad, float* g_bias_grad, void* stream) {
    RBR_REQUIRE(u_text && i_text && u_id && i_id && Wu && Wi && fm_h && u_lat && i_lat && pred_grad && u_text_grad &&
                    i_text_grad && Wu_grad && bu_grad && ebd_u_grad && Wi_grad && bi_grad && ebd_i_grad && fm_h_grad &&
                    user_bias_grad && item_bias_grad && g_bias_grad,
                RBR_EINVAL, "rbr_head_bwd: null pointer");
    RBR_REQUIRE(batch >= 0 && hidden > 0 && latent > 0 && latent <= 32 * HD_KQ, RBR_EUNSUPPORTED,
                "rbr_head_bwd: latent_dim must be in [1,%d]", 32 * HD_KQ);
    if (batch == 0) return RBR_OK;
    const int H = (int)hidden, K = (int)latent;
    {
        const int Hp = (H + 3) & ~3;
        const bool small = false;                                      // 32-sample tiles: half the weight-gradient atomics of 16 (22.6 vs 26.8 us)
        const int ts = small ? 16 : 32;
        const size_t smem2 = ((size_t)2 * H * (K + 1) + 4 + (size_t)2 * ts * Hp + (size_t)2 * ts * K) * 4;
        const bool aligned = (((uintptr_t)u_text | (uintptr_t)i_text) & 15) == 0;
        if (K % 4 == 0 && smem2 <= 200 * 1024) {
            static bool attr2 = false;
            if (!attr2) {
                RBR_CUDA(cudaFuncSetAttribute(head_bwd2_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
                RBR_CUDA(cudaFuncSetAttribute(head_bwd2_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
                attr2 = true;
            }
            int64_t blocks = (batch + ts - 1) / ts;
            if (blocks > 148 * 4) blocks = 148 * 4;
            auto kern = small ? head_bwd2_kernel<4> : head_bwd2_kernel<8>;
            kern<<<(unsigned)blocks, ts * 8, smem2, as_stream(stream)>>>(
                u_text, i_text, u_id, i_id, batch, H, K, Wu, Wi, fm_h, u_lat, i_lat, drop_p, drop_seed, drop_seed_dev, ebd_u_padding_idx,
                ebd_i_padding_idx, user_bias_padding_idx, item_bias_padding_idx, users, items, pred_grad, u_text_grad, i_text_grad, Wu_grad,
                bu_grad, ebd_u_grad, Wi_grad, bi_grad, ebd_i_grad, fm_h_grad, user_bias_grad, item_bias_grad, g_bias_grad, aligned ? 1 : 0);
            RBR_LAUNCH_CHECK("head_bwd2_kernel");
            return RBR_OK;
        }
    }
    const size_t smem = ((size_t)2 * H * (K + 1) + (size_t)2 * H * K + (size_t)2 * HD_BS * H + (size_t)2 * HD_BS * K) * 4;
    RBR_REQUIRE(smem <= 200 * 1024, RBR_EUNSUPPORTED, "rbr_head_bwd: hidden*latent too large for shared memory");
    RBR_CUDA(cudaFuncSetAttribute(head_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t blocks = (batch + HD_BS - 1) / HD_BS;
    if (blocks > 148 * 2) blocks = 148 * 2;
    head_bwd_kernel<<<(unsigned)blocks, HD_WARPS * 32, smem, as_stream(stream)>>>(
        u_text, i_text, u_id, i_id, batch, H, K, Wu, Wi, fm_h, u_lat, i_lat, drop_p, drop_seed, drop_seed_dev, ebd_u_padding_idx,
        ebd_i_padding_idx, user_bias_padding_idx, item_bias_padding_idx, users, items, pred_grad, u_text_grad, i_text_grad, Wu_grad, bu_grad, ebd_u_grad, Wi_grad, bi_grad,
        ebd_i_grad, fm_h_grad, user_bias_grad, item_bias_grad, g_bias_grad);
    RBR_LAUNCH_CHECK("head_bwd_kernel");
    return RBR_OK;
}

RBR_DEFINE_OOB_ACCESSOR(head)
