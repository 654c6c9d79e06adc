// explain.cu — K12: token attributions of a predicted rating from the per-entity feature cache.  sm_100a only.
//
// After max-over-time (NgramFeat.forward, models/deepconn/layers.py:123-136) each pooled feature feat[n,h] depends on
// exactly one k-token window, the one starting at t*[n,h] - pad (t* = the forward's first arg-max).  Its pre-activation is
// bias[h] plus k tap contributions
//   c[n,h,j] = sum_e W[h,e,j] * x[n, t*[n,h] + j - pad, e]
// which depend on the entity's own document only, so they are computed once per entity (rbr_conv_window_contrib, at cache
// build time).  With g[n,h] = d pred / d feat[n,h] for one (user, item) pair, gradient x input on the embedded tokens is
//   attr[n,t] = sum_{h : feat[n,h] > 0} sum_{j : t*[n,h] + j - pad = t} g[n,h] * c[n,h,j]
// (rbr_explain_attrib, per pair and side).
//
// Determinism: the scatter of the g*c terms onto positions runs as 64-bit FIXED-POINT integer atomics in shared memory.  Each
// term is rounded once onto a grid of 2^-61 times a per-row bound on the total, so integer sums are exact and the map, its
// total, the per-review sums and the windows do not depend on the order of the atomics, the batch or the position of the pair
// in it.  Window sums are taken in double over the fp32 map (<= 16 floats: exact in practice), so a caller re-deriving the
// windows from the returned map in float64 finds the same ones.
#include <math.h>

#include "rbr_common.cuh"

namespace rbr {

constexpr int EX_MAX_POSITIONS = 16384;   // docs_per_entity * doc_len: the map (int64 + fp32 + flags) must fit shared memory
constexpr int EX_MAX_M = 32;
constexpr int EX_MAX_WIDTH = 16;
constexpr int EX_MAX_CONVS = 8;
constexpr int EX_THREADS = 256;
constexpr int EX_MAX_SMEM = 227 * 1024;

static bool ex_supported(int64_t positions, int64_t m, int64_t width, int64_t n_conv) {
    return positions >= 1 && positions <= EX_MAX_POSITIONS && m >= 1 && m <= EX_MAX_M && width >= 1 && width <= EX_MAX_WIDTH &&
           n_conv >= 1 && n_conv <= EX_MAX_CONVS;
}

// ---- the row the forward multiplies at one position, dotted with a weight vector -------------------------------------------
// Warp-wide: every lane returns sum_e x[n, t, e] * w[e].  x is zero outside the document, at masked positions and for ids
// outside the table (conv_fp32.cu's row resolution), so any position t is memory-safe.
__device__ __forceinline__ float ex_row_dot(const float* __restrict__ table, int64_t vocab, int64_t emb, const IdView& iv,
                                            const uint8_t* __restrict__ mask, int64_t n, int64_t doc_len, int64_t t,
                                            const float* __restrict__ w) {
    const int lane = threadIdx.x & 31;
    int64_t row = -1;
    if (t >= 0 && t < doc_len) {
        const int64_t id = ld_id(iv, n * doc_len + t);
        if (ld_mask(iv, mask, n * doc_len + t, id) && id >= 0 && id < vocab) row = id;
    }
    float s = 0.f;
    if (row >= 0) {
        const float* x = table + row * emb;
        for (int64_t e = lane; e < emb; e += 32) s = fmaf(__ldg(x + e), __ldg(w + e), s);
    }
    return warp_sum(s);
}

// ---- c[n, h, j]: one warp per (document, filter) ---------------------------------------------------------------------------
__global__ void conv_window_contrib_kernel(const float* __restrict__ table, int64_t vocab, int64_t emb, IdView iv,
                                           const uint8_t* __restrict__ mask, int64_t n_docs, int64_t doc_len,
                                           const float* __restrict__ whke, int64_t epad4, int64_t filters, int64_t ksize,
                                           int64_t pad, const int32_t* __restrict__ argmax, int64_t argmax_ld,
                                           float* __restrict__ contrib, int64_t contrib_ld) {
    const int lane = threadIdx.x & 31;
    const int64_t gw = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (gw >= n_docs * filters) return;
    const int64_t n = gw / filters, h = gw % filters;
    const int64_t t0 = (int64_t)__ldg(argmax + n * argmax_ld + h) - pad;
    for (int64_t j = 0; j < ksize; ++j) {
        const float s = ex_row_dot(table, vocab, emb, iv, mask, n, doc_len, t0 + j, whke + (h * ksize + j) * epad4);
        if (lane == 0) contrib[n * contrib_ld + h * ksize + j] = s;
    }
}

// ---- D-ATT: per-entity terms of gradient x input through both gates (models/dual_att/layers.py:25-89) ---------------------
// One warp per (document, item): items [0, htot) are the pooled features (local filters first, then the k = 2, 3, 4 global
// convs), items [htot, htot + L) the positions of gate_vec.  With d = 1 - f^2 (tanh' at the pooled output f) and t* the arg-max:
//   local filter h (k = 1 conv on gl * x), q = W_h . x[t*]:
//     contrib[h, j] = d q gl(1-gl)[t*] (w_l[:, j] . x[t* + j - pad_l])  +  [j == pad_l] d gl[t*] q        (width-k_l window)
//   global filter h (k-wide conv on gg * x, no padding), c_j = W_h[:, j] . x[t* + j]:
//     contrib[h, j] = d gg c_j,   gate_coef[h] = d sum_j c_j   (0 on the local columns)
//   gate_vec[s] = gg(1-gg) (w_g[:, s] . x[s])
struct DattExArgs {
    const float* table;
    int64_t vocab, emb, n_docs, L;
    IdView iv;
    const float* wlT;          // [kl][emb]: the local gate's weight, transposed
    const float* wgT;          // [L][emb]:  the global gate's weight, transposed
    int kl;
    const float* whke[4];      // fp32 [H][k][Epad4] copies of the four conv weights (conv_pack)
    int64_t epad4[4];
    int h_end[4], k[4];        // filter column where conv c ends; its kernel width (1, 2, 3, 4)
    int64_t coff[4];           // first contribution column of conv c (the local conv spans kl taps per filter)
    const float* gate_l;       // [n_docs, L]
    const float* gate_g;       // [n_docs]
    const float* feat;         // [n_docs, feat_ld]
    const int32_t* argmax;     // [n_docs, feat_ld]
    int64_t feat_ld;
    float* contrib; int64_t contrib_ld;
    float* gate_coef; int64_t coef_ld;
    float* gate_vec; int64_t vec_ld;
};

__global__ void datt_explain_contrib_kernel(const DattExArgs a) {
    const int lane = threadIdx.x & 31;
    const int htot = a.h_end[3];
    const int64_t items = htot + a.L;
    const int64_t gw = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (gw >= a.n_docs * items) return;
    const int64_t n = gw / items, it = gw % items;
    const float gg = __ldg(a.gate_g + n);
    if (it >= htot) {
        const int64_t s = it - htot;
        const float v = ex_row_dot(a.table, a.vocab, a.emb, a.iv, nullptr, n, a.L, s, a.wgT + s * a.emb);
        if (lane == 0) a.gate_vec[n * a.vec_ld + s] = gg * (1.f - gg) * v;
        return;
    }
    int c = 0;
    while (c < 3 && it >= a.h_end[c]) ++c;
    const int64_t h = it - (c ? a.h_end[c - 1] : 0);
    const float f = __ldg(a.feat + n * a.feat_ld + it);
    const float d = 1.f - f * f;
    const int64_t ts = __ldg(a.argmax + n * a.feat_ld + it);
    float* out = a.contrib + n * a.contrib_ld + a.coff[c];
    if (c == 0) {
        const float q = ex_row_dot(a.table, a.vocab, a.emb, a.iv, nullptr, n, a.L, ts, a.whke[0] + h * a.epad4[0]);
        const float gl = (ts >= 0 && ts < a.L) ? __ldg(a.gate_l + n * a.L + ts) : 0.f;
        const float dq = d * q, slope = gl * (1.f - gl);
        const int pad = (a.kl - 1) / 2;
        for (int j = 0; j < a.kl; ++j) {
            const float tap = ex_row_dot(a.table, a.vocab, a.emb, a.iv, nullptr, n, a.L, ts + j - pad, a.wlT + j * a.emb);
            float v = dq * (slope * tap);
            if (j == pad) v += dq * gl;
            if (lane == 0) out[h * a.kl + j] = v;
        }
        if (lane == 0) a.gate_coef[n * a.coef_ld + it] = 0.f;
    } else {
        const int k = a.k[c];
        float sum = 0.f;
        for (int j = 0; j < k; ++j) {
            const float cj = ex_row_dot(a.table, a.vocab, a.emb, a.iv, nullptr, n, a.L, ts + j, a.whke[c] + (h * k + j) * a.epad4[c]);
            sum += cj;
            if (lane == 0) out[h * k + j] = d * gg * cj;
        }
        if (lane == 0) a.gate_coef[n * a.coef_ld + it] = d * sum;
    }
}

// ---- per (pair, side) row: attribution map, total, per-review sums, top / bottom windows ------------------------------------
struct ExConvs {
    int n;
    int h_end[EX_MAX_CONVS];   // filter column where conv c ends (exclusive), within feat / argmax / g rows
    int k[EX_MAX_CONVS], pad[EX_MAX_CONVS];
    int64_t coff[EX_MAX_CONVS];   // column of conv c's first tap within a contribution row
};

// dynamic shared memory of explain_attrib_kernel: the map (int64 + fp32 + flags), then the dense scalars
__host__ __device__ inline int64_t ex_dscal_off(int64_t S) { return (S * 13 + 7) & ~(int64_t)7; }
__host__ inline size_t ex_smem_bytes(int64_t S, int64_t R, bool dense) { return (size_t)(ex_dscal_off(S) + (dense ? R * 8 : 0)); }

// where a row's outputs go: text_total [P], top / bottom windows [P, m], map [P, R*T] and review_attr [P, R] (both optional)
struct ExOut {
    float* text_total;
    int64_t* top_pos; float* top_attr; int64_t* bot_pos; float* bot_attr;
    float* map;
    float* review_attr;
};

struct ExArgs {
    const int64_t* ent_row;
    const float* g;          // [P, R, Htot]
    const float* feat;       // [n_docs, feat_ld] or NULL: every filter counts (no liveness predicate, e.g. tanh)
    const int32_t* argmax;   // [n_docs, feat_ld]
    const float* contrib;    // [n_docs, contrib_ld]
    const float* dense_coef; // [n_docs, coef_ld] or NULL: no dense term
    const float* dense_vec;  // [n_docs, vec_ld]
    int64_t n_docs, feat_ld, contrib_ld, coef_ld, vec_ld, htot;
    int R, T, m, width;
    ExConvs cv;
    ExOut out;
};

__device__ __forceinline__ int ex_conv_of(const ExConvs& cv, int hh) {
    int c = 0;
    while (c + 1 < cv.n && hh >= cv.h_end[c]) ++c;
    return c;
}

// block-wide reductions (EX_THREADS threads); `red` holds EX_THREADS / 32 entries of the widest type
__device__ __forceinline__ float ex_block_max(float v, double* red) {
    v = warp_max(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    float r = 0.f;
    for (int w = 0; w < EX_THREADS / 32; ++w) r = fmaxf(r, (float)red[w]);
    return r;
}

__device__ __forceinline__ long long ex_warp_sum_ll(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ long long ex_block_sum_ll(long long v, double* red) {
    v = ex_warp_sum_ll(v);
    long long* r = reinterpret_cast<long long*>(red);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) r[threadIdx.x >> 5] = v;
    __syncthreads();
    long long s = 0;
    for (int w = 0; w < EX_THREADS / 32; ++w) s += r[w];
    return s;
}

// (value, start) order of the greedy selection: larger (top) / smaller (bottom) value first, then the lower start; s < 0 = none
__device__ __forceinline__ bool ex_better(double v, int s, double bv, int bs, bool top) {
    if (s < 0) return false;
    if (bs < 0) return true;
    if (v != bv) return top ? v > bv : v < bv;
    return s < bs;
}

__device__ __forceinline__ void ex_block_pick(double& v, int& s, bool top, double* red_v, int* red_s) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, v, o);
        const int os = __shfl_xor_sync(0xffffffffu, s, o);
        if (ex_better(ov, os, v, s, top)) { v = ov; s = os; }
    }
    __syncthreads();
    if ((threadIdx.x & 31) == 0) { red_v[threadIdx.x >> 5] = v; red_s[threadIdx.x >> 5] = s; }
    __syncthreads();
    v = 0.0; s = -1;
    for (int w = 0; w < EX_THREADS / 32; ++w)
        if (ex_better(red_v[w], red_s[w], v, s, top)) { v = red_v[w]; s = red_s[w]; }
}

// The fixed-point grid of a row whose |total| is at most n_terms * mx: with mx * n_terms < 2^e, terms on a grid of 2^(e-61)
// keep every partial sum below 2^61 in magnitude.  0 when there is nothing to add.
__device__ __forceinline__ double ex_fixed_scale(float mx, double n_terms) {
    double scale = 0.0;
    if (mx > 0.f && isfinite(mx)) {
        int e;
        frexp((double)mx * n_terms, &e);
        scale = ldexp(1.0, 61 - e);
    }
    return scale;
}

// Everything of row p after its fixed-point map acc [S] (S = R * T) and total are known: text_total, the fp32 map (mapf and,
// if asked, out.map), the per-review sums and the top / bottom windows of `width` positions (greedy without overlap, ties to
// the lower start, never across a review).  A row that is not `ok` gets NaN / -1.  Block-wide; acc becomes the window sums.
__device__ __forceinline__ void ex_emit_row(long long* acc, float* mapf, uint8_t* avail, double* red_v, int* red_s, long long tot,
                            double scale, bool ok, int64_t p, int R, int T, int m, int w, const ExOut& out) {
    const int S = R * T;
    const float nanf_ = __int_as_float(0x7fc00000);
    const double inv = scale > 0.0 ? 1.0 / scale : 0.0;
    if (threadIdx.x == 0) out.text_total[p] = ok ? (float)((double)tot * inv) : nanf_;
    __syncthreads();                                                   // the map has landed
    for (int i = threadIdx.x; i < S; i += EX_THREADS) {
        const float v = ok ? (float)((double)acc[i] * inv) : nanf_;
        mapf[i] = v;
        if (out.map) out.map[p * S + i] = v;
    }
    if (out.review_attr) {
        for (int r = threadIdx.x >> 5; r < R; r += EX_THREADS / 32) {
            long long s = 0;
            for (int t = threadIdx.x & 31; t < T; t += 32) s += acc[r * T + t];
            s = ex_warp_sum_ll(s);
            if ((threadIdx.x & 31) == 0) out.review_attr[p * R + r] = ok ? (float)((double)s * inv) : nanf_;
        }
    }
    __syncthreads();                                                   // acc is read for the last time above
    double* wsum = reinterpret_cast<double*>(acc);
    for (int s = threadIdx.x; s < S; s += EX_THREADS) {
        double v = 0.0;
        if ((s % T) + w <= T)
            for (int j = 0; j < w; ++j) v += (double)mapf[s + j];
        wsum[s] = v;
    }
    for (int pass = 0; pass < 2; ++pass) {
        const bool top = pass == 0;
        int64_t* out_pos = (top ? out.top_pos : out.bot_pos) + p * m;
        float* out_attr = (top ? out.top_attr : out.bot_attr) + p * m;
        for (int s = threadIdx.x; s < S; s += EX_THREADS) avail[s] = ok && (s % T) + w <= T;
        __syncthreads();
        for (int it = 0; it < m; ++it) {
            double bv = 0.0;
            int bs = -1;
            for (int s = threadIdx.x; s < S; s += EX_THREADS)
                if (avail[s] && ex_better(wsum[s], s, bv, bs, top)) { bv = wsum[s]; bs = s; }
            ex_block_pick(bv, bs, top, red_v, red_s);
            if (threadIdx.x == 0) {
                out_pos[it] = bs;
                out_attr[it] = bs >= 0 ? (float)bv : nanf_;
            }
            if (bs < 0) {
                for (int j = it + 1 + (int)threadIdx.x; j < m; j += EX_THREADS) { out_pos[j] = -1; out_attr[j] = nanf_; }
                break;
            }
            // windows never cross a review boundary, so every start whose window overlaps [bs, bs + w) lies in (bs - w, bs + w)
            for (int s = max(0, bs - w + 1) + (int)threadIdx.x; s < min(S, bs + w); s += EX_THREADS) avail[s] = 0;
            __syncthreads();
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(EX_THREADS) explain_attrib_kernel(const ExArgs a) {
    extern __shared__ __align__(16) unsigned char ex_smem[];
    __shared__ double red_v[EX_THREADS / 32];
    __shared__ int red_s[EX_THREADS / 32];
    const int S = a.R * a.T;
    long long* acc = reinterpret_cast<long long*>(ex_smem);          // [S] fixed-point map; later the window sums (double)
    float* mapf = reinterpret_cast<float*>(acc + S);                  // [S]
    uint8_t* avail = reinterpret_cast<uint8_t*>(mapf + S);            // [S] window start still selectable
    double* dscal = reinterpret_cast<double*>(ex_smem + ex_dscal_off(S)); // [R] dense scalars (when there is a dense term)
    const int64_t p = blockIdx.x;
    const int64_t row0 = __ldg(a.ent_row + p);
    const bool ok = row0 >= 0 && row0 + a.R <= a.n_docs;              // the host validates; a bad row yields NaN / -1, no read
    const int n_items = a.R * (int)a.htot;
    const float* gp = a.g + p * n_items;

    for (int i = threadIdx.x; i < S; i += EX_THREADS) acc[i] = 0;
    const bool dense = a.dense_coef != nullptr;
    // pass 0: the dense term's per-document scalar sum_h g * dense_coef, one warp per document, a fixed summation order
    if (ok && dense) {
        for (int r = threadIdx.x >> 5; r < a.R; r += EX_THREADS / 32) {
            const float* cf = a.dense_coef + (row0 + r) * a.coef_ld;
            double v = 0.0;
            for (int hh = threadIdx.x & 31; hh < (int)a.htot; hh += 32)
                v += (double)__ldg(gp + r * a.htot + hh) * (double)__ldg(cf + hh);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if ((threadIdx.x & 31) == 0) dscal[r] = v;
        }
        __syncthreads();
    }
    // pass 1: the largest |term| bounds the total, which fixes the fixed-point scale
    float mx = 0.f;
    int max_k = 0;
    for (int c = 0; c < a.cv.n; ++c) max_k = max(max_k, a.cv.k[c]);
    if (ok) {
        if (dense)
            for (int i = threadIdx.x; i < S; i += EX_THREADS) {
                const int r = i / a.T;
                mx = fmaxf(mx, (float)fabs(dscal[r] * (double)__ldg(a.dense_vec + (row0 + r) * a.vec_ld + i % a.T)));
            }
        for (int i = threadIdx.x; i < n_items; i += EX_THREADS) {
            const int r = i / (int)a.htot, hh = i % (int)a.htot;
            const int64_t doc = row0 + r;
            if (a.feat && !(__ldg(a.feat + doc * a.feat_ld + hh) > 0.f)) continue;
            const float gv = __ldg(gp + i);
            const int c = ex_conv_of(a.cv, hh);
            const int h = hh - (c ? a.cv.h_end[c - 1] : 0);
            const float* cp = a.contrib + doc * a.contrib_ld + a.cv.coff[c] + (int64_t)h * a.cv.k[c];
            for (int j = 0; j < a.cv.k[c]; ++j) mx = fmaxf(mx, fabsf(gv * __ldg(cp + j)));
        }
    }
    mx = ex_block_max(mx, red_v);
    // |total| <= (n_items * max_k + dense positions) * mx
    const double scale = ex_fixed_scale(mx, (double)n_items * (double)max_k + (dense ? (double)S : 0.0));
    __syncthreads();
    // pass 2: scatter the rounded terms; every term enters the total, the ones at a position inside the document also the map
    long long tot = 0;
    if (ok && scale > 0.0) {
        if (dense)
            for (int i = threadIdx.x; i < S; i += EX_THREADS) {
                const int r = i / a.T;
                const long long q = llrint(dscal[r] * (double)__ldg(a.dense_vec + (row0 + r) * a.vec_ld + i % a.T) * scale);
                if (q == 0) continue;
                tot += q;
                atomicAdd(reinterpret_cast<unsigned long long*>(acc + i), (unsigned long long)q);
            }
        for (int i = threadIdx.x; i < n_items; i += EX_THREADS) {
            const int r = i / (int)a.htot, hh = i % (int)a.htot;
            const int64_t doc = row0 + r;
            if (a.feat && !(__ldg(a.feat + doc * a.feat_ld + hh) > 0.f)) continue;
            const double gv = (double)__ldg(gp + i);
            const int c = ex_conv_of(a.cv, hh);
            const int h = hh - (c ? a.cv.h_end[c - 1] : 0);
            const float* cp = a.contrib + doc * a.contrib_ld + a.cv.coff[c] + (int64_t)h * a.cv.k[c];
            const int t0 = __ldg(a.argmax + doc * a.feat_ld + hh) - a.cv.pad[c];
            for (int j = 0; j < a.cv.k[c]; ++j) {
                const long long q = llrint(gv * (double)__ldg(cp + j) * scale);     // exact product, one rounding
                if (q == 0) continue;
                tot += q;
                const int t = t0 + j;
                if (t >= 0 && t < a.T)
                    atomicAdd(reinterpret_cast<unsigned long long*>(acc + r * a.T + t), (unsigned long long)q);
            }
        }
    }
    tot = ex_block_sum_ll(tot, red_v);
    ex_emit_row(acc, mapf, avail, red_v, red_s, tot, scale, ok, p, a.R, a.T, a.m, a.width, a.out);
}

// ---- K13: SimpleSiamese — gradient x input through masked average pooling and the review attention ------------------------
// One side of an entity (models/simple_siamese/simple_siamese.py:55-88, eval mode): pooled p_r = sum_t m x / (n_r + 1e-8),
// v_r = tanh(Lt p_r + bt) (or p_r), s = softmax(l), l_r = w . tanh(P v_r + c) (-1e8 where the review is masked), f = sum_r s_r v_r.
// With g = d pred / d f and the per-entity a_r = P^T (w * (1 - tanh^2(P v_r + c))) (0 for a masked review):
//   dv_r = s_r (g + (g . (v_r - f)) a_r),   G_r = Lt^T ((1 - v_r^2) * dv_r) (or dv_r),   attr[r,t] = m x[r,t] . G_r / (n_r + 1e-8)
// Every token has exactly one term, so the map is one fp32 dot per position, rounded once onto K12b's fixed-point grid.
constexpr int XA_RB = 4;      // reviews per pass of the G_r product (each Lt element read once per XA_RB reviews)

struct XaArgs {
    const float* table;
    int64_t vocab, emb;
    IdView iv;
    const uint8_t* mask;     // [n_ent, R, T] or NULL (iv.mask_ids: ids != 0)
    int64_t n_ent;
    int R, T, F, K;
    const int64_t* ent;      // [P] entity of each row
    const float* g;          // [P, F] d pred / d f, or NULL: from the latents below
    const int64_t* other;    // [P] the pair's other entity
    const float* lat;        // [n_ent, K] this side's LastFeat outputs
    const float* lat_other;  // [n_other, K]
    int64_t n_other;
    const float* w_side;     // [F, K] this side's LastFeat.W
    const float* fm_h;       // [K]
    const float* v;          // [n_ent, R, F]
    const float* att_a;      // [n_ent, R, F]
    const float* att_s;      // [n_ent, R]
    const float* f;          // [n_ent, F]
    const float* lt_w;       // [F, emb] or NULL (F == emb)
    int m, width;
    ExOut out;
};

// dynamic shared memory: K12b's map region, then g [F], dots [R], 1 / (n_r + 1e-8) [R], dv [R, F], G [R, emb]
__host__ __device__ inline int64_t xa_smem_bytes(int64_t R, int64_t T, int64_t emb, int64_t F) {
    return ex_dscal_off(R * T) + 4 * (F + 2 * R + R * F + R * emb);
}

__global__ void __launch_bounds__(EX_THREADS) explain_avgpool_attrib_kernel(const XaArgs a) {
    extern __shared__ __align__(16) unsigned char ex_smem[];
    __shared__ double red_v[EX_THREADS / 32];
    __shared__ int red_s[EX_THREADS / 32];
    const int R = a.R, T = a.T, S = R * T, F = a.F, E = (int)a.emb;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long* acc = reinterpret_cast<long long*>(ex_smem);
    float* mapf = reinterpret_cast<float*>(acc + S);
    uint8_t* avail = reinterpret_cast<uint8_t*>(mapf + S);
    float* gv = reinterpret_cast<float*>(ex_smem + ex_dscal_off(S));
    float* dots = gv + F;
    float* inv_n = dots + R;
    float* dv = inv_n + R;
    float* G = dv + R * F;
    const int64_t p = blockIdx.x;
    const int64_t e = __ldg(a.ent + p);
    const int64_t o = a.g ? 0 : __ldg(a.other + p);
    const bool ok = e >= 0 && e < a.n_ent && (a.g || (o >= 0 && o < a.n_other));   // the host validates; else NaN / -1
    if (ok) {
        // g: given, or W_side (h * 1[lat * lat_other > 0] * lat_other), k in order
        for (int i = threadIdx.x; i < F; i += EX_THREADS) {
            float x = 0.f;
            if (a.g) {
                x = __ldg(a.g + p * F + i);
            } else {
                const float* ls = a.lat + e * a.K;
                const float* lo = a.lat_other + o * a.K;
                for (int k = 0; k < a.K; ++k) {
                    const float us = __ldg(ls + k), ot = __ldg(lo + k);
                    if ((us > 0.f && ot > 0.f) || (us < 0.f && ot < 0.f))
                        x = fmaf(__ldg(a.w_side + (int64_t)i * a.K + k), __ldg(a.fm_h + k) * ot, x);
                }
            }
            gv[i] = x;
        }
        // the forward's token count per review (masked-in ids outside the table count, as in K9)
        for (int r = warp; r < R; r += EX_THREADS / 32) {
            int c = 0;
            for (int t = lane; t < T; t += 32) {
                const int64_t idx = (e * R + r) * T + t;
                c += ld_mask(a.iv, a.mask, idx, ld_id(a.iv, idx)) ? 1 : 0;
            }
#pragma unroll
            for (int s = 16; s > 0; s >>= 1) c += __shfl_xor_sync(0xffffffffu, c, s);
            if (lane == 0) inv_n[r] = 1.f / ((float)c + 1e-8f);
        }
        __syncthreads();
        const float* vr = a.v + e * R * F;
        const float* fe = a.f + e * F;
        for (int r = warp; r < R; r += EX_THREADS / 32) {
            float d = 0.f;
            for (int i = lane; i < F; i += 32) d = fmaf(gv[i], __ldg(vr + r * F + i) - __ldg(fe + i), d);
            d = warp_sum(d);
            if (lane == 0) dots[r] = d;
        }
        __syncthreads();
        const float* ar = a.att_a + e * R * F;
        for (int i = threadIdx.x; i < R * F; i += EX_THREADS) {
            const int r = i / F;
            float d = __ldg(a.att_s + e * R + r) * fmaf(dots[r], __ldg(ar + i), gv[i % F]);
            if (a.lt_w) {
                const float vv = __ldg(vr + i);
                d *= 1.f - vv * vv;
            }
            dv[i] = d;
        }
        __syncthreads();
        // G[r, c] = (sum_k Lt[k, c] dv[r, k]) / (n_r + 1e-8), k in order
        if (a.lt_w) {
            for (int i = threadIdx.x; i < ((R + XA_RB - 1) / XA_RB) * E; i += EX_THREADS) {
                const int r0 = (i / E) * XA_RB, c = i % E;
                float x[XA_RB] = {};
                for (int k = 0; k < F; ++k) {
                    const float wk = __ldg(a.lt_w + (int64_t)k * E + c);
#pragma unroll
                    for (int j = 0; j < XA_RB; ++j)
                        if (r0 + j < R) x[j] = fmaf(wk, dv[(r0 + j) * F + k], x[j]);
                }
#pragma unroll
                for (int j = 0; j < XA_RB; ++j)
                    if (r0 + j < R) G[(r0 + j) * E + c] = x[j] * inv_n[r0 + j];
            }
        } else {
            for (int i = threadIdx.x; i < R * E; i += EX_THREADS) G[i] = dv[i] * inv_n[i / E];
        }
        __syncthreads();
        // one warp per position: attr = x . G_r (0 where masked and for ids outside the table)
        const int64_t base = e * S;
        for (int i = warp; i < S; i += EX_THREADS / 32) {
            const int64_t id = ld_id(a.iv, base + i);
            float s = 0.f;
            if (ld_mask(a.iv, a.mask, base + i, id) && id >= 0 && id < a.vocab) {
                const float* x = a.table + id * E;
                const float* gr = G + (i / T) * E;
                for (int c = lane; c < E; c += 32) s = fmaf(__ldg(x + c), gr[c], s);
                s = warp_sum(s);
            }
            if (lane == 0) mapf[i] = s;
        }
    }
    __syncthreads();
    float mx = 0.f;
    if (ok)
        for (int i = threadIdx.x; i < S; i += EX_THREADS) mx = fmaxf(mx, fabsf(mapf[i]));
    mx = ex_block_max(mx, red_v);
    const double scale = ex_fixed_scale(mx, (double)S);                // one term per position: |total| <= S * mx
    long long tot = 0;
    for (int i = threadIdx.x; i < S; i += EX_THREADS) {
        const long long q = (ok && scale > 0.0) ? llrint((double)mapf[i] * scale) : 0;
        acc[i] = q;
        tot += q;
    }
    tot = ex_block_sum_ll(tot, red_v);
    ex_emit_row(acc, mapf, avail, red_v, red_s, tot, scale, ok, p, R, T, a.m, a.width, a.out);
}

// ---- D-ATT: g = d pred / d cat per pair and side, through the shared FC stack (dual_att.py:31-35, 51, 57-61) ----------------
// pred = fc(cat_u) . fc(cat_i), fc(x) = W3 relu(W0 x + b0) + b3, so for the user side (the item side is symmetric)
//   g_u = W0^T (1[z_u > 0] * W3^T fc(cat_i))        z_u = the user's hidden pre-activation (its cached ReLU mask)
// One CTA per FG_BM pairs and side.  Stage A writes v = mask * W3^T fc(other) [FG_BM, hidden] to shared memory (fp32 FMAs in
// order o = 0, 1, ...); stage B is the [FG_BM, hidden] x [hidden, in_dim] product on the tensor cores at fp32 grade: 3xTF32
// mma.sync (a = a_hi + a_lo, b = b_hi + b_lo, d += a_lo b_hi + a_hi b_lo + a_hi b_hi), k-steps in order.  Every output element
// is reduced in the same fixed order whatever the batch, its position in it or the tile it falls in, so results are
// bit-identical across calls, chunk sizes and pair orders.
constexpr int FG_BM = 64;
constexpr int FG_THREADS = 256;
constexpr int FG_MAX_HIDDEN = 768;

// k padded to whole mma k-steps; the shared-memory row stride is = 4 (mod 32) floats, so the A-fragment loads (rows g,
// columns t of an 8-row x 4-column lane grid) hit 32 distinct banks
__host__ __device__ inline int64_t fg_kpad(int64_t hidden) { return (hidden + 7) & ~(int64_t)7; }
__host__ __device__ inline int64_t fg_stride(int64_t hidden) {
    const int64_t kp = fg_kpad(hidden);
    return kp + ((4 - kp % 32) + 32) % 32;
}

struct FgArgs {
    const int64_t* ids[2];      // [P] user / item entity ids of each pair
    const float* out[2];        // [n_ent, out_dim] cached FC outputs
    const uint8_t* mask[2];     // [n_ent, hidden] cached 1[z > 0]
    int64_t n_ent[2];
    int64_t P, out_dim, hidden, in_dim;
    const float* w0;            // [hidden, in_dim]  (fc.0.weight)
    const float* w3;            // [out_dim, hidden] (fc.3.weight)
    float* g[2];                // [P, in_dim]
    int kp, vs;
};

__device__ __forceinline__ uint32_t fg_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ void fg_split(float x, uint32_t& hi, uint32_t& lo) {
    hi = fg_tf32(x);
    lo = fg_tf32(x - __uint_as_float(hi));
}
__device__ __forceinline__ void fg_mma(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__global__ void __launch_bounds__(FG_THREADS) datt_fc_grads_kernel(const FgArgs a) {
    extern __shared__ __align__(16) float fg_v[];                    // [FG_BM][vs]
    const int side = blockIdx.y, other = 1 - side;
    const int64_t p0 = (int64_t)blockIdx.x * FG_BM;
    const int kp = a.kp, vs = a.vs;
    const int H = (int)a.hidden;
    // stage A: v[r, k] = mask_self[k] ? sum_o out_other[o] * W3[o, k] : 0  (zero past `hidden`, past P and for bad ids)
    for (int idx = threadIdx.x; idx < FG_BM * kp; idx += FG_THREADS) {
        const int r = idx / kp, k = idx % kp;
        const int64_t p = p0 + r;
        float v = 0.f;
        if (p < a.P && k < H) {
            const int64_t es = __ldg(a.ids[side] + p), eo = __ldg(a.ids[other] + p);
            if (es >= 0 && es < a.n_ent[side] && eo >= 0 && eo < a.n_ent[other] && __ldg(a.mask[side] + es * a.hidden + k)) {
                const float* fo = a.out[other] + eo * a.out_dim;
                for (int64_t o = 0; o < a.out_dim; ++o) v = fmaf(__ldg(fo + o), __ldg(a.w3 + o * a.hidden + k), v);
            }
        }
        fg_v[r * vs + k] = v;
    }
    __syncthreads();
    // stage B: g[r, n] = sum_k v[r, k] * W0[k, n]; warp w takes the 8-column tiles w, w + 8, ...; all FG_BM rows per tile
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gq = lane >> 2, tq = lane & 3;
    const int64_t n_tiles = (a.in_dim + 7) / 8;
    float* gout = a.g[side];
    for (int64_t nt = warp; nt < n_tiles; nt += FG_THREADS / 32) {
        const int64_t col = nt * 8 + gq;                              // the B column this lane loads
        const bool col_ok = col < a.in_dim;
        float acc[FG_BM / 16][4];
#pragma unroll
        for (int mt = 0; mt < FG_BM / 16; ++mt)
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[mt][q] = 0.f;
        for (int k0 = 0; k0 < kp; k0 += 8) {
            const int ka = k0 + tq, kb = k0 + tq + 4;
            const float bf0 = (col_ok && ka < H) ? __ldg(a.w0 + (int64_t)ka * a.in_dim + col) : 0.f;
            const float bf1 = (col_ok && kb < H) ? __ldg(a.w0 + (int64_t)kb * a.in_dim + col) : 0.f;
            uint32_t b0h, b0l, b1h, b1l;
            fg_split(bf0, b0h, b0l);
            fg_split(bf1, b1h, b1l);
#pragma unroll
            for (int mt = 0; mt < FG_BM / 16; ++mt) {
                const float* vr = fg_v + (mt * 16 + gq) * vs + k0 + tq;
                uint32_t ah[4], al[4];
                fg_split(vr[0], ah[0], al[0]);
                fg_split(vr[8 * vs], ah[1], al[1]);
                fg_split(vr[4], ah[2], al[2]);
                fg_split(vr[8 * vs + 4], ah[3], al[3]);
                fg_mma(acc[mt], al, b0h, b1h);
                fg_mma(acc[mt], ah, b0l, b1l);
                fg_mma(acc[mt], ah, b0h, b1h);
            }
        }
        const int64_t c0 = nt * 8 + 2 * tq;
#pragma unroll
        for (int mt = 0; mt < FG_BM / 16; ++mt)
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int64_t p = p0 + mt * 16 + gq + (q >> 1) * 8, c = c0 + (q & 1);
                if (p < a.P && c < a.in_dim) gout[p * a.in_dim + c] = acc[mt][q];
            }
    }
}

}  // namespace rbr

using namespace rbr;

extern "C" int rbr_explain_supported(int64_t positions, int64_t m, int64_t width, int64_t n_conv) {
    return ex_supported(positions, m, width, n_conv) ? 1 : 0;
}

extern "C" int rbr_conv_window_contrib(const float* table, int64_t vocab, int64_t emb, const void* ids, const uint8_t* mask,
                                       int64_t n_docs, int64_t doc_len, const void* packed, int64_t filters, int64_t ksize,
                                       int64_t pad, const int32_t* argmax, int64_t argmax_ld, float* contrib,
                                       int64_t contrib_ld, int flags, void* stream) {
    RBR_REQUIRE(n_docs >= 0 && doc_len >= 1 && vocab >= 1 && emb >= 1 && filters >= 1 && ksize >= 1 && pad >= 0 &&
                    argmax_ld >= filters && contrib_ld >= filters * ksize,
                RBR_EINVAL, "rbr_conv_window_contrib: bad shape (n_docs=%lld doc_len=%lld filters=%lld ksize=%lld pad=%lld "
                "argmax_ld=%lld contrib_ld=%lld)", (long long)n_docs, (long long)doc_len, (long long)filters, (long long)ksize,
                (long long)pad, (long long)argmax_ld, (long long)contrib_ld);
    if (n_docs == 0) return RBR_OK;
    RBR_REQUIRE(table && ids && packed && argmax && contrib, RBR_EINVAL, "rbr_conv_window_contrib: null pointer");
    const PackLayout L = pack_layout(emb, filters, ksize);
    const float* whke = reinterpret_cast<const float*>(reinterpret_cast<const uint8_t*>(packed) + L.off_hke);
    const int64_t warps = n_docs * filters;
    const int wpb = 8;
    conv_window_contrib_kernel<<<(unsigned)((warps + wpb - 1) / wpb), wpb * 32, 0, as_stream(stream)>>>(
        table, vocab, emb, id_view(ids, flags), mask, n_docs, doc_len, whke, L.Epad4, filters, ksize, pad, argmax, argmax_ld,
        contrib, contrib_ld);
    RBR_LAUNCH_CHECK("conv_window_contrib_kernel");
    return RBR_OK;
}

extern "C" int rbr_explain_attrib_ex(const int64_t* ent_row, int64_t n_rows, int64_t docs_per_entity, int64_t doc_len,
                                     const float* g, const float* feat, const int32_t* argmax, int64_t feat_ld,
                                     const float* contrib, int64_t contrib_ld, int64_t n_docs, int64_t n_conv,
                                     const int64_t* host_convs, const float* dense_coef, int64_t dense_coef_ld,
                                     const float* dense_vec, int64_t dense_vec_ld, int64_t m, int64_t width, float* text_total,
                                     int64_t* top_pos, float* top_attr, int64_t* bottom_pos, float* bottom_attr, float* map,
                                     float* review_attr, void* stream) {
    RBR_REQUIRE(docs_per_entity >= 1 && doc_len >= 1 &&
                    ex_supported(docs_per_entity * doc_len, m, width, n_conv),
                RBR_EUNSUPPORTED, "rbr_explain_attrib: need 1 <= docs_per_entity * doc_len <= %d, 1 <= m <= %d, 1 <= width <= %d, "
                "1 <= n_conv <= %d (got %lld x %lld, m=%lld, width=%lld, n_conv=%lld)", EX_MAX_POSITIONS, EX_MAX_M, EX_MAX_WIDTH,
                EX_MAX_CONVS, (long long)docs_per_entity, (long long)doc_len, (long long)m, (long long)width, (long long)n_conv);
    const bool dense = dense_coef != nullptr;
    const int64_t S = docs_per_entity * doc_len;
    const size_t smem = ex_smem_bytes(S, docs_per_entity, dense);
    RBR_REQUIRE(smem <= EX_MAX_SMEM, RBR_EUNSUPPORTED, "rbr_explain_attrib: %lld documents per entity with a dense term need "
                "%zu bytes of shared memory (at most %d)", (long long)docs_per_entity, smem, EX_MAX_SMEM);
    RBR_REQUIRE(host_convs, RBR_EINVAL, "rbr_explain_attrib: null host_convs");
    ExArgs a;
    a.cv.n = (int)n_conv;
    int64_t hcol = 0, ccol = 0;
    for (int c = 0; c < n_conv; ++c) {
        const int64_t h = host_convs[3 * c], k = host_convs[3 * c + 1], pd = host_convs[3 * c + 2];
        RBR_REQUIRE(h >= 1 && k >= 1 && pd >= 0, RBR_EINVAL, "rbr_explain_attrib: conv %d has filters=%lld ksize=%lld pad=%lld",
                    c, (long long)h, (long long)k, (long long)pd);
        a.cv.coff[c] = ccol;
        a.cv.k[c] = (int)k;
        a.cv.pad[c] = (int)pd;
        hcol += h;
        ccol += h * k;
        a.cv.h_end[c] = (int)hcol;
    }
    RBR_REQUIRE(feat_ld >= hcol && contrib_ld >= ccol && n_docs >= 0 && n_rows >= 0, RBR_EINVAL,
                "rbr_explain_attrib: feat_ld=%lld < %lld filters or contrib_ld=%lld < %lld taps", (long long)feat_ld,
                (long long)hcol, (long long)contrib_ld, (long long)ccol);
    RBR_REQUIRE(!dense || (dense_coef_ld >= hcol && dense_vec_ld >= doc_len), RBR_EINVAL,
                "rbr_explain_attrib: dense_coef_ld=%lld < %lld filters or dense_vec_ld=%lld < doc_len=%lld",
                (long long)dense_coef_ld, (long long)hcol, (long long)dense_vec_ld, (long long)doc_len);
    if (n_rows == 0) return RBR_OK;
    RBR_REQUIRE(ent_row && g && argmax && contrib && text_total && top_pos && top_attr && bottom_pos && bottom_attr &&
                    (!dense || dense_vec),
                RBR_EINVAL, "rbr_explain_attrib: null pointer");
    a.ent_row = ent_row; a.g = g; a.feat = feat; a.argmax = argmax; a.contrib = contrib;
    a.dense_coef = dense_coef; a.dense_vec = dense_vec; a.coef_ld = dense_coef_ld; a.vec_ld = dense_vec_ld;
    a.n_docs = n_docs; a.feat_ld = feat_ld; a.contrib_ld = contrib_ld; a.htot = hcol;
    a.R = (int)docs_per_entity; a.T = (int)doc_len; a.m = (int)m; a.width = (int)width;
    a.out = {text_total, top_pos, top_attr, bottom_pos, bottom_attr, map, review_attr};
    RBR_CUDA(cudaFuncSetAttribute(explain_attrib_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    explain_attrib_kernel<<<(unsigned)n_rows, EX_THREADS, smem, as_stream(stream)>>>(a);
    RBR_LAUNCH_CHECK("explain_attrib_kernel");
    return RBR_OK;
}

extern "C" int rbr_explain_attrib(const int64_t* ent_row, int64_t n_rows, int64_t docs_per_entity, int64_t doc_len,
                                  const float* g, const float* feat, const int32_t* argmax, int64_t feat_ld, const float* contrib,
                                  int64_t contrib_ld, int64_t n_docs, int64_t n_conv, const int64_t* host_convs, int64_t m,
                                  int64_t width, float* text_total, int64_t* top_pos, float* top_attr, int64_t* bottom_pos,
                                  float* bottom_attr, float* map, float* review_attr, void* stream) {
    return rbr_explain_attrib_ex(ent_row, n_rows, docs_per_entity, doc_len, g, feat, argmax, feat_ld, contrib, contrib_ld, n_docs,
                                 n_conv, host_convs, nullptr, 0, nullptr, 0, m, width, text_total, top_pos, top_attr, bottom_pos,
                                 bottom_attr, map, review_attr, stream);
}

static bool xa_supported(int64_t positions, int64_t reviews, int64_t emb, int64_t feat, int64_t m, int64_t width) {
    return reviews >= 1 && positions >= reviews && positions % reviews == 0 && emb >= 1 && feat >= 1 &&
           ex_supported(positions, m, width, 1) && xa_smem_bytes(reviews, positions / reviews, emb, feat) <= EX_MAX_SMEM;
}

extern "C" int rbr_explain_avgpool_supported(int64_t positions, int64_t reviews, int64_t emb, int64_t feat, int64_t m,
                                             int64_t width) {
    return xa_supported(positions, reviews, emb, feat, m, width) ? 1 : 0;
}

extern "C" int rbr_explain_avgpool_attrib(const float* table, int64_t vocab, int64_t emb, const void* ids, const uint8_t* mask,
                                          int64_t n_ent, int64_t reviews, int64_t doc_len, const int64_t* ent, int64_t n_rows,
                                          const float* g, const int64_t* other, const float* lat, const float* lat_other,
                                          int64_t n_other, const float* w_side, const float* fm_h, int64_t latent,
                                          const float* v, const float* att_a, const float* att_s, const float* f, int64_t feat,
                                          const float* lt_w, int64_t m, int64_t width, float* text_total, int64_t* top_pos,
                                          float* top_attr, int64_t* bottom_pos, float* bottom_attr, float* map,
                                          float* review_attr, int flags, void* stream) {
    RBR_REQUIRE(reviews >= 1 && doc_len >= 1 && xa_supported(reviews * doc_len, reviews, emb, feat, m, width), RBR_EUNSUPPORTED,
                "rbr_explain_avgpool_attrib: need 1 <= reviews * doc_len <= %d, 1 <= m <= %d, 1 <= width <= %d and %lld bytes "
                "of shared memory at most %d (got %lld x %lld, emb=%lld, feat=%lld, m=%lld, width=%lld)", EX_MAX_POSITIONS,
                EX_MAX_M, EX_MAX_WIDTH, (long long)(reviews >= 1 && doc_len >= 1 ? xa_smem_bytes(reviews, doc_len, emb, feat) : 0),
                EX_MAX_SMEM, (long long)reviews, (long long)doc_len, (long long)emb, (long long)feat, (long long)m,
                (long long)width);
    RBR_REQUIRE(n_ent >= 0 && n_rows >= 0 && vocab >= 1 && (lt_w || feat == emb) && (g || (latent >= 1 && n_other >= 0)),
                RBR_EINVAL, "rbr_explain_avgpool_attrib: bad shape (n_ent=%lld n_rows=%lld vocab=%lld emb=%lld feat=%lld "
                "latent=%lld; without the latent transform feat must equal emb)", (long long)n_ent, (long long)n_rows,
                (long long)vocab, (long long)emb, (long long)feat, (long long)latent);
    if (n_rows == 0) return RBR_OK;
    RBR_REQUIRE(table && ids && ent && v && att_a && att_s && f && text_total && top_pos && top_attr && bottom_pos &&
                    bottom_attr && (g || (other && lat && lat_other && w_side && fm_h)),
                RBR_EINVAL, "rbr_explain_avgpool_attrib: null pointer");
    XaArgs a;
    a.table = table; a.vocab = vocab; a.emb = emb; a.iv = id_view(ids, flags); a.mask = mask; a.n_ent = n_ent;
    a.R = (int)reviews; a.T = (int)doc_len; a.F = (int)feat; a.K = g ? 0 : (int)latent;
    a.ent = ent; a.g = g; a.other = other; a.lat = lat; a.lat_other = lat_other; a.n_other = n_other;
    a.w_side = w_side; a.fm_h = fm_h;
    a.v = v; a.att_a = att_a; a.att_s = att_s; a.f = f; a.lt_w = lt_w;
    a.m = (int)m; a.width = (int)width;
    a.out = {text_total, top_pos, top_attr, bottom_pos, bottom_attr, map, review_attr};
    const size_t smem = (size_t)xa_smem_bytes(reviews, doc_len, emb, feat);
    RBR_CUDA(cudaFuncSetAttribute(explain_avgpool_attrib_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    explain_avgpool_attrib_kernel<<<(unsigned)n_rows, EX_THREADS, smem, as_stream(stream)>>>(a);
    RBR_LAUNCH_CHECK("explain_avgpool_attrib_kernel");
    return RBR_OK;
}

extern "C" int rbr_datt_explain_contrib(const float* table, int64_t vocab, int64_t emb, const void* ids, int64_t n_docs,
                                        int64_t doc_len, const float* w_local_t, int64_t window, const float* w_global_t,
                                        const void* packed_local, int64_t l_out, const void* packed_g2, const void* packed_g3,
                                        const void* packed_g4, int64_t g_out, const float* gate_local, const float* gate_global,
                                        const float* feat, const int32_t* argmax, int64_t feat_ld, float* contrib,
                                        int64_t contrib_ld, float* gate_coef, int64_t coef_ld, float* gate_vec, int64_t vec_ld,
                                        int flags, void* stream) {
    RBR_REQUIRE(window >= 1 && window <= EX_MAX_WIDTH && window % 2 == 1 && doc_len >= 4, RBR_EUNSUPPORTED,
                "rbr_datt_explain_contrib: need an odd window <= %d and doc_len >= 4 (got window=%lld doc_len=%lld)", EX_MAX_WIDTH,
                (long long)window, (long long)doc_len);
    const int64_t htot = l_out + 3 * g_out, taps = l_out * window + g_out * (2 + 3 + 4);
    RBR_REQUIRE(n_docs >= 0 && vocab >= 1 && emb >= 1 && l_out >= 1 && g_out >= 1 && feat_ld >= htot && contrib_ld >= taps &&
                    coef_ld >= htot && vec_ld >= doc_len && htot < (1ll << 30),
                RBR_EINVAL, "rbr_datt_explain_contrib: bad shape (n_docs=%lld l_out=%lld g_out=%lld feat_ld=%lld contrib_ld=%lld "
                "coef_ld=%lld vec_ld=%lld)", (long long)n_docs, (long long)l_out, (long long)g_out, (long long)feat_ld,
                (long long)contrib_ld, (long long)coef_ld, (long long)vec_ld);
    if (n_docs == 0) return RBR_OK;
    RBR_REQUIRE(table && ids && w_local_t && w_global_t && packed_local && packed_g2 && packed_g3 && packed_g4 && gate_local &&
                    gate_global && feat && argmax && contrib && gate_coef && gate_vec,
                RBR_EINVAL, "rbr_datt_explain_contrib: null pointer");
    DattExArgs a;
    a.table = table; a.vocab = vocab; a.emb = emb; a.n_docs = n_docs; a.L = doc_len;
    a.iv = id_view(ids, flags & RBR_IDS_I32);                       // D-ATT has no masks
    a.wlT = w_local_t; a.wgT = w_global_t; a.kl = (int)window;
    const void* packs[4] = {packed_local, packed_g2, packed_g3, packed_g4};
    int64_t hcol = 0, ccol = 0;
    for (int c = 0; c < 4; ++c) {
        const int64_t h = c ? g_out : l_out, k = c ? c + 1 : 1;
        const PackLayout L = pack_layout(emb, h, k);
        a.whke[c] = reinterpret_cast<const float*>(reinterpret_cast<const uint8_t*>(packs[c]) + L.off_hke);
        a.epad4[c] = L.Epad4;
        a.k[c] = (int)k;
        a.coff[c] = ccol;
        hcol += h;
        ccol += h * (c ? k : window);
        a.h_end[c] = (int)hcol;
    }
    a.gate_l = gate_local; a.gate_g = gate_global; a.feat = feat; a.argmax = argmax; a.feat_ld = feat_ld;
    a.contrib = contrib; a.contrib_ld = contrib_ld; a.gate_coef = gate_coef; a.coef_ld = coef_ld;
    a.gate_vec = gate_vec; a.vec_ld = vec_ld;
    const int64_t warps = n_docs * (htot + doc_len);
    const int wpb = 8;
    datt_explain_contrib_kernel<<<(unsigned)((warps + wpb - 1) / wpb), wpb * 32, 0, as_stream(stream)>>>(a);
    RBR_LAUNCH_CHECK("datt_explain_contrib_kernel");
    return RBR_OK;
}

extern "C" int rbr_datt_fc_grads(const int64_t* u_ids, const int64_t* i_ids, int64_t n_pairs, const float* user_out,
                                 int64_t n_users, const float* item_out, int64_t n_items, int64_t out_dim, const uint8_t* user_mask,
                                 const uint8_t* item_mask, int64_t hidden, const float* w0, int64_t in_dim, const float* w3,
                                 float* g_user, float* g_item, void* stream) {
    RBR_REQUIRE(hidden >= 1 && hidden <= FG_MAX_HIDDEN && out_dim >= 1 && in_dim >= 1, RBR_EUNSUPPORTED,
                "rbr_datt_fc_grads: need 1 <= hidden <= %d, out_dim >= 1, in_dim >= 1 (got %lld, %lld, %lld)", FG_MAX_HIDDEN,
                (long long)hidden, (long long)out_dim, (long long)in_dim);
    RBR_REQUIRE(n_pairs >= 0 && n_users >= 0 && n_items >= 0, RBR_EINVAL, "rbr_datt_fc_grads: bad shape");
    if (n_pairs == 0) return RBR_OK;
    RBR_REQUIRE(u_ids && i_ids && user_out && item_out && user_mask && item_mask && w0 && w3 && g_user && g_item, RBR_EINVAL,
                "rbr_datt_fc_grads: null pointer");
    FgArgs a;
    a.ids[0] = u_ids; a.ids[1] = i_ids; a.P = n_pairs;
    a.out[0] = user_out; a.out[1] = item_out; a.n_ent[0] = n_users; a.n_ent[1] = n_items; a.out_dim = out_dim;
    a.mask[0] = user_mask; a.mask[1] = item_mask; a.hidden = hidden;
    a.w0 = w0; a.in_dim = in_dim; a.w3 = w3; a.g[0] = g_user; a.g[1] = g_item;
    a.kp = (int)fg_kpad(hidden);
    a.vs = (int)fg_stride(hidden);
    const size_t smem = (size_t)FG_BM * a.vs * 4;
    RBR_CUDA(cudaFuncSetAttribute(datt_fc_grads_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const dim3 grid((unsigned)((n_pairs + FG_BM - 1) / FG_BM), 2);
    datt_fc_grads_kernel<<<grid, FG_THREADS, smem, as_stream(stream)>>>(a);
    RBR_LAUNCH_CHECK("datt_fc_grads_kernel");
    return RBR_OK;
}
