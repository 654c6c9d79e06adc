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

static bool ex_supported(int64_t positions, int64_t m, int64_t width, int64_t n_conv) {
    return positions >= 1 && positions <= EX_MAX_POSITIONS && m >= 1 && m <= EX_MAX_M && width >= 1 && width <= EX_MAX_WIDTH &&
           n_conv >= 1 && n_conv <= EX_MAX_CONVS;
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
        // the row the forward multiplies: zero outside the document, at masked positions and for ids outside the table
        // (conv_fp32.cu's row resolution); any arg-max value is therefore memory-safe
        const int64_t t = t0 + j;
        int64_t row = -1;
        if (t >= 0 && t < doc_len) {
            const int64_t id = ld_id(iv, n * doc_len + t);
            if (ld_mask(iv, mask, n * doc_len + t, id) && id >= 0 && id < vocab) row = id;
        }
        float s = 0.f;
        if (row >= 0) {
            const float* x = table + row * emb;
            const float* w = whke + (h * ksize + j) * epad4;
            for (int64_t e = lane; e < emb; e += 32) s = fmaf(__ldg(x + e), __ldg(w + e), s);
        }
        s = warp_sum(s);
        if (lane == 0) contrib[n * contrib_ld + h * ksize + j] = s;
    }
}

// ---- per (pair, side) row: attribution map, total, per-review sums, top / bottom windows ------------------------------------
struct ExConvs {
    int n;
    int h_end[EX_MAX_CONVS];   // filter column where conv c ends (exclusive), within feat / argmax / g rows
    int k[EX_MAX_CONVS], pad[EX_MAX_CONVS];
    int64_t coff[EX_MAX_CONVS];   // column of conv c's first tap within a contribution row
};

struct ExArgs {
    const int64_t* ent_row;
    const float* g;          // [P, R, Htot]
    const float* feat;       // [n_docs, feat_ld]
    const int32_t* argmax;   // [n_docs, feat_ld]
    const float* contrib;    // [n_docs, contrib_ld]
    int64_t n_docs, feat_ld, contrib_ld, htot;
    int R, T, m, width;
    ExConvs cv;
    float* text_total;       // [P]
    int64_t* top_pos; float* top_attr; int64_t* bot_pos; float* bot_attr;   // [P, m]
    float* map;              // [P, R*T] or NULL
    float* review_attr;      // [P, R] or NULL
};

__device__ __forceinline__ int ex_conv_of(const ExConvs& cv, int hh) {
    int c = 0;
    while (c + 1 < cv.n && hh >= cv.h_end[c]) ++c;
    return c;
}

// block-wide reductions (EX_THREADS threads); `red` holds EX_THREADS / 32 entries of the widest type
__device__ float ex_block_max(float v, double* red) {
    v = warp_max(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    float r = 0.f;
    for (int w = 0; w < EX_THREADS / 32; ++w) r = fmaxf(r, (float)red[w]);
    return r;
}

__device__ long long ex_warp_sum_ll(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ long long ex_block_sum_ll(long long v, double* red) {
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

__device__ void ex_block_pick(double& v, int& s, bool top, double* red_v, int* red_s) {
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

__global__ void __launch_bounds__(EX_THREADS) explain_attrib_kernel(const ExArgs a) {
    extern __shared__ __align__(16) unsigned char ex_smem[];
    __shared__ double red_v[EX_THREADS / 32];
    __shared__ int red_s[EX_THREADS / 32];
    const int S = a.R * a.T;
    long long* acc = reinterpret_cast<long long*>(ex_smem);          // [S] fixed-point map; later the window sums (double)
    float* mapf = reinterpret_cast<float*>(acc + S);                  // [S]
    uint8_t* avail = reinterpret_cast<uint8_t*>(mapf + S);            // [S] window start still selectable
    const int64_t p = blockIdx.x;
    const int64_t row0 = __ldg(a.ent_row + p);
    const bool ok = row0 >= 0 && row0 + a.R <= a.n_docs;              // the host validates; a bad row yields NaN / -1, no read
    const int n_items = a.R * (int)a.htot;
    const float* gp = a.g + p * n_items;

    for (int i = threadIdx.x; i < S; i += EX_THREADS) acc[i] = 0;
    // pass 1: the largest |g * c| of a live term bounds the total, which fixes the fixed-point scale
    float mx = 0.f;
    int max_k = 0;
    for (int c = 0; c < a.cv.n; ++c) max_k = max(max_k, a.cv.k[c]);
    if (ok) {
        for (int i = threadIdx.x; i < n_items; i += EX_THREADS) {
            const int r = i / (int)a.htot, hh = i % (int)a.htot;
            const int64_t doc = row0 + r;
            if (!(__ldg(a.feat + doc * a.feat_ld + hh) > 0.f)) continue;
            const float gv = __ldg(gp + i);
            const int c = ex_conv_of(a.cv, hh);
            const int h = hh - (c ? a.cv.h_end[c - 1] : 0);
            const float* cp = a.contrib + doc * a.contrib_ld + a.cv.coff[c] + (int64_t)h * a.cv.k[c];
            for (int j = 0; j < a.cv.k[c]; ++j) mx = fmaxf(mx, fabsf(gv * __ldg(cp + j)));
        }
    }
    mx = ex_block_max(mx, red_v);
    // |total| <= n_items * max_k * mx < 2^e  →  terms on a grid of 2^(e-61): every partial sum stays below 2^61 in magnitude
    double scale = 0.0;
    if (mx > 0.f && isfinite(mx)) {
        int e;
        frexp((double)mx * (double)n_items * (double)max_k, &e);
        scale = ldexp(1.0, 61 - e);
    }
    __syncthreads();
    // pass 2: scatter the rounded terms; every term enters the total, the ones at a position inside the document also the map
    long long tot = 0;
    if (ok && scale > 0.0) {
        for (int i = threadIdx.x; i < n_items; i += EX_THREADS) {
            const int r = i / (int)a.htot, hh = i % (int)a.htot;
            const int64_t doc = row0 + r;
            if (!(__ldg(a.feat + doc * a.feat_ld + hh) > 0.f)) continue;
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
    const float nanf_ = __int_as_float(0x7fc00000);
    const double inv = scale > 0.0 ? 1.0 / scale : 0.0;
    if (threadIdx.x == 0) a.text_total[p] = ok ? (float)((double)tot * inv) : nanf_;
    __syncthreads();                                                   // the atomics have landed
    for (int i = threadIdx.x; i < S; i += EX_THREADS) {
        const float v = ok ? (float)((double)acc[i] * inv) : nanf_;
        mapf[i] = v;
        if (a.map) a.map[p * S + i] = v;
    }
    if (a.review_attr) {
        for (int r = threadIdx.x >> 5; r < a.R; r += EX_THREADS / 32) {
            long long s = 0;
            for (int t = threadIdx.x & 31; t < a.T; t += 32) s += acc[r * a.T + t];
            s = ex_warp_sum_ll(s);
            if ((threadIdx.x & 31) == 0) a.review_attr[p * a.R + r] = ok ? (float)((double)s * inv) : nanf_;
        }
    }
    __syncthreads();                                                   // acc is read for the last time above
    double* wsum = reinterpret_cast<double*>(acc);
    const int w = a.width;
    for (int s = threadIdx.x; s < S; s += EX_THREADS) {
        double v = 0.0;
        if ((s % a.T) + w <= a.T)
            for (int j = 0; j < w; ++j) v += (double)mapf[s + j];
        wsum[s] = v;
    }
    for (int pass = 0; pass < 2; ++pass) {
        const bool top = pass == 0;
        int64_t* out_pos = (top ? a.top_pos : a.bot_pos) + p * a.m;
        float* out_attr = (top ? a.top_attr : a.bot_attr) + p * a.m;
        for (int s = threadIdx.x; s < S; s += EX_THREADS) avail[s] = ok && (s % a.T) + w <= a.T;
        __syncthreads();
        for (int it = 0; it < a.m; ++it) {
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
                for (int j = it + 1 + (int)threadIdx.x; j < a.m; j += EX_THREADS) { out_pos[j] = -1; out_attr[j] = nanf_; }
                break;
            }
            // windows never cross a review boundary, so every start whose window overlaps [bs, bs + w) lies in (bs - w, bs + w)
            for (int s = max(0, bs - w + 1) + (int)threadIdx.x; s < min(S, bs + w); s += EX_THREADS) avail[s] = 0;
            __syncthreads();
        }
        __syncthreads();
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

extern "C" int rbr_explain_attrib(const int64_t* ent_row, int64_t n_rows, int64_t docs_per_entity, int64_t doc_len,
                                  const float* g, const float* feat, const int32_t* argmax, int64_t feat_ld, const float* contrib,
                                  int64_t contrib_ld, int64_t n_docs, int64_t n_conv, const int64_t* host_convs, int64_t m,
                                  int64_t width, float* text_total, int64_t* top_pos, float* top_attr, int64_t* bottom_pos,
                                  float* bottom_attr, float* map, float* review_attr, void* stream) {
    RBR_REQUIRE(docs_per_entity >= 1 && doc_len >= 1 &&
                    ex_supported(docs_per_entity * doc_len, m, width, n_conv),
                RBR_EUNSUPPORTED, "rbr_explain_attrib: need 1 <= docs_per_entity * doc_len <= %d, 1 <= m <= %d, 1 <= width <= %d, "
                "1 <= n_conv <= %d (got %lld x %lld, m=%lld, width=%lld, n_conv=%lld)", EX_MAX_POSITIONS, EX_MAX_M, EX_MAX_WIDTH,
                EX_MAX_CONVS, (long long)docs_per_entity, (long long)doc_len, (long long)m, (long long)width, (long long)n_conv);
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
    if (n_rows == 0) return RBR_OK;
    RBR_REQUIRE(ent_row && g && feat && argmax && contrib && text_total && top_pos && top_attr && bottom_pos && bottom_attr,
                RBR_EINVAL, "rbr_explain_attrib: null pointer");
    a.ent_row = ent_row; a.g = g; a.feat = feat; a.argmax = argmax; a.contrib = contrib;
    a.n_docs = n_docs; a.feat_ld = feat_ld; a.contrib_ld = contrib_ld; a.htot = hcol;
    a.R = (int)docs_per_entity; a.T = (int)doc_len; a.m = (int)m; a.width = (int)width;
    a.text_total = text_total; a.top_pos = top_pos; a.top_attr = top_attr; a.bot_pos = bottom_pos; a.bot_attr = bottom_attr;
    a.map = map; a.review_attr = review_attr;
    const int64_t S = docs_per_entity * doc_len;
    const size_t smem = (size_t)S * (8 + 4 + 1);
    RBR_CUDA(cudaFuncSetAttribute(explain_attrib_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    explain_attrib_kernel<<<(unsigned)n_rows, EX_THREADS, smem, as_stream(stream)>>>(a);
    RBR_LAUNCH_CHECK("explain_attrib_kernel");
    return RBR_OK;
}
