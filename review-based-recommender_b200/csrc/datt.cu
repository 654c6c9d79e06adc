// datt.cu — D-ATT gates: the two attention convolutions of the dual-attention encoder, forward and backward.
//
// Replaces LocalAttention.attn  = Sequential(Conv1d(E, 1, k=window, padding=(window-1)/2), Sigmoid)
//          (reference models/dual_att/layers.py:34-36, applied :49) → one gate per token, [N, L]
// and      GlobalAttention.attn = Sequential(Conv1d(E, 1, k=doc_len), Sigmoid)
//          (models/dual_att/layers.py:65-67, applied :83)          → ONE gate per document, [N]
// computed straight from the token ids and the fp32 table: the [N,E,L] permuted copy of the embeddings
// (layers.py:48,82) and the gated copies score*x (layers.py:50,84) are never materialised — the gated convolutions
// apply the gate inside the conv kernels (conv_fp32.cu / conv_tc.cu, gate_mode 1 / 2).
// All kernels are L2/HBM-bound gathers of 4*E-byte rows; E <= 128, E % 4 == 0 (D-ATT's emb_size is 100).
#include "rbr_common.cuh"
#include "token_sort.cuh"

namespace rbr {

constexpr int DA_WARPS = 8;
constexpr int DA_MAXWIN = 8;

__device__ __forceinline__ float sigmoidf_(float z) { return 1.f / (1.f + expf(-z)); }
__device__ __forceinline__ float dot4(const float4& a, const float4& b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; }
__device__ __forceinline__ void fma4(float4& acc, float s, const float4& v) {
    acc.x = fmaf(s, v.x, acc.x); acc.y = fmaf(s, v.y, acc.y); acc.z = fmaf(s, v.z, acc.z); acc.w = fmaf(s, v.w, acc.w);
}

// elements 4*lane .. 4*lane+3 of a table row of E floats (zero beyond E).  V4: E % 4 == 0 → one 16-byte load.
template <bool V4>
__device__ __forceinline__ float4 ld_row4(const float* __restrict__ row, int E, int lane) {
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    const int e = lane * 4;
    if (V4) {
        if (e < E) x = __ldg(reinterpret_cast<const float4*>(row) + lane);
    } else {
        if (e < E) x.x = __ldg(row + e);
        if (e + 1 < E) x.y = __ldg(row + e + 1);
        if (e + 2 < E) x.z = __ldg(row + e + 2);
        if (e + 3 < E) x.w = __ldg(row + e + 3);
    }
    return x;
}
template <bool V4>
__device__ __forceinline__ void atomic_add_row4(float* __restrict__ row, int E, int lane, const float4& v) {
    const int e = lane * 4;
    if (V4) {
        if (e < E) atomicAdd(reinterpret_cast<float4*>(row) + lane, v);
    } else {
        if (e < E) atomicAdd(row + e, v.x);
        if (e + 1 < E) atomicAdd(row + e + 1, v.y);
        if (e + 2 < E) atomicAdd(row + e + 2, v.z);
        if (e + 3 < E) atomicAdd(row + e + 3, v.w);
    }
}

// w [1][E][K] (nn.Conv1d) → wT [K][Ep], Ep = E rounded up to 4, zero padded (rows stay 16-byte aligned)
__global__ void datt_transpose_kernel(const float* __restrict__ w, int E, int Ep, int K, float* __restrict__ wT) {
    const int total = Ep * K;
    for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < total; q += gridDim.x * blockDim.x) {
        const int e = q % Ep, k = q / Ep;
        wT[q] = e < E ? w[e * K + k] : 0.f;
    }
}

// one CTA per document: warp w takes tokens w, w+8, ...; lane c owns elements 4c..4c+3 of the row
template <bool V4, int WIN>
__global__ void __launch_bounds__(DA_WARPS * 32) datt_gate_fwd_kernel(
    const float* __restrict__ table, int64_t vocab, int E, const IdView ids, int L, const float* __restrict__ waT,
    const float* __restrict__ b_local, int win, const float* __restrict__ wgT, const float* __restrict__ b_global,
    float* __restrict__ gate_local, float* __restrict__ gate_global) {
    extern __shared__ __align__(16) float smem[];
    float* dloc = smem;                        // [win][L]   d_j(t) = Wa[:, j] . x_t
    const int Ep = (E + 3) & ~3;
    float* wa_s = dloc + ((win * L + 3) & ~3); // [win][Ep]
    float* gpart = wa_s + win * Ep;            // [DA_WARPS]
    const int64_t n = blockIdx.x;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int e4 = Ep >> 2;
    for (int i = threadIdx.x; i < win * Ep; i += blockDim.x) wa_s[i] = waT[i];
    __syncthreads();
    float gacc = 0.f;
    // The `win` window dot products of a token are reduced TOGETHER: a transposed butterfly (8 values → 4 → 2 → 1 per lane
    // over the xor-16/8/4 steps, then two plain steps) needs 9 shuffles instead of 5 per value; afterwards the lane whose
    // bits (4,3,2) spell j holds d_j.  (The kernel was issue-bound: 242 warp instructions per token, mostly reductions.)
    const int my_j = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
    for (int t = wib; t < L; t += DA_WARPS) {
        const int64_t id = ld_id(ids, n * L + t);
        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
        const bool ok = id >= 0 && id < vocab;
        if (!ok && lane == 0) note_oob();
        if (ok) x = ld_row4<V4>(table + id * E, E, lane);
        if (lane < e4) gacc += dot4(x, __ldg(reinterpret_cast<const float4*>(wgT + (int64_t)t * Ep) + lane));
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j)
            v[j] = (j < WIN && lane < e4) ? dot4(x, *reinterpret_cast<const float4*>(wa_s + j * Ep + lane * 4)) : 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {                                  // xor 16: 8 → 4 values
            const bool up = lane & 16;
            const float keep = up ? v[i + 4] : v[i], send = up ? v[i] : v[i + 4];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {                                  // xor 8: 4 → 2
            const bool up = lane & 8;
            const float keep = up ? v[i + 2] : v[i], send = up ? v[i] : v[i + 2];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
        {                                                              // xor 4: 2 → 1
            const bool up = lane & 4;
            const float keep = up ? v[1] : v[0], send = up ? v[0] : v[1];
            v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
        }
        v[0] += __shfl_xor_sync(0xffffffffu, v[0], 2);
        v[0] += __shfl_xor_sync(0xffffffffu, v[0], 1);
        if ((lane & 3) == 0 && my_j < WIN) dloc[my_j * L + t] = v[0];
    }
    gacc = warp_sum(gacc);
    if (lane == 0) gpart[wib] = gacc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float z = b_global[0];
        for (int w = 0; w < DA_WARPS; ++w) z += gpart[w];
        gate_global[n] = sigmoidf_(z);
    }
    const int pad = (win - 1) / 2;
    for (int t = threadIdx.x; t < L; t += blockDim.x) {
        float z = b_local[0];
        for (int j = 0; j < win; ++j) {
            const int tp = t + j - pad;                       // out[t] = b + sum_j W[:, j] . x[t + j - pad]
            if (tp >= 0 && tp < L) z += dloc[j * L + tp];
        }
        gate_local[n * L + t] = sigmoidf_(z);
    }
}

// dz = d gate * gate * (1 - gate); bias grads; sort keys (token id, or -1 for the padding row / bad ids)
__global__ void __launch_bounds__(256) datt_gate_dz_kernel(const IdView ids, int64_t n_docs, int L, int64_t vocab,
                                                           int64_t padding_idx, const float* __restrict__ gl,
                                                           const float* __restrict__ gg, const float* __restrict__ gl_grad,
                                                           const float* __restrict__ gg_grad, float* __restrict__ dz_l,
                                                           float* __restrict__ dz_g, int32_t* __restrict__ keys,
                                                           float* __restrict__ b_local_grad, float* __restrict__ b_global_grad) {
    const int64_t total = n_docs * L;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    float sl = 0.f, sg = 0.f;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += stride) {
        const float g = gl[q];
        const float d = gl_grad[q] * g * (1.f - g);
        dz_l[q] = d;
        sl += d;
        const int64_t id = ld_id(ids, q);
        keys[q] = (id >= 0 && id < vocab && id != padding_idx) ? (int32_t)id : -1;
        if (q < n_docs) {
            const float g2 = gg[q];
            const float d2 = gg_grad[q] * g2 * (1.f - g2);
            dz_g[q] = d2;
            sg += d2;
        }
    }
    sl = warp_sum(sl);
    sg = warp_sum(sg);
    if ((threadIdx.x & 31) == 0) {
        if (sl != 0.f) atomicAdd(b_local_grad, sl);
        if (sg != 0.f) atomicAdd(b_global_grad, sg);
    }
}

// one CTA per position t: sums over all documents
//   w_global_grad[e, t]  = sum_n dz_g[n] * x[n, t, e]
//   w_local_grad[e, j]  += sum_n dz_l[n, t - j + pad] * x[n, t, e]
template <int WIN, bool V4>
__global__ void __launch_bounds__(DA_WARPS * 32) datt_gate_wgrad_kernel(const float* __restrict__ table, int64_t vocab, int E,
                                                                        const IdView ids, int64_t n_docs, int L,
                                                                        const float* __restrict__ dz_l, const float* __restrict__ dz_g,
                                                                        float* __restrict__ w_local_grad /*[E][WIN]*/,
                                                                        float* __restrict__ w_global_grad /*[E][L]*/) {
    __shared__ float4 red[DA_WARPS][WIN + 1][32];
    const int t = blockIdx.x;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int e4 = (E + 3) >> 2;
    constexpr int pad = (WIN - 1) / 2;
    float4 accg = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 acca[WIN];
#pragma unroll
    for (int j = 0; j < WIN; ++j) acca[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int64_t nb = wib * 32; nb < n_docs; nb += DA_WARPS * 32) {
        // lane l resolves document nb+l (id and coefficients), then the warp walks the 32 documents
        const int64_t n = nb + lane;
        int64_t id_l = -1;
        float zg_l = 0.f, zl_l[WIN];
#pragma unroll
        for (int j = 0; j < WIN; ++j) zl_l[j] = 0.f;
        if (n < n_docs) {
            const int64_t id = ld_id(ids, n * L + t);
            if (id >= 0 && id < vocab) id_l = id;
            zg_l = dz_g[n];
#pragma unroll
            for (int j = 0; j < WIN; ++j) {
                const int to = t - j + pad;                    // output position whose window reads x[t] at tap j
                if (to >= 0 && to < L) zl_l[j] = dz_l[n * L + to];
            }
        }
        const int cnt = (int)min((int64_t)32, n_docs - nb);
#pragma unroll 2
        for (int d = 0; d < cnt; ++d) {
            const int64_t id = __shfl_sync(0xffffffffu, id_l, d);
            if (id < 0) continue;
            const float4 x = ld_row4<V4>(table + id * E, E, lane);
            fma4(accg, __shfl_sync(0xffffffffu, zg_l, d), x);
#pragma unroll
            for (int j = 0; j < WIN; ++j) fma4(acca[j], __shfl_sync(0xffffffffu, zl_l[j], d), x);
        }
    }
    red[wib][0][lane] = accg;
#pragma unroll
    for (int j = 0; j < WIN; ++j) red[wib][j + 1][lane] = acca[j];
    __syncthreads();
    for (int o = threadIdx.x; o < (WIN + 1) * e4; o += blockDim.x) {
        const int which = o / e4, c = o - which * e4;
        float4 s = red[0][which][c];
        for (int w = 1; w < DA_WARPS; ++w) {
            const float4 v = red[w][which][c];
            s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
        }
        const float vals[4] = {s.x, s.y, s.z, s.w};
        for (int i = 0; i < 4; ++i) {
            const int e = c * 4 + i;
            if (e >= E) break;
            if (which == 0) w_global_grad[(int64_t)e * L + t] += vals[i];           // this CTA owns column t
            else if (vals[i] != 0.f) atomicAdd(w_local_grad + e * WIN + (which - 1), vals[i]);
        }
    }
}

// table gradient of both gates (warp-segmented scatter-add over token-sorted positions):
//   table_grad[ids[n,t], :] += dz_g[n] * Wg[:, t] + sum_j dz_l[n, t - j + pad] * Wa[:, j]
template <int WIN, bool V4>
__global__ void __launch_bounds__(256) datt_gate_table_kernel(const int32_t* __restrict__ order, const int32_t* __restrict__ keys,
                                                              int64_t n_tok, const int32_t* __restrict__ n_kept, int L, int E,
                                                              const float* __restrict__ dz_l, const float* __restrict__ dz_g,
                                                              const float* __restrict__ waT, const float* __restrict__ wgT,
                                                              float* __restrict__ table_grad) {
    const int lane = threadIdx.x & 31;
    const int Ep = (E + 3) & ~3;
    const int e4 = Ep >> 2;
    constexpr int pad = (WIN - 1) / 2;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    n_tok = min(n_tok, (int64_t)__ldg(n_kept));
    const int64_t i0 = warp * 32;
    if (i0 >= n_tok) return;
    float4 wa[WIN];
#pragma unroll
    for (int j = 0; j < WIN; ++j) wa[j] = (lane < e4) ? __ldg(reinterpret_cast<const float4*>(waT + j * Ep) + lane) : make_float4(0.f, 0.f, 0.f, 0.f);
    int key_l = -1, t_l = 0;
    float zg_l = 0.f, zl_l[WIN];
#pragma unroll
    for (int j = 0; j < WIN; ++j) zl_l[j] = 0.f;
    if (i0 + lane < n_tok) {
        const int tok = __ldg(order + i0 + lane);
        key_l = __ldg(keys + tok);
        const int64_t n = tok / L;
        t_l = tok - (int)(n * L);
        zg_l = __ldg(dz_g + n);
#pragma unroll
        for (int j = 0; j < WIN; ++j) {
            const int to = t_l - j + pad;
            if (to >= 0 && to < L) zl_l[j] = __ldg(dz_l + n * L + to);
        }
    }
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int cur = -1;
#pragma unroll 2
    for (int d = 0; d < 32; ++d) {
        const int key = __shfl_sync(0xffffffffu, key_l, d);
        if (key < 0) break;
        const int t = __shfl_sync(0xffffffffu, t_l, d);
        float4 wg = make_float4(0.f, 0.f, 0.f, 0.f);
        if (lane < e4) wg = __ldg(reinterpret_cast<const float4*>(wgT + (int64_t)t * Ep) + lane);
        if (key != cur) {
            if (cur >= 0) atomic_add_row4<V4>(table_grad + (int64_t)cur * E, E, lane, acc);
            acc = make_float4(0.f, 0.f, 0.f, 0.f);
            cur = key;
        }
        fma4(acc, __shfl_sync(0xffffffffu, zg_l, d), wg);
#pragma unroll
        for (int j = 0; j < WIN; ++j) fma4(acc, __shfl_sync(0xffffffffu, zl_l[j], d), wa[j]);
    }
    if (cur >= 0) atomic_add_row4<V4>(table_grad + (int64_t)cur * E, E, lane, acc);
}

struct DattWs {
    float *waT, *wgT, *dz_l, *dz_g;
    int32_t* keys;
    void* sort;
    int64_t total;
};
static DattWs datt_ws(void* base, int64_t n_docs, int64_t L, int64_t E, int64_t win, int64_t vocab) {
    char* p = reinterpret_cast<char*>(base);
    int64_t off = 0;
    DattWs w;
    const int64_t Ep = round_up(E, 4);
    w.waT = reinterpret_cast<float*>(p + off); off += round_up(win * Ep * 4, 256);
    w.wgT = reinterpret_cast<float*>(p + off); off += round_up(L * Ep * 4, 256);
    w.dz_l = reinterpret_cast<float*>(p + off); off += round_up(n_docs * L * 4, 256);
    w.dz_g = reinterpret_cast<float*>(p + off); off += round_up(n_docs * 4, 256);
    w.keys = reinterpret_cast<int32_t*>(p + off); off += round_up(n_docs * L * 4, 256);
    w.sort = p + off; off += token_sort_workspace_bytes(n_docs * L, vocab);
    w.total = off;
    return w;
}

}  // namespace rbr

using namespace rbr;

static int datt_check(int64_t emb, int64_t doc_len, int64_t window, const char* who) {
    RBR_REQUIRE(emb > 0 && emb <= 128, RBR_EUNSUPPORTED, "%s: emb_size must be <= 128", who);
    RBR_REQUIRE(window >= 1 && window <= DA_MAXWIN && window % 2 == 1, RBR_EUNSUPPORTED, "%s: window must be odd and <= %d", who,
                DA_MAXWIN);
    RBR_REQUIRE(doc_len > 0, RBR_EINVAL, "%s: bad doc_len", who);
    return RBR_OK;
}

extern "C" int64_t rbr_datt_gate_workspace_bytes(int64_t n_docs, int64_t doc_len, int64_t emb, int64_t window, int64_t vocab) {
    return datt_ws(nullptr, n_docs, doc_len, emb, window, vocab).total;
}

extern "C" int rbr_datt_gate_fwd(const float* table, int64_t vocab, int64_t emb, const void* ids_raw, int64_t n_docs,
                                 int64_t doc_len, const float* w_local, const float* b_local, int64_t window,
                                 const float* w_global, const float* b_global, float* gate_local, float* gate_global, void* ws,
                                 int64_t ws_bytes, int flags, void* stream) {
    int rc = datt_check(emb, doc_len, window, "rbr_datt_gate_fwd");
    if (rc != RBR_OK) return rc;
    if (n_docs == 0) return RBR_OK;
    const IdView ids = id_view(ids_raw, flags);
    RBR_REQUIRE(table && ids_raw && w_local && b_local && w_global && b_global && gate_local && gate_global && ws, RBR_EINVAL,
                "rbr_datt_gate_fwd: null pointer");
    RBR_REQUIRE(ws_bytes >= rbr_datt_gate_workspace_bytes(n_docs, doc_len, emb, window, vocab), RBR_EWORKSPACE,
                "rbr_datt_gate_fwd: workspace too small");
    cudaStream_t s = as_stream(stream);
    DattWs w = datt_ws(ws, n_docs, doc_len, emb, window, vocab);
    const int E = (int)emb, L = (int)doc_len, win = (int)window, Ep = (E + 3) & ~3;
    // declined before anything is enqueued: the caller's workspace and outputs stay untouched
    const size_t smem = ((size_t)((win * L + 3) & ~3) + (size_t)win * Ep + DA_WARPS) * 4;
    RBR_REQUIRE(smem <= 200 * 1024, RBR_EUNSUPPORTED, "rbr_datt_gate_fwd: doc_len too large for shared memory");
    datt_transpose_kernel<<<4, 256, 0, s>>>(w_local, E, Ep, win, w.waT);
    RBR_LAUNCH_CHECK("datt_transpose(local)");
    datt_transpose_kernel<<<(Ep * L + 255) / 256, 256, 0, s>>>(w_global, E, Ep, L, w.wgT);
    RBR_LAUNCH_CHECK("datt_transpose(global)");
    void (*kern)(const float*, int64_t, int, IdView, int, const float*, const float*, int, const float*, const float*, float*,
                 float*) = nullptr;
#define RBR_GF(W_) case W_: kern = (E % 4 == 0) ? datt_gate_fwd_kernel<true, W_> : datt_gate_fwd_kernel<false, W_>; break;
    switch (win) { RBR_GF(1) RBR_GF(3) RBR_GF(5) RBR_GF(7) }
#undef RBR_GF
    RBR_REQUIRE(kern != nullptr, RBR_EUNSUPPORTED, "rbr_datt_gate_fwd: window must be 1, 3, 5 or 7");
    RBR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(unsigned)n_docs, DA_WARPS * 32, smem, s>>>(table, vocab, E, ids, L, w.waT, b_local, win, w.wgT, b_global, gate_local,
                                                       gate_global);
    RBR_LAUNCH_CHECK("datt_gate_fwd_kernel");
    return RBR_OK;
}

extern "C" int rbr_datt_gate_bwd(const float* table, int64_t vocab, int64_t emb, const void* ids_raw, int64_t n_docs,
                                 int64_t doc_len, const float* w_local, int64_t window, const float* w_global,
                                 const float* gate_local, const float* gate_global, const float* gate_local_grad,
                                 const float* gate_global_grad, int64_t padding_idx, float* w_local_grad, float* b_local_grad,
                                 float* w_global_grad, float* b_global_grad, float* table_grad, void* ws, int64_t ws_bytes,
                                 int flags, void* stream) {
    int rc = datt_check(emb, doc_len, window, "rbr_datt_gate_bwd");
    if (rc != RBR_OK) return rc;
    if (n_docs == 0) return RBR_OK;
    const IdView ids = id_view(ids_raw, flags);
    RBR_REQUIRE(table && ids_raw && w_local && w_global && gate_local && gate_global && gate_local_grad && gate_global_grad &&
                    w_local_grad && b_local_grad && w_global_grad && b_global_grad && ws,
                RBR_EINVAL, "rbr_datt_gate_bwd: null pointer");
    RBR_REQUIRE(ws_bytes >= rbr_datt_gate_workspace_bytes(n_docs, doc_len, emb, window, vocab), RBR_EWORKSPACE,
                "rbr_datt_gate_bwd: workspace too small");
    RBR_REQUIRE(n_docs * doc_len < (1ll << 31), RBR_EUNSUPPORTED, "rbr_datt_gate_bwd: more than 2^31 tokens");
    cudaStream_t s = as_stream(stream);
    DattWs w = datt_ws(ws, n_docs, doc_len, emb, window, vocab);
    const int E = (int)emb, L = (int)doc_len, win = (int)window, Ep = (E + 3) & ~3;
    const bool v4 = E % 4 == 0;
    const int64_t ntok = n_docs * doc_len;
    datt_transpose_kernel<<<4, 256, 0, s>>>(w_local, E, Ep, win, w.waT);
    RBR_LAUNCH_CHECK("datt_transpose(local)");
    datt_transpose_kernel<<<(Ep * L + 255) / 256, 256, 0, s>>>(w_global, E, Ep, L, w.wgT);
    RBR_LAUNCH_CHECK("datt_transpose(global)");
    int blocks = (int)((ntok + 255) / 256);
    if (blocks > 148 * 8) blocks = 148 * 8;
    datt_gate_dz_kernel<<<blocks, 256, 0, s>>>(ids, n_docs, L, vocab, padding_idx, gate_local, gate_global, gate_local_grad,
                                               gate_global_grad, w.dz_l, w.dz_g, w.keys, b_local_grad, b_global_grad);
    RBR_LAUNCH_CHECK("datt_gate_dz_kernel");
#define RBR_DW(W_)                                                                                                            \
    case W_:                                                                                                                  \
        if (v4) datt_gate_wgrad_kernel<W_, true><<<(unsigned)L, DA_WARPS * 32, 0, s>>>(table, vocab, E, ids, n_docs, L, w.dz_l, \
                                                                                       w.dz_g, w_local_grad, w_global_grad);  \
        else datt_gate_wgrad_kernel<W_, false><<<(unsigned)L, DA_WARPS * 32, 0, s>>>(table, vocab, E, ids, n_docs, L, w.dz_l,  \
                                                                                     w.dz_g, w_local_grad, w_global_grad);    \
        break;
    switch (win) { RBR_DW(1) RBR_DW(3) RBR_DW(5) RBR_DW(7) }
#undef RBR_DW
    RBR_LAUNCH_CHECK("datt_gate_wgrad_kernel");
    if (table_grad) {
        TokenSort ts;
        rc = token_sort(w.keys, ntok, vocab, w.sort, ts, s);
        if (rc != RBR_OK) return rc;
        const int64_t warps = (ntok + 31) / 32;
        const int tb = (int)((warps * 32 + 255) / 256);
#define RBR_DT(W_)                                                                                                         \
    case W_:                                                                                                               \
        if (v4) datt_gate_table_kernel<W_, true><<<tb, 256, 0, s>>>(ts.order, w.keys, ntok, ts.start + vocab, L, E, w.dz_l, \
                                                                    w.dz_g, w.waT, w.wgT, table_grad);                     \
        else datt_gate_table_kernel<W_, false><<<tb, 256, 0, s>>>(ts.order, w.keys, ntok, ts.start + vocab, L, E, w.dz_l,   \
                                                                  w.dz_g, w.waT, w.wgT, table_grad);                       \
        break;
        switch (win) { RBR_DT(1) RBR_DT(3) RBR_DT(5) RBR_DT(7) }
#undef RBR_DT
        RBR_LAUNCH_CHECK("datt_gate_table_kernel");
    }
    return RBR_OK;
}

RBR_DEFINE_OOB_ACCESSOR(datt)
