// diverse.cu — K14: diversified top-k by maximal marginal relevance (MMR, Carbonell & Goldstein 1998), a greedy re-rank of
// each row's relevance pool (K10's top-P) over item-vector similarity.  sm_100a only.
//
// One CTA per row, one thread per pool position c (blockDim = P rounded up to a warp).  Thread c keeps its candidate's
// score, relevance rel(c), maxsim(c) and "picked" flag in registers.  Each round forms every candidate's objective, takes
// the block's largest 64-bit key (order-preserving objective bits << 32 | ~position: the larger objective, then the lower
// position, wins), writes the pick, and then each remaining candidate does ONE dot product, with the item just picked, to
// update its maxsim.  Work per row is k * P * dim FMAs; the k rounds of a row are serial, rows are independent.
//
// Item vectors: when the row's P vectors fit in shared memory (P * ld * 4 bytes, ld = dim padded to a multiple of 4 whose
// float4 count is odd, so eight consecutive threads' 16-byte reads hit distinct banks) they are staged once per row and
// every dot reads shared memory; otherwise each candidate reads its own row from global memory (L2-resident for catalogue
// sizes) and the picked vector is copied to shared memory each round.  Both read the same values in the same order:
//   sim(c, j) = fmaf(v_c[dim-1], v_j[dim-1], ... fmaf(v_c[1], v_j[1], fmaf(v_c[0], v_j[0], 0)))
// (the staged path's zero padding adds fmaf(0, 0, s) = s exactly: s is never -0), so results do not depend on the path, the
// batch, the row order or the chunking.  The objective is evaluated with explicitly rounded operations (no contraction):
//   obj(c) = lam * rel(c) - (1 - lam) * maxsim(c)          (lam and 1 - lam in fp32)
// and -0 is folded into +0 so that equal objectives tie on position.
#include <math.h>

#include "tc_ptx.cuh"

namespace rbr {

constexpr int MMR_MAX_POOL = 256;
constexpr int MMR_MAX_DIM = 512;

static bool mmr_supported(int64_t pool, int64_t dim, int64_t k) {
    return k >= 1 && k <= pool && pool <= MMR_MAX_POOL && dim >= 1 && dim <= MMR_MAX_DIM;
}

// shared-memory row stride of a staged vector: dim rounded up to a multiple of 4 floats with an odd number of float4s
static int mmr_ld(int64_t dim) {
    const int d4 = (int)round_up(dim, 4);
    return ((d4 / 4) & 1) ? d4 : d4 + 4;
}

struct MmrArgs {
    const float* pool_scores;     // [n_rows, pool]
    const int64_t* pool_items;    // [n_rows, pool]
    const float* vecs;            // [n_items, dim]
    float* out_scores;            // [n_rows, k]
    int64_t* out_items;
    int64_t n_items;
    int pool, dim, ld, k;
    float lam;
};

__device__ __forceinline__ unsigned long long warp_max_u64(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long w = __shfl_xor_sync(0xffffffffu, v, o);
        v = w > v ? w : v;
    }
    return v;
}

template <bool STAGED>
__global__ void __launch_bounds__(MMR_MAX_POOL) mmr_select_kernel(const MmrArgs a) {
    extern __shared__ __align__(16) float vs[];        // STAGED: the pool's vectors [pool][ld]; else the picked vector [dim]
    __shared__ unsigned long long red_key[2][MMR_MAX_POOL / 32];
    __shared__ float red_lo[MMR_MAX_POOL / 32], red_hi[MMR_MAX_POOL / 32];
    const int c = threadIdx.x, lane = c & 31, warp = c >> 5, nw = blockDim.x >> 5;
    const int P = a.pool, k = a.k, dim = a.dim;
    const int64_t row = blockIdx.x;
    const float* ps = a.pool_scores + row * P;
    const int64_t* pi = a.pool_items + row * P;

    float s = -INFINITY;
    int64_t item = -1;
    bool live = false;                                  // eligible and not yet picked
    if (c < P) {
        s = __ldg(ps + c);
        item = __ldg(pi + c);
        live = item >= 0 && item < a.n_items && isfinite(s);
    }
    if (STAGED) {
        for (int r = warp; r < P; r += nw) {
            const int64_t it = __ldg(pi + r);
            const bool in = it >= 0 && it < a.n_items;
            for (int d = lane; d < a.ld; d += 32)
                vs[r * a.ld + d] = (in && d < dim) ? __ldg(a.vecs + it * dim + d) : 0.f;
        }
    }
    // relevance: the row's eligible scores min-max scaled to [0, 1]
    float lo = warp_max(live ? -s : -INFINITY), hi = warp_max(live ? s : -INFINITY);
    if (lane == 0) { red_lo[warp] = lo; red_hi[warp] = hi; }
    __syncthreads();
    lo = -INFINITY; hi = -INFINITY;
    for (int w = 0; w < nw; ++w) { lo = fmaxf(lo, red_lo[w]); hi = fmaxf(hi, red_hi[w]); }
    lo = -lo;
    const float rel = !live ? 0.f : (hi == lo ? 1.f : __fdiv_rn(__fsub_rn(s, lo), __fsub_rn(hi, lo)));
    const float lam = a.lam, oml = __fsub_rn(1.f, a.lam);
    float maxsim = -INFINITY;

    for (int t = 0; t < k; ++t) {
        unsigned long long key = 0ull;
        if (live) {
            float obj = t == 0 ? rel : __fsub_rn(__fmul_rn(lam, rel), __fmul_rn(oml, maxsim));
            obj = obj == 0.f ? 0.f : obj;
            key = ((unsigned long long)f2ord(__float_as_uint(obj)) << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)c);
        }
        key = warp_max_u64(key);
        if (lane == 0) red_key[t & 1][warp] = key;
        __syncthreads();                                // also: every dot of round t-1 is done before vs is rewritten
        unsigned long long best = 0ull;
        for (int w = 0; w < nw; ++w) best = red_key[t & 1][w] > best ? red_key[t & 1][w] : best;
        if (best == 0ull) {                             // nothing eligible left: (-inf, -1) tail
            for (int j = t + c; j < k; j += blockDim.x) {
                a.out_scores[row * k + j] = -INFINITY;
                a.out_items[row * k + j] = -1;
            }
            return;
        }
        const int p = (int)(0xFFFFFFFFu - (uint32_t)best);
        if (c == p) {
            live = false;
            a.out_scores[row * k + t] = s;
            a.out_items[row * k + t] = item;
        }
        if (t == k - 1) break;
        const float* vp;
        if (STAGED) {
            vp = vs + p * a.ld;
        } else {
            const int64_t ip = __ldg(pi + p);
            for (int d = c; d < dim; d += blockDim.x) vs[d] = __ldg(a.vecs + ip * dim + d);
            __syncthreads();
            vp = vs;
        }
        if (live) {
            float acc = 0.f;
            if (STAGED) {
                const float4* x = reinterpret_cast<const float4*>(vs + c * a.ld);
                const float4* y = reinterpret_cast<const float4*>(vp);
#pragma unroll 4
                for (int q = 0; q < a.ld / 4; ++q) {
                    const float4 u = x[q], v = y[q];
                    acc = fmaf(u.x, v.x, acc);
                    acc = fmaf(u.y, v.y, acc);
                    acc = fmaf(u.z, v.z, acc);
                    acc = fmaf(u.w, v.w, acc);
                }
            } else {
                const float* x = a.vecs + item * dim;
#pragma unroll 4
                for (int d = 0; d < dim; ++d) acc = fmaf(__ldg(x + d), vp[d], acc);
            }
            maxsim = fmaxf(maxsim, acc);
        }
    }
}

static int mmr_smem_optin() {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess ||
        n <= 0) {
        cudaGetLastError();
        return 227 * 1024;                              // B200
    }
    return n;
}

}  // namespace rbr

using namespace rbr;

extern "C" int rbr_mmr_supported(int64_t pool, int64_t dim, int64_t k) { return mmr_supported(pool, dim, k) ? 1 : 0; }

extern "C" int rbr_mmr_select(const float* pool_scores, const int64_t* pool_items, int64_t n_rows, int64_t pool,
                              const float* item_vecs, int64_t n_items, int64_t dim, int64_t k, float lam, float* out_scores,
                              int64_t* out_items, void* stream) {
    RBR_REQUIRE(mmr_supported(pool, dim, k), RBR_EUNSUPPORTED,
                "rbr_mmr_select: need 1 <= k <= pool <= %d and 1 <= dim <= %d (got k=%lld pool=%lld dim=%lld)", MMR_MAX_POOL,
                MMR_MAX_DIM, (long long)k, (long long)pool, (long long)dim);
    RBR_REQUIRE(lam >= 0.f && lam <= 1.f, RBR_EINVAL, "rbr_mmr_select: lam must lie in [0, 1]");
    RBR_REQUIRE(n_rows >= 0 && n_rows < (1ll << 31) && n_items >= 0, RBR_EINVAL, "rbr_mmr_select: bad n_rows / n_items");
    if (n_rows == 0) return RBR_OK;
    RBR_REQUIRE(pool_scores && pool_items && item_vecs && out_scores && out_items, RBR_EINVAL, "rbr_mmr_select: null pointer");
    MmrArgs a;
    a.pool_scores = pool_scores; a.pool_items = pool_items; a.vecs = item_vecs; a.out_scores = out_scores;
    a.out_items = out_items; a.n_items = n_items; a.pool = (int)pool; a.dim = (int)dim; a.ld = mmr_ld(dim); a.k = (int)k;
    a.lam = lam;
    const int threads = (int)round_up(pool, 32);
    const int64_t staged_bytes = pool * a.ld * 4;
    cudaStream_t s = as_stream(stream);
    if (staged_bytes + 1024 <= mmr_smem_optin()) {              // + the static reduction slots
        RBR_CUDA(cudaFuncSetAttribute(mmr_select_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)staged_bytes));
        mmr_select_kernel<true><<<(unsigned)n_rows, threads, (size_t)staged_bytes, s>>>(a);
    } else {
        mmr_select_kernel<false><<<(unsigned)n_rows, threads, (size_t)dim * 4, s>>>(a);
    }
    RBR_LAUNCH_CHECK("mmr_select_kernel");
    return RBR_OK;
}
