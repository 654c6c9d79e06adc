// conv_tc2.cu — K2, CTA-pair tensor-core variant: gather → mask → Conv1d → bias → activation → max-over-time as an
// implicit GEMM on tcgen05 with cta_group::2 (two SMs, M = 256 positions per MMA), operands staged by TMA.  sm_100a only.
//
// Same contract and same maths as conv_tc.cu (reference models/deepconn/layers.py:22-24,123-136); what changes is how
// the operands reach the tensor cores, because conv_tc.cu is bound by shared-memory bandwidth, not by the MMA pipe:
//   * A operand (gathered token rows): TMA `cp.async.bulk.tensor.2d…tile::gather4` pulls 4 table rows x 64 bf16 columns
//     (4 x 128 B) per instruction straight from the bf16 shadow table into a K-major SWIZZLE_128B tile — one full
//     128-byte shared-memory line per row instead of eight scattered 16-byte cp.async granules.  Rows that must read as
//     zeros (conv padding, masked tokens, bad ids, tail tiles) use row index -1: the TMA unit zero-fills out-of-range
//     rows without touching memory.  The operand of tap j is still the SAME tile with the descriptor start advanced by
//     j rows (j * 128 B): the 128B swizzle is a function of absolute shared-memory address bits (tools/probe_umma.cu).
//   * B operand (conv weights, K-major no-swizzle core-matrix tiles, resident for the whole persistent kernel): each CTA
//     of the pair keeps only HALF of the filters (cta_group::2 reads N/2 rows of B from each SM), which halves the
//     per-SM operand read traffic of every MMA and frees ~100 KB for a 7-stage ring of 64-wide K blocks.
//   * D: each CTA owns the accumulator rows of its own 128-position tile (TMEM, double buffered); the epilogue (exact
//     fp32 max-over-time with first-arg-max via redux/ballot) is per CTA, unchanged from conv_tc.cu.
// Pipeline: per CTA four TMA producer warps, 16 epilogue warps; the LEADER CTA's MMA warp issues every tcgen05.mma for the
// pair.  full[s] lives in the leader (both CTAs' TMA bytes complete on it), empty[s] / acc_full[b] are multicast by
// tcgen05.commit to both CTAs, acc_empty[b] collects one arrive per epilogue warp of both CTAs.
#include <cuda.h>   // CUtensorMap (types only: the encoder is fetched through cudaGetDriverEntryPoint, no -lcuda)

#include "rbr_common.cuh"
#include "tc_ptx.cuh"

namespace rbr {

constexpr int T2_M = 128;                  // positions per CTA tile (UMMA M = 256 over the pair)
// Epilogue warps EW (template parameter of the kernel): 8 or 16 = 2 or 4 per TMEM lane quadrant, each reducing a share of
// the 16-column chunks.  The max-reduction is a chain of fixed-latency warp ops: 16 warps hide it when there is a lot of it
// per tile relative to the MMA/gather work (many filter chunks, short documents = per-tile finalisation, or a narrow
// embedding = few K blocks per tile), 8 leave more issue slots to the MMA warp.
// Warp roles: [0, EW) epilogue, [EW, EW+4) TMA producers (TMA issue is serialised per warp), EW+4 = TMEM owner + MMA issuer,
// EW+5 = index warp (resolves the table row of every staged tile row ahead of the producers).
// Producer warps: issuing one gather4 costs a warp ~100 cycles (the TMA unit accepts the instruction's uniform-register
// operands serially per warp), so the 32 + halo gather4s of a K block are spread over 4 warps; each stages 32 tile rows.
// 8 measured = 4: the floor is the TMA unit's row rate, not per-warp issue.
constexpr int T2_PROD_WARPS = 4;
constexpr int t2_threads(int ew) { return (ew + T2_PROD_WARPS + 2) * 32; }
constexpr int T2_IDX_BUFS = 3;               // index buffers at most (plan: nib = as many as fit without costing a ring stage, >= 1; the
                                             // producers copy a tile's indices to registers at the top of the tile, so one buffer already
                                             // lets the index warp finish tile g+1 while tile g streams — more only absorb jitter)
constexpr int T2_IDX_AHEAD = 2;              // unit steps ahead of the index warp's cursor whose id / mask rows are prefetched into L2
constexpr int T2_IDX_ROWS = 136;             // ints per index buffer (128 tile rows + 8 halo rows)
constexpr int T2_SMEM_MAX = 232448;          // 227 KB opt-in dynamic shared memory per CTA
// shared memory after the ring and the weights: bias, arg-max keys, nib index buffers (+ their 2 barriers each), barriers, TMEM slot
constexpr int t2_tail_bytes(int Nb, int nib) {
    return Nb * 4 + 8 + 2 * 4 * Nb * 8 + 16 + nib * (T2_IDX_ROWS * 4 + 16) + 8 * (2 * 16 + 9) + 16 + 16;
}
constexpr int T2_MIN_STAGES = 3;

struct Tc2Plan {
    int E, H, K, L, pad, Lout, Lext;
    int nkb;          // 64-element K blocks per staged row = emb_pad / 64
    int ksteps;       // UMMA K-steps (16 elements) = Epad16 / 16
    int C;            // 16-byte K chunks per weight row = Epad16 / 8
    int P, Nb, NL;    // filter passes, filters per pass (multiple of 16), filters per CTA = Nb / 2
    int rows;         // 128 + K - 1 staged rows carry data
    int groups;       // gather4 groups per stage = ceil(rows / 4)   (<= 64)
    int stage_bytes;  // groups * 512 rounded up to 1024 (stages stay swizzle-atom aligned)
    int stage_tx;     // bytes one CTA's TMA delivers per stage = groups * 512
    int nst;          // ring stages
    int w_bytes;      // resident weights per CTA = K * C * NL * 16
    int mode_b, D, tpu;
    int S;            // mode B: tile rows between consecutive documents = Lext rounded up to 32 (one document per epilogue warp row block)
    int64_t n_units;
    int tmem_cols, acc_stride;
    int nacc_log2;    // accumulator buffers in TMEM: 4 (filters per pass <= 128) or 2 — the MMA warp runs that many tiles ahead of the epilogue
    int nib;          // index buffers (1..T2_IDX_BUFS)
    int RS;           // row-index table: int32 entries per document row (tpu * 128 + 8, or S with several documents per tile)
    int off_ring, off_w, off_bias, off_keys, off_idx, off_bars, off_slot, smem_bytes;   // offsets from the 1024-aligned base
    int act;
    uint32_t boff[4 * 8];   // B-descriptor offset (16-byte units) of (K-step ks, tap j) inside a K block: [ks * 8 + j]
};

static inline int t2_stage_bytes(int K) {
    const int groups = (T2_M + K - 1 + 3) / 4;
    return (int)round_up(groups * 512, 1024);
}

// filters-per-pass decision shared with rbr_conv_pack (the packed B operand is laid out per pass and per CTA half)
void tc2_pass_split(int64_t E, int64_t H, int64_t K, int64_t* P, int64_t* Nb) {
    *P = 0; *Nb = 0;
    if (K < 1 || K > 8) return;
    const int64_t epad16 = round_up(E, 16);
    const int64_t bytes_per_row = K * epad16 * 2;                    // one local filter row of B
    // the most local filters (multiple of 8, UMMA N = 2 * nl <= 256) that leave room for T2_MIN_STAGES ring stages and the tail
    int64_t nl_max = 0;
    for (int64_t nl = 128; nl >= 8; nl -= 8)
        if (1024 + bytes_per_row * nl + T2_MIN_STAGES * t2_stage_bytes((int)K) + t2_tail_bytes((int)(2 * nl), 1) + 256 <= T2_SMEM_MAX) {
            nl_max = nl;
            break;
        }
    if (nl_max < 8) return;
    const int64_t npad = round_up(H, 16);
    *P = (npad + 2 * nl_max - 1) / (2 * nl_max);
    *Nb = round_up((H + *P - 1) / *P, 16);
}

struct Tc2Args {
    int64_t vocab;
    IdView ids;
    const uint8_t* mask;
    int64_t n_docs;
    const __nv_bfloat16* wpack;      // [P][2][K][C][NL][8]
    const float* bias;
    float* feat;
    int32_t* argmax;
    float* preact;
    const float* gate;
    int gate_mode;
    int feat_ld;
    // optional document selection (conv_doc_select_kernel): live[0] = number of documents with at least one unmasked token,
    // live[1 + i] = their indices.  The kernel then tiles only those; the all-padding documents (NARRE pads every user / item
    // to 10 reviews: ~45 % of the "documents" are empty) were given act(bias) / arg-max 0 by the selection pass.
    const int32_t* live;
    // optional (long documents): ntl[i] = number of 128-position tiles document live[1 + i] needs — the tiles that lie entirely
    // in its padding tail are skipped (conv_doc_tiles_* kernels; the list is sorted by tile count so that the two CTAs of a
    // pair, which advance in lockstep, get documents of equal length)
    const int32_t* ntl;
    // optional row-index table (conv_rowidx_kernel): rowidx[doc][e] = table row staged for extended position e of the document
    // (input position e - pad), or -1 = reads as zeros (outside the document, masked out, or an id outside the table); row n_docs
    // is all -1.  With it a tile's 136 row indices are ONE contiguous run (or one run per document slot), and the index warp
    // only issues bulk copies of them into the index buffers — no id / mask loads on the conv kernel's critical path.
    const int32_t* rowidx;
    Tc2Plan p;
};

// list slot li (unit * D + slot) → document index
__device__ __forceinline__ int64_t t2_doc_of(const int32_t* live, int64_t li) { return live ? (int64_t)__ldg(live + 1 + li) : li; }

template <int KT, int EW>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(t2_threads(EW), 1)
conv_tc2_kernel(const __grid_constant__ CUtensorMap tmap, const Tc2Args a) {
    constexpr int ROWS_PW = T2_M / T2_PROD_WARPS, G4_PW = ROWS_PW / 4;
    constexpr int T2_EPI_WARPS = EW, T2_EPI_SHARES = EW / 4;
    constexpr int MAXC = 1;   // TMEM chunks held in registers at once (2 or 4 with an earlier accumulator release measured slower: 0.34 / 0.38 vs 0.31 ms)
    constexpr int T2_PROD_WARP0 = EW, T2_MMA_WARP = EW + T2_PROD_WARPS, T2_IDX_WARP = T2_MMA_WARP + 1;
    extern __shared__ uint8_t smem_raw[];
    const Tc2Plan& p = a.p;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t sbase = (raw + 1023u) & ~1023u;                   // SWIZZLE_128B atoms are 1024-byte aligned
    uint8_t* smem = smem_raw + (sbase - raw);
    const uint32_t ring_s = sbase + p.off_ring, w_s = sbase + p.off_w;
    float* bias_s = reinterpret_cast<float*>(smem + p.off_bias);
    unsigned long long* keys_s = reinterpret_cast<unsigned long long*>(smem + p.off_keys);
    int* idx_s = reinterpret_cast<int*>(smem + p.off_idx);
    const uint32_t bars = sbase + p.off_bars;
    // barrier slots: full[nst] (used in the leader), empty[nst], acc_full[4], acc_empty[4] (used in the leader), w_ready,
    // idx_full[nib] (32 index-warp lanes arrive), idx_empty[nib] (one arrival per producer warp)
    const uint32_t bar_full = bars, bar_empty = bars + 8 * p.nst, bar_accf = bars + 16 * p.nst, bar_acce = bar_accf + 32,
                   bar_w = bar_acce + 32, bar_idxf = bar_w + 8, bar_idxe = bar_idxf + 8 * p.nib;
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + p.off_slot);

    const uint32_t rank = cluster_ctarank();
    const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
    const int pass = pair % p.P;
    const int ctas_per_pass = (n_pairs / p.P) * 2;
    const int ci = (pair / p.P) * 2 + (int)rank;                     // this CTA's index among the CTAs of its pass
    const int h0 = pass * p.Nb;
    // units this CTA owns: ci, ci + ctas_per_pass, ...; the pair runs as many tiles as its even CTA (never fewer than the odd one)
    const int ci_even = ci & ~1;
    const int64_t n_live = a.live ? (int64_t)__ldg(a.live) : a.n_docs;
    const int64_t n_units = p.mode_b ? (n_live + p.D - 1) / p.D : n_live;
    const int64_t pair_units = (n_units > ci_even) ? (n_units - ci_even + ctas_per_pass - 1) / ctas_per_pass : 0;
    // tiles of the pair's j-th unit step: fixed (tiles per unit), or — with a tile-count list — what the longer of the pair's
    // two documents needs (the shorter one then runs over padding rows, which changes neither its max nor its first arg-max)
    auto step_tiles = [&](int64_t j) -> int {
        if (!a.ntl) return p.tpu;
        const int64_t li0 = ci_even + j * ctas_per_pass;
        const int n0 = li0 < n_live ? __ldg(a.ntl + li0) : 0, n1 = li0 + 1 < n_live ? __ldg(a.ntl + li0 + 1) : 0;
        const int n = n0 > n1 ? n0 : n1;
        return n < 1 ? 1 : n;
    };
    int64_t pair_tiles = pair_units * p.tpu;
    if (a.ntl) {
        pair_tiles = 0;
        for (int64_t j = 0; j < pair_units; ++j) pair_tiles += step_tiles(j);
    }

    if (threadIdx.x == 0) {
        for (int i = 0; i < p.nst; ++i) { mbar_init(bar_full + 8 * i, 2); mbar_init(bar_empty + 8 * i, 1); }
        for (int i = 0; i < 4; ++i) { mbar_init(bar_accf + 8 * i, 1); mbar_init(bar_acce + 8 * i, 2 * T2_EPI_WARPS); }
        mbar_init(bar_w, 1);
        for (int i = 0; i < p.nib; ++i) { mbar_init(bar_idxf + 8 * i, a.rowidx ? 1 : 32); mbar_init(bar_idxe + 8 * i, T2_PROD_WARPS); }
        fence_barrier_init();
    }
    for (int i = threadIdx.x; i < p.Nb; i += blockDim.x) bias_s[i] = (h0 + i < p.H) ? a.bias[h0 + i] : 0.f;
    for (int i = threadIdx.x; i < 2 * 4 * p.Nb; i += blockDim.x) keys_s[i] = 0ull;
    if (warp == T2_MMA_WARP) tmem_alloc2(smem_u32((const void*)tmem_slot), (uint32_t)p.tmem_cols);
    if (warp == T2_PROD_WARP0 && lane == 0) tma_prefetch_desc(&tmap);
    tc_fence_before();
    cluster_sync_all();              // barriers of BOTH CTAs initialised before any remote arrive / multicast commit
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == T2_MMA_WARP) {
        // =========================== resident weights (each CTA its half) + MMA issuer (leader CTA only) ===========================
        if (pair_tiles > 0) {
            const bool leader_lane = elect_one();
            if (leader_lane) {
                mbar_expect_tx(bar_w, (uint32_t)p.w_bytes);
                const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(a.wpack) + (size_t)(pass * 2 + (int)rank) * p.w_bytes;
                for (int off = 0; off < p.w_bytes; off += 32768) {
                    const int n = min(32768, p.w_bytes - off);
                    bulk_g2s(w_s + off, wsrc + off, (uint32_t)n, bar_w);
                }
            }
            __syncwarp();
            if (rank == 0) {
                mbar_wait(bar_w, 0);
                const uint32_t idesc = umma_idesc(2 * T2_M, p.Nb);
                const uint64_t a_desc0 = umma_desc_sw128(ring_s);                          // stage 0, tap 0, K-step 0
                const uint64_t b_desc0 = umma_desc(w_s, (uint32_t)p.NL * 16u, 128u);       // tap 0, K-step 0
                const uint32_t a_stage_inc = (uint32_t)p.stage_bytes >> 4;                 // descriptor address units (16 B)
                const uint32_t b_step_inc = (uint32_t)(2 * p.NL);                          // one K-step = 2 chunk columns
                int stage = 0;
                uint32_t ph = 0;
                uint32_t full_bar = bar_full, empty_bar = bar_empty;
                uint64_t ad = a_desc0;
                for (int64_t g = 0; g < pair_tiles; ++g) {
                    const int buf = (int)(g & ((1 << p.nacc_log2) - 1));
                    mbar_wait(bar_acce + 8 * buf, (uint32_t)(((g >> p.nacc_log2) & 1) ^ 1));        // both CTAs' epilogues drained this buffer
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + (uint32_t)(buf * p.acc_stride);
                    uint64_t bd = b_desc0;
                    int ks_left = p.ksteps;
                    for (int kb = 0; kb < p.nkb; ++kb) {
                        mbar_wait(full_bar, ph);                                           // both CTAs' TMA bytes have landed
                        tc_fence_after();
                        if (leader_lane) {
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks) {
                                if (ks < ks_left) {
#pragma unroll
                                    for (int j = 0; j < KT; ++j)
                                        umma_bf16_2(d_tmem, ad + (uint64_t)(ks * 2 + j * 8), bd + (uint64_t)p.boff[ks * 8 + j], idesc,
                                                    (uint32_t)((kb | ks | j) != 0));
                                }
                            }
                            umma_commit2(empty_bar);                                       // frees the ring slot in both CTAs
                            if (kb == p.nkb - 1) umma_commit2(bar_accf + 8 * buf);         // accumulators complete → both epilogues
                        }
                        __syncwarp();
                        ks_left -= 4;
                        bd += (uint64_t)(4 * b_step_inc);
                        ad += a_stage_inc;
                        full_bar += 8;
                        empty_bar += 8;
                        if (++stage == p.nst) { stage = 0; ph ^= 1; ad = a_desc0; full_bar = bar_full; empty_bar = bar_empty; }
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp >= T2_PROD_WARP0 && warp < T2_MMA_WARP) {
        // =========================== TMA gather producers (4 warps per CTA) ===========================
        // Producer warp pw stages tile rows ROWS_PW·pw .. +ROWS_PW-1 (warp 0 also the k-1 halo rows 128..): it takes the tile's row
        // indices (table row, or -1 = reads as zeros) from the index warp's shared-memory buffer and ONE elected lane issues the
        // warp's gather4s of each K block as straight-line code with its operands in registers (TMA issue is serialised per warp,
        // hence four warps; a per-lane issue loop serialises on the TMA unit accepting each instruction's uniform registers).
        // Resolving the indices here (list -> document -> ids -> range checks, then 40 shuffles) was 30-36 % of a producer
        // warp's time, all four warps at once at the top of every tile with the TMA unit running dry: hence the index warp.
        const int pw = warp - T2_PROD_WARP0;
        const int halo_groups = p.groups - 32;                      // 0 (k == 1), 1 or 2
        int stage = 0, ib = 0;
        uint32_t ph = 0, iph = 0;
        bool w_checked = false;
        const uint32_t dst0 = ring_s + (uint32_t)(pw * G4_PW) * 512u;
        const uint32_t dst_halo = ring_s + 32u * 512u;
        for (int64_t g = 0; g < pair_tiles; ++g) {
            mbar_wait(bar_idxf + 8 * ib, iph);
            int idx[ROWS_PW], hidx[8];
            {
                const int4* src = reinterpret_cast<const int4*>(idx_s + ib * T2_IDX_ROWS + pw * ROWS_PW);
#pragma unroll
                for (int gi = 0; gi < G4_PW; ++gi) {
                    const int4 v = src[gi];
                    idx[4 * gi] = v.x; idx[4 * gi + 1] = v.y; idx[4 * gi + 2] = v.z; idx[4 * gi + 3] = v.w;
                }
                const int4* hsrc = reinterpret_cast<const int4*>(idx_s + ib * T2_IDX_ROWS + T2_M);
                const int4 h0v = hsrc[0], h1v = hsrc[1];
                hidx[0] = h0v.x; hidx[1] = h0v.y; hidx[2] = h0v.z; hidx[3] = h0v.w;
                hidx[4] = h1v.x; hidx[5] = h1v.y; hidx[6] = h1v.z; hidx[7] = h1v.w;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_idxe + 8 * ib);          // the buffer may be rewritten (tile g + nib)
            if (++ib == p.nib) { ib = 0; iph ^= 1; }
            for (int kb = 0; kb < p.nkb; ++kb) {
                mbar_wait(bar_empty + 8 * stage, ph ^ 1);
                const uint32_t fb = bar_full + 8 * stage;
                if (pw == 0 && lane == 0) {
                    if (rank == 0) {
                        mbar_expect_tx(fb, 2u * (uint32_t)p.stage_tx);        // this CTA's bytes + the peer's
                    } else {
                        if (!w_checked) { mbar_wait(bar_w, 0); w_checked = true; }   // the leader's MMAs also read OUR weights
                        mbar_arrive_cluster(fb, 0);
                    }
                }
                const uint32_t so = (uint32_t)(stage * p.stage_bytes);
                if (elect_one()) {
#pragma unroll
                    for (int gi = 0; gi < G4_PW; ++gi)
                        tma_gather4_pair(dst0 + so + (uint32_t)gi * 512u, &tmap, kb * 64, idx[4 * gi], idx[4 * gi + 1], idx[4 * gi + 2],
                                         idx[4 * gi + 3], fb);
                    if (pw == 0) {
                        if (halo_groups > 0) tma_gather4_pair(dst_halo + so, &tmap, kb * 64, hidx[0], hidx[1], hidx[2], hidx[3], fb);
                        if (halo_groups > 1) tma_gather4_pair(dst_halo + so + 512u, &tmap, kb * 64, hidx[4], hidx[5], hidx[6], hidx[7], fb);
                    }
                }
                __syncwarp();
                if (++stage == p.nst) { stage = 0; ph ^= 1; }
            }
        }
    } else if (warp == T2_IDX_WARP) {
        // =========================== index warp: table row (or -1) of every staged row, a few tiles ahead of the producers ===========
        // Lane l resolves tile rows l, 32 + l, 64 + l, 96 + l and halo row 128 + l (slots 0..4).  The resolution is pipelined over
        // THREE tiles, each step one iteration after the loads it depends on were issued, so no load is waited for where it is issued:
        //   stage A (tile g+2): schedule position -> list slot -> document index        (loads: live[], tile counts ntl[])
        //   stage B (tile g+1): document index -> token id and mask byte                (loads: ids, mask)
        //   stage C (tile g)  : id / mask byte -> table row or -1, written to the tile's index buffer
        // Everything loaded stays RAW in registers (either id width, the mask byte, the list entry, a unit step's two tile counts)
        // and is converted an iteration later.
        if (a.rowidx) {
            // ---- row-index table present: one elected lane copies each tile's indices (544 bytes) into the next index buffer ----
            // Lane l of the warp holds the documents and the tile count of unit step jb + l (one coalesced read of the lists per 32
            // unit steps); they reach the issuing code by shuffle, so no list load is waited for per tile.
            const uint32_t idx_sa = sbase + p.off_idx;
            const int nseg = p.mode_b ? (T2_IDX_ROWS + p.S - 1) / p.S : 1;
            int32_t docq[4] = {0, 0, 0, 0};
            int cnt = 1;
            int ib = 0;
            uint32_t iph = 0;
            for (int64_t uj = 0; uj < pair_units; ++uj) {
                if ((uj & 31) == 0) {
                    const int64_t j = uj + lane;
                    const int64_t unit = ci + j * ctas_per_pass;
                    const bool uok = j < pair_units && unit < n_units;
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int64_t li = p.mode_b ? unit * p.D + q : unit;
                        docq[q] = (uok && q < p.D && li < n_live) ? (int32_t)t2_doc_of(a.live, li) : (int32_t)a.n_docs;
                    }
                    cnt = j < pair_units ? step_tiles(j) : 1;
                }
                const int src = (int)(uj & 31);
                int32_t dq[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) dq[q] = __shfl_sync(0xffffffffu, docq[q], src);
                const int unt = __shfl_sync(0xffffffffu, cnt, src);
                for (int utt = 0; utt < unt; ++utt) {
                    if (lane == 0) {
                        mbar_wait(bar_idxe + 8 * ib, iph ^ 1);          // every producer warp has read this buffer's previous tile
                        const uint32_t fb = bar_idxf + 8 * ib, dst = idx_sa + (uint32_t)(ib * T2_IDX_ROWS * 4);
                        mbar_expect_tx(fb, (uint32_t)(T2_IDX_ROWS * 4));
                        if (!p.mode_b) {
                            bulk_g2s(dst, a.rowidx + (int64_t)dq[0] * p.RS + utt * T2_M, (uint32_t)(T2_IDX_ROWS * 4), fb);
                        } else {
                            for (int q = 0; q < nseg; ++q) {
                                const int n = min(p.S, T2_IDX_ROWS - q * p.S);
                                const int64_t d = q < 4 ? (q == 0 ? dq[0] : q == 1 ? dq[1] : q == 2 ? dq[2] : dq[3]) : a.n_docs;
                                bulk_g2s(dst + (uint32_t)(q * p.S * 4), a.rowidx + d * p.RS, (uint32_t)(n * 4), fb);
                            }
                        }
                    }
                    if (++ib == p.nib) { ib = 0; iph ^= 1; }
                }
            }
        } else {
        constexpr int NS = 5;
        const int halo_groups = p.groups - 32;
        int row[NS], qb[NS], extb[NS];
        bool rowok[NS];
#pragma unroll
        for (int i = 0; i < NS; ++i) {
            row[i] = i * 32 + lane;
            rowok[i] = i < 4 ? true : (lane < 4 * halo_groups && row[i] < p.rows);
            qb[i] = 0; extb[i] = 0;
            if (p.mode_b) {                                         // several documents per tile: slot and offset are tile-invariant
                qb[i] = row[i] / p.S;
                extb[i] = row[i] - qb[i] * p.S;
                rowok[i] = rowok[i] && qb[i] < p.D && extb[i] < p.Lext;
            }
        }
        // stage A state: schedule position (unit step, tile within it) and the step's raw tile counts
        int uj = 0, utt = 0;
        int32_t n0r = 0, n1r = 0;
        auto load_counts = [&](int j) {
            n0r = 0; n1r = 0;
            if (a.ntl && j < pair_units) {
                const int64_t li0 = ci_even + (int64_t)j * ctas_per_pass;
                if (li0 < n_live) n0r = __ldg(a.ntl + li0);
                if (li0 + 1 < n_live) n1r = __ldg(a.ntl + li0 + 1);
            }
        };
        // The ids / mask of a batch come from HBM (a batch is read once per step), and under this kernel's gather traffic a miss
        // takes several microseconds — longer than a tile.  So the id / mask rows of the unit T2_IDX_AHEAD unit steps ahead of
        // the stage-A cursor are pulled into L2 when the cursor enters a new unit (a whole document row: 128-byte lines spread
        // over the lanes), and stage B's loads are L2 hits.
        const int idsz = a.ids.u16 ? 2 : a.ids.i32 ? 4 : 8;
        auto prefetch_unit = [&](int j) {
            // (long documents only: with several documents per tile every tile is a new unit, and the list loads in here —
            // waited for on the spot — cost the index warp more than the misses they avoid: NARRE shape, 6 % -> 36 % producer wait)
            if (p.mode_b) return;
            const int64_t unit = ci + (int64_t)j * ctas_per_pass;
            if (j >= pair_units || unit >= n_units) return;
            for (int q = 0; q < p.D; ++q) {
                const int64_t li = p.mode_b ? unit * p.D + q : unit;
                if (li >= n_live) break;
                const int64_t doc = t2_doc_of(a.live, li);
                const char* ib0 = reinterpret_cast<const char*>(a.ids.p) + doc * p.L * idsz;
                const char* ie = ib0 + (int64_t)p.L * idsz;
                for (const char* c = reinterpret_cast<const char*>(reinterpret_cast<uintptr_t>(ib0) & ~(uintptr_t)127) + lane * 128; c < ie;
                     c += 32 * 128)
                    prefetch_l2(c);
                if (a.mask) {
                    const char* mb0 = reinterpret_cast<const char*>(a.mask) + doc * p.L;
                    const char* me = mb0 + p.L;
                    for (const char* c = reinterpret_cast<const char*>(reinterpret_cast<uintptr_t>(mb0) & ~(uintptr_t)127) + lane * 128; c < me;
                         c += 32 * 128)
                        prefetch_l2(c);
                }
            }
        };
        auto advance = [&]() {
            int unt = p.tpu;
            if (a.ntl) { unt = n0r > n1r ? n0r : n1r; unt = unt < 1 ? 1 : unt; }
            if (++utt >= unt) { ++uj; utt = 0; load_counts(uj); prefetch_unit(uj + T2_IDX_AHEAD); }
        };
        // A -> B
        int32_t docr[NS];                // document index: the raw list entry, or the slot itself without a list (n_docs < 2^31)
        int tB[NS];
        bool vB[NS];
        auto stage_a = [&]() {
            const int64_t unit = ci + (int64_t)uj * ctas_per_pass;
            const bool unit_ok = uj < pair_units && unit < n_units;
#pragma unroll
            for (int i = 0; i < NS; ++i) {
                const int64_t li = p.mode_b ? unit * p.D + qb[i] : unit;
                const int ext = p.mode_b ? extb[i] : utt * T2_M + row[i];
                const int t = ext - p.pad;
                vB[i] = unit_ok && rowok[i] && ext < p.Lext && li < n_live && t >= 0 && t < p.L;
                tB[i] = t;
                docr[i] = (int32_t)li;
                if (vB[i] && a.live) docr[i] = __ldg(a.live + 1 + li);
            }
        };
        // B -> C
        int2 rawid[NS];                  // int32 id in .x, or the two halves of an int64 id
        uint8_t rawm[NS];
        bool vC[NS];
#pragma unroll
        for (int i = 0; i < NS; ++i) { rawid[i] = make_int2(0, 0); rawm[i] = 0; vC[i] = false; }
        auto stage_b = [&]() {
#pragma unroll
            for (int i = 0; i < NS; ++i) {
                vC[i] = vB[i];
                if (!vB[i]) continue;
                const int64_t at = (int64_t)docr[i] * p.L + tB[i];
                if (a.ids.u16) rawid[i].x = (int)__ldg(reinterpret_cast<const uint16_t*>(a.ids.p) + at);
                else if (a.ids.i32) rawid[i].x = __ldg(reinterpret_cast<const int32_t*>(a.ids.p) + at);
                else rawid[i] = __ldg(reinterpret_cast<const int2*>(a.ids.p) + at);
                if (a.mask) rawm[i] = __ldg(a.mask + at);
            }
        };
        for (int j = 1; j <= T2_IDX_AHEAD; ++j) prefetch_unit(j);
        load_counts(0);
        stage_a();                          // tile 0
        stage_b();
        advance();
        stage_a();                          // tile 1
        int ib = 0;
        uint32_t iph = 0;
        for (int64_t g = 0; g < pair_tiles; ++g) {
            int mine[NS];
#pragma unroll
            for (int i = 0; i < NS; ++i) {
                mine[i] = -1;
                if (vC[i]) {
                    const int64_t id = (a.ids.i32 || a.ids.u16) ? (int64_t)rawid[i].x
                                                 : (int64_t)(((unsigned long long)(uint32_t)rawid[i].y << 32) | (uint32_t)rawid[i].x);
                    const bool ok = a.mask ? rawm[i] != 0 : (a.ids.mask_ids ? id != 0 : true);
                    if (ok) {
                        if (id >= 0 && id < a.vocab) mine[i] = (int)id;
                        else note_oob();
                    }
                }
            }
            stage_b();                      // tile g + 1
            advance();
            stage_a();                      // tile g + 2
            mbar_wait(bar_idxe + 8 * ib, iph ^ 1);                  // every producer warp has read this buffer's previous tile
            int* dst = idx_s + ib * T2_IDX_ROWS;
#pragma unroll
            for (int i = 0; i < 4; ++i) dst[row[i]] = mine[i];
            if (lane < 8) dst[T2_M + lane] = mine[4];
            mbar_arrive(bar_idxf + 8 * ib);                         // 32 arrivals (release): the tile's indices are visible
            if (++ib == p.nib) { ib = 0; iph ^= 1; }
        }
        }
    } else {
        // =========================== epilogue (16 warps; warp w reads TMEM lanes 32(w&3)..+31 and reduces 1/4 of the column chunks:
        // the reduction is a chain of fixed-latency warp ops, so it is latency- not issue-bound and more warps hide it) ===========================
        const int quad = warp & 3;
        const int share = warp >> 2;
        const int m = quad * 32 + lane;                       // tile row = TMEM lane
        const int n_chunks = p.Nb / 16;
        const int chunk_lo = n_chunks * share / T2_EPI_SHARES;
        const int chunk_hi = n_chunks * (share + 1) / T2_EPI_SHARES;
        int64_t uj = 0;
        int tt = -1, unt = pair_units > 0 ? step_tiles(0) : 0;
        // Finalisation (a unit's last tile) is local to a warp GROUP: the warps of one column share that hold the rows of one
        // document slot (all four quadrants with one document per tile, S / 32 of them with several).  Only they touch that
        // slot's keys in those columns, so they synchronise among themselves on a named barrier of their own (one warp: no
        // barrier) and write their share of the slot's outputs — the CTA-wide barrier made every warp wait for the slowest of
        // 8 or 16 on every tile of a short-document batch.  The slot's document index is fetched from the list at the TOP of
        // the unit's last tile: no dependent global load between the barrier and the stores.
        const int qps = p.mode_b ? p.S / 32 : 4;              // quadrants (warps of a share) per document slot
        const int grp_bar = 1 + share * (4 / qps) + quad / qps, grp_threads = qps * 32, grp_tid = (quad % qps) * 32 + lane;
        int32_t fin_doc = -1;
        for (int64_t g = 0; g < pair_tiles; ++g) {
            if (++tt >= unt) { ++uj; tt = 0; unt = step_tiles(uj); }
            const int64_t unit = ci + uj * ctas_per_pass;
            const int buf = (int)(g & ((1 << p.nacc_log2) - 1));
            // Pooled keys (value, ~position) live in shared memory per TMEM lane quadrant: entry [quad][column] is owned by exactly
            // one warp (quad = warp & 3, column chunk by share), so the running max over the tiles of a document is a plain
            // read-modify-write — no atomics (a 64-bit shared atomicMax is a CAS loop, and four quadrants contended for every
            // column).  Double buffered by unit parity: ONE (group) barrier per unit (the buffer is next written two units
            // later, i.e. after the following unit's barrier, which a thread of the group passes only once all of them have
            // finalised this unit).
            unsigned long long* keys_u = keys_s + (uj & 1) * (4 * p.Nb);
            // mode B packs documents on 32-row (warp) boundaries: a warp's rows all belong to one document slot
            const int slot = p.mode_b ? (quad * 32) / p.S : 0;
            const int t = p.mode_b ? m - slot * p.S : tt * T2_M + m;
            const int64_t my_li = p.mode_b ? unit * p.D + slot : unit;
            const bool valid = (t < p.Lout) && (slot < p.D) && (unit < n_units) && (my_li < n_live);
            if (tt == unt - 1) fin_doc = (slot < p.D && unit < n_units && my_li < n_live) ? (int32_t)t2_doc_of(a.live, my_li) : -1;
            float row_gate = 1.f;
            if (a.gate_mode == 1 && valid) row_gate = a.gate[t2_doc_of(a.live, my_li) * p.L + t];

            mbar_wait(bar_accf + 8 * buf, (uint32_t)((g >> p.nacc_log2) & 1));
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(buf * p.acc_stride);
            // Chunks are pulled out of TMEM MAXC at a time; the accumulator is handed back to the MMA warp as soon as the warp's
            // LAST chunk is in registers, i.e. before any reduction when all its chunks fit one group (8-warp mode, <= 4 chunks
            // per warp): the max-reduction then overlaps the MMAs of tile g+2 instead of delaying them.
            for (int chg = chunk_lo; chg < chunk_hi; chg += MAXC) {
                uint32_t v[MAXC][16];
#pragma unroll
                for (int u = 0; u < MAXC; ++u)
                    if (chg + u < chunk_hi) tmem_ld16(taddr + (uint32_t)((chg + u) * 16), v[u]);
                tmem_ld_wait();
                if (chg + MAXC >= chunk_hi) {                 // last group: release the accumulator
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_cluster(bar_acce + 8 * buf, 0);
                }
#pragma unroll
                for (int u = 0; u < MAXC; ++u) {
                    if (chg + u >= chunk_hi) continue;
                    const int c0 = (chg + u) * 16;
                    if (a.gate_mode == 1) {                   // per-token gate (k == 1): conv(g_t * x_t) = g_t * conv(x_t)
#pragma unroll
                        for (int i = 0; i < 16; ++i) v[u][i] = __float_as_uint(__uint_as_float(v[u][i]) * row_gate);
                    }
                    uint32_t keep_v = 0, keep_b = 0;
                    if (__all_sync(0xffffffffu, valid)) tc_colmax<true>(v[u], true, lane, keep_v, keep_b);
                    else tc_colmax<false>(v[u], valid, lane, keep_v, keep_b);
                    if (lane < 16 && keep_b) {
                        const int first = __ffs(keep_b) - 1;          // first (smallest-position) row attaining the max
                        const int tf = p.mode_b ? (quad * 32 + first - slot * p.S) : (tt * T2_M + quad * 32 + first);
                        const unsigned long long key =
                            ((unsigned long long)f2ord(keep_v) << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)tf);
                        unsigned long long* kp = keys_u + quad * p.Nb + c0 + lane;
                        if (key > *kp) *kp = key;
                    }
                }
            }
            if (chunk_lo == chunk_hi) {                       // fewer chunks than shares: a warp without a chunk still owes its arrive
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(bar_acce + 8 * buf, 0);
            }
            if (tt == unt - 1) {
                // (A/B on one box, DeepCoNN shape: the group barrier 4258 clk per tile, a CTA-wide one 4338)
                if (qps > 1) asm volatile("bar.sync %0, %1;" ::"r"(grp_bar), "r"(grp_threads) : "memory");
                else __syncwarp();
                const int q0 = (quad / qps) * qps;
                for (int c = chunk_lo * 16 + grp_tid; c < chunk_hi * 16; c += grp_threads) {
                    unsigned long long key = 0ull;
                    for (int q = q0; q < q0 + qps; ++q) {
                        const unsigned long long k2 = keys_u[q * p.Nb + c];
                        keys_u[q * p.Nb + c] = 0ull;
                        key = k2 > key ? k2 : key;
                    }
                    if (fin_doc >= 0 && h0 + c < p.H) {
                        const int64_t doc = fin_doc;
                        const float raw_v = __uint_as_float(ord2f((uint32_t)(key >> 32)));
                        const int tbest = (int)(0xFFFFFFFFu - (uint32_t)key);
                        const float gated = a.gate_mode == 2 ? raw_v * a.gate[doc] : raw_v;                 // per-doc gate > 0: monotone
                        a.feat[doc * a.feat_ld + h0 + c] = act_apply(p.act, gated + bias_s[c]);
                        if (a.preact) a.preact[doc * a.feat_ld + h0 + c] = gated;                           // pool_raw: no bias
                        a.argmax[doc * a.feat_ld + h0 + c] = tbest;
                    }
                }
            }
        }
    }
    // teardown: neither CTA may free TMEM / exit while the pair's MMAs can still touch its shared or tensor memory
    tc_fence_before();
    cluster_sync_all();
    if (warp == T2_MMA_WARP) tmem_dealloc2(tmem_base, (uint32_t)p.tmem_cols);
}

// Document selection: one warp per document.  A document none of whose tokens is unmasked reads as all zeros, so its conv
// output is the bias at every position: pooled value act(bias), first arg-max 0 — written here; the others are appended to
// the list the conv kernel tiles (live[0] = count, zeroed by the caller).
__global__ void __launch_bounds__(256) conv_doc_select_kernel(const IdView ids, const uint8_t* __restrict__ mask, int64_t n_docs, int L,
                                                              int32_t* __restrict__ live, const float* __restrict__ bias, int H, int act,
                                                              float* __restrict__ feat, int32_t* __restrict__ argmax,
                                                              float* __restrict__ pool_raw, int feat_ld,
                                                              int32_t* __restrict__ rowidx, int RS, int pad, int Lext, int64_t vocab) {
    __shared__ int s_any[8], s_base;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t d = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    bool any = false;
    if (rowidx) {
        // the pass sees every id / mask byte anyway: it also writes the document's row of the row-index table (see
        // conv_rowidx_kernel; the warp of "document" n_docs writes the all -1 row that stands in for absent documents)
        if (d <= n_docs) {
            for (int e = lane; e < RS; e += 32) {
                const int t = e - pad;
                int32_t v = -1;
                if (d < n_docs && e < Lext && t >= 0 && t < L) {
                    const int64_t at = d * L + t;
                    const int64_t id = ld_id(ids, at);
                    if (ld_mask(ids, mask, at, id)) {
                        any = true;
                        if (id >= 0 && id < vocab) v = (int32_t)id;
                        else note_oob();
                    }
                }
                rowidx[d * RS + e] = v;
            }
        }
    } else if (d < n_docs) {
        for (int t = lane; t < L && !any; t += 32) {
            const int64_t i = d * L + t;
            any = mask ? (__ldg(mask + i) != 0) : (ld_id(ids, i) != 0);
        }
    }
    any = __any_sync(0xffffffffu, any);
    // one list reservation per CTA (8 documents), not per document: the counter is a single address
    if (lane == 0) s_any[w] = any ? 1 : 0;
    __syncthreads();
    if (threadIdx.x == 0) {
        int n = 0;
        for (int i = 0; i < 8; ++i) n += s_any[i];
        s_base = n ? atomicAdd(live, n) : 0;
    }
    __syncthreads();
    if (d >= n_docs) return;
    if (any) {
        if (lane == 0) {
            int pos = s_base;
            for (int i = 0; i < w; ++i) pos += s_any[i];
            live[1 + pos] = (int32_t)d;
        }
    } else {
        for (int h = lane; h < H; h += 32) {
            feat[d * feat_ld + h] = act_apply(act, __ldg(bias + h));
            argmax[d * feat_ld + h] = 0;
            if (pool_raw) pool_raw[d * feat_ld + h] = 0.f;
        }
    }
}

// ---- long documents: tiles per document and a list sorted by tile count (descending) ------------------------------------
// Position t reads tokens t - pad .. t - pad + k - 1, so every position t >= len + pad (len = last unmasked token + 1) sees only
// zero rows: its conv output is the bias, the same value as at position len + pad.  Covering positions 0 .. len + pad therefore
// yields the same max and the same FIRST arg-max as covering all of them: tiles beyond ceil(min(Lout, len + pad + 1) / 128) are
// skipped.  (Tried on top of this and rejected: not staging the 32-row blocks / gather4 groups past a document's end inside its
// last tile, with the epilogue ignoring those positions.  12-25 % fewer gather4s, but no faster: a producer warp's stage time is
// its own 8-10 serial gather4 issues of ~100 cycles each, so dropping whole warps' groups shortens nothing, and any per-gather4
// predicate or branch makes the compiler rebuild the uniform-register operands in front of every one — 25-35 % slower.)  ws layout (int32): [0] count, [16..80) bucket counts,
// [80..144) bucket cursors, [256 ..) list, then tiles-per-entry, then tiles-per-document.
constexpr int T2_WS_HDR = 256;
__global__ void __launch_bounds__(256) conv_doc_tiles_count_kernel(const IdView ids, const uint8_t* __restrict__ mask, int64_t n_docs, int L,
                                                                   int Lout, int pad, int32_t* __restrict__ ws) {
    const int lane = threadIdx.x & 31;
    const int64_t d = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (d >= n_docs) return;
    int len = 0;
    for (int t0 = ((L - 1) / 32) * 32; t0 >= 0 && len == 0; t0 -= 32) {
        const int t = t0 + lane;
        bool on = false;
        if (t < L) {
            const int64_t i = d * L + t;
            on = mask ? (__ldg(mask + i) != 0) : (ld_id(ids, i) != 0);
        }
        const unsigned b = __ballot_sync(0xffffffffu, on);
        if (b) len = t0 + (32 - __clz(b));
    }
    const int covered = min(Lout, len + pad + 1);          // positions 0 .. len + pad (the first one over zero rows only)
    const int nt = max(1, (covered + T2_M - 1) / T2_M);
    if (lane == 0) {
        ws[T2_WS_HDR + 2 * n_docs + d] = nt;
        atomicAdd(ws + 16 + min(nt, 63), 1);
    }
}
// bucket offsets (longest documents first) are recomputed by every CTA from the 64 counters — cheaper than a scan launch; the
// cursors [80..144) count within a bucket.  Thread 0 of CTA 0 also publishes the list's entry count where the conv kernel
// reads it (just below the list).
__global__ void __launch_bounds__(256) conv_doc_tiles_fill_kernel(int32_t* __restrict__ ws, int64_t n_docs) {
    __shared__ int s_off[64];
    if (threadIdx.x < 64) {
        int off = 0;
        for (int b = 63; b > (int)threadIdx.x; --b) off += ws[16 + b];
        s_off[threadIdx.x] = off;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) { ws[0] = (int32_t)n_docs; ws[T2_WS_HDR - 1] = (int32_t)n_docs; }
    __syncthreads();
    const int64_t d = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= n_docs) return;
    const int nt = ws[T2_WS_HDR + 2 * n_docs + d];
    const int bkt = min(nt, 63);
    const int pos = s_off[bkt] + atomicAdd(ws + 80 + bkt, 1);
    ws[T2_WS_HDR + pos] = (int32_t)d;
    ws[T2_WS_HDR + n_docs + pos] = nt;
}

int64_t conv_tc2_select_bytes(int64_t n_docs) { return round_up((T2_WS_HDR + 3 * n_docs) * 4, 256); }

// ---- row-index table: the table row (or -1) of every extended position of every document ------------------------------------
// One thread per entry, coalesced over a document row; a CTA walks documents blockIdx.x, blockIdx.x + gridDim.x, ...
// Row n_docs (all -1) stands in for absent documents.  With `tiles_ws` the pass also does conv_doc_tiles_count_kernel's job
// (it sees every mask byte anyway): the document's tile count and its bucket counter.
__global__ void __launch_bounds__(256) conv_rowidx_kernel(const IdView ids, const uint8_t* __restrict__ mask, int64_t n_docs, int L, int pad,
                                                          int Lext, int RS, int64_t vocab, int32_t* __restrict__ rowidx, int Lout,
                                                          int32_t* __restrict__ tiles_ws) {
    __shared__ int s_len;
    for (int64_t d = blockIdx.x; d <= n_docs; d += gridDim.x) {
        if (tiles_ws) {
            __syncthreads();
            if (threadIdx.x == 0) s_len = 0;
            __syncthreads();
        }
        int len = 0;
        for (int e = threadIdx.x; e < RS; e += 256) {
            const int t = e - pad;
            int32_t v = -1;
            if (d < n_docs && e < Lext && t >= 0 && t < L) {
                const int64_t at = d * L + t;
                const int64_t id = ld_id(ids, at);
                if (ld_mask(ids, mask, at, id)) {
                    len = t + 1;
                    if (id >= 0 && id < vocab) v = (int32_t)id;
                    else note_oob();
                }
            }
            rowidx[d * RS + e] = v;
        }
        if (tiles_ws && d < n_docs) {
            len = __reduce_max_sync(0xffffffffu, len);
            if ((threadIdx.x & 31) == 0 && len > 0) atomicMax(&s_len, len);
            __syncthreads();
            if (threadIdx.x == 0) {
                const int covered = min(Lout, s_len + pad + 1);
                const int nt = max(1, (covered + T2_M - 1) / T2_M);
                tiles_ws[T2_WS_HDR + 2 * n_docs + d] = nt;
                atomicAdd(tiles_ws + 16 + min(nt, 63), 1);
            }
        }
    }
}
// the same for short rows (RS = 32 or 64, a multiple of 32): one thread per entry over the flat table
__global__ void __launch_bounds__(256) conv_rowidx_short_kernel(const IdView ids, const uint8_t* __restrict__ mask, int64_t n_docs, int L,
                                                                int pad, int Lext, int RS, int64_t vocab, int32_t* __restrict__ rowidx) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (n_docs + 1) * RS) return;
    const int64_t d = i / RS;
    const int e = (int)(i - d * RS), t = e - pad;
    int32_t v = -1;
    if (d < n_docs && e < Lext && t >= 0 && t < L) {
        const int64_t at = d * L + t;
        const int64_t id = ld_id(ids, at);
        if (ld_mask(ids, mask, at, id)) {
            if (id >= 0 && id < vocab) v = (int32_t)id;
            else note_oob();
        }
    }
    rowidx[i] = v;
}
static int tc2_rowidx_stride(int K, int L, int pad) {
    const int Lext = L + 2 * pad, Lout = Lext - K + 1, S = (int)round_up(Lext, 32);
    if (Lout < 1) return 0;
    if (S + Lext <= T2_M + K - 1) return S;                          // several documents per tile (as tc2_make_plan decides)
    return (Lout + T2_M - 1) / T2_M * T2_M + 8;
}
int64_t conv_tc2_workspace_bytes(int64_t n_docs, int64_t L, int64_t K, int64_t pad) {
    int64_t b = conv_tc2_select_bytes(n_docs);
    if (K >= 1 && K <= 8 && L >= 1 && L < (1 << 24) && pad >= 0 && pad < 64) b += (n_docs + 1) * tc2_rowidx_stride((int)K, (int)L, (int)pad) * 4;
    return b;
}

static bool tc2_make_plan(int E, int H, int K, int L, int pad, int act, int64_t n_docs, Tc2Plan* out) {
    Tc2Plan p{};
    p.E = E; p.H = H; p.K = K; p.L = L; p.pad = pad; p.act = act;
    p.Lout = L + 2 * pad - K + 1;
    p.Lext = L + 2 * pad;
    if (p.Lout < 1) return false;
    const int epad16 = (int)round_up(E, 16);
    p.C = epad16 / 8;
    p.ksteps = epad16 / 16;
    p.nkb = (int)(rbr_emb_pad(E) / 64);
    int64_t P, Nb;
    tc2_pass_split(E, H, K, &P, &Nb);
    if (P == 0) return false;
    p.P = (int)P; p.Nb = (int)Nb; p.NL = p.Nb / 2;
    p.rows = T2_M + K - 1;
    p.groups = (p.rows + 3) / 4;
    p.stage_tx = p.groups * 512;
    p.stage_bytes = t2_stage_bytes(K);
    p.w_bytes = K * p.C * p.NL * 16;
    // short documents: several per tile, each starting on a 32-row (epilogue-warp) boundary
    p.S = (int)round_up(p.Lext, 32);
    if (p.S + p.Lext <= T2_M + K - 1) {
        p.mode_b = 1;
        p.D = (T2_M + K - 1 - p.Lext) / p.S + 1;
        if (p.D > 4) p.D = 4;
        p.tpu = 1;
        p.n_units = (n_docs + p.D - 1) / p.D;
    } else {
        p.mode_b = 0;
        p.D = 1;
        p.tpu = (p.Lout + T2_M - 1) / T2_M;
        p.n_units = n_docs;
    }
    for (int ks = 0; ks < 4; ++ks)
        for (int j = 0; j < 8; ++j) p.boff[ks * 8 + j] = (uint32_t)(ks * 2 * p.NL + j * p.C * p.NL);   // K-step = 2 chunk columns, tap = C
    p.acc_stride = p.Nb <= 128 ? 128 : 256;
    p.nacc_log2 = p.acc_stride == 128 ? 2 : 1;
    p.tmem_cols = 512;
    p.RS = tc2_rowidx_stride(K, L, pad);
    auto stages_with = [&](int nib) {
        const int n = (T2_SMEM_MAX - 1024 - p.w_bytes - t2_tail_bytes(p.Nb, nib) - 256) / p.stage_bytes;
        return n > 16 ? 16 : n;
    };
    const int nst = stages_with(1);
    if (nst < T2_MIN_STAGES) return false;
    p.nst = nst;
    p.nib = 1;
    while (p.nib < T2_IDX_BUFS && stages_with(p.nib + 1) == nst) ++p.nib;
    const int idx_bytes = p.nib * T2_IDX_ROWS * 4;
    int off = 0;
    p.off_ring = off; off += nst * p.stage_bytes;
    p.off_w = off; off += p.w_bytes;
    off = (off + 15) / 16 * 16;
    p.off_bias = off; off += p.Nb * 4;
    off = (off + 7) / 8 * 8;
    p.off_keys = off; off += 2 * 4 * p.Nb * 8;
    off = (off + 15) / 16 * 16;
    p.off_idx = off; off += idx_bytes;
    p.off_bars = off; off += 8 * (2 * nst + 9 + 2 * p.nib);
    p.off_slot = off; off += 16;
    p.smem_bytes = off + 1024;                   // slack for the manual 1024-byte alignment of the base
    if (p.smem_bytes > T2_SMEM_MAX) return false;
    *out = p;
    return true;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn tc2_encoder() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(f);
        else
            (void)cudaGetLastError();
    }
    return fn;
}

template <int KT, int EW>
static int tc2_launch(const CUtensorMap& tm, const Tc2Args& a, cudaStream_t s) {
    static int max_clusters = -1;
    constexpr int T2_THREADS = t2_threads(EW);
    auto kern = conv_tc2_kernel<KT, EW>;
    if (max_clusters < 0) {
        RBR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, T2_SMEM_MAX));
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(2); cfg.blockDim = dim3(T2_THREADS); cfg.dynamicSmemBytes = T2_SMEM_MAX;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        int n = 0;
        if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess || n < 1) {
            (void)cudaGetLastError();
            int dev = 0, sms = 0;
            RBR_CUDA(cudaGetDevice(&dev));
            RBR_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
            n = sms / 2;
        }
        max_clusters = n;
    }
    // persistent grid: one CTA pair per co-resident cluster slot (a multiple of the pass count), never more pairs than work
    int64_t pairs = max_clusters / a.p.P * a.p.P;
    if (pairs < a.p.P) pairs = a.p.P;
    const int64_t max_useful = (a.p.n_units + 1) / 2 * a.p.P;
    if (pairs > max_useful) pairs = max_useful;
    kern<<<(unsigned)(2 * pairs), T2_THREADS, a.p.smem_bytes, s>>>(tm, a);
    RBR_LAUNCH_CHECK("conv_tc2_kernel");
    return RBR_OK;
}

// returns RBR_EUNSUPPORTED (without setting an error message the caller must surface) when the shape is outside this variant
int conv_tc2_dispatch(const __nv_bfloat16* shadow, int64_t vocab, int E, IdView ids, const uint8_t* mask,
                      const float* gate, int gate_mode, int64_t n_docs, int L, const __nv_bfloat16* umma_w2, const float* bias,
                      int H, int K, int pad, int act, float* feat, int32_t* argmax, float* preact, int feat_ld, void* ws,
                      int64_t ws_bytes, cudaStream_t s) {
    Tc2Args a{};
    if (vocab >= (1ll << 31) || n_docs >= (1ll << 31) || !tc2_make_plan(E, H, K, L, pad, act, n_docs, &a.p)) return RBR_EUNSUPPORTED;
    if (K != 1 && K != 2 && K != 3 && K != 4 && K != 5 && K != 7) return RBR_EUNSUPPORTED;
    EncodeTiledFn enc = tc2_encoder();
    if (!enc) return RBR_EUNSUPPORTED;
    const int64_t emb_pad = rbr_emb_pad(E);
    CUtensorMap tm;
    cuuint64_t gdim[2] = {(cuuint64_t)emb_pad, (cuuint64_t)vocab};
    cuuint64_t gstr[1] = {(cuuint64_t)emb_pad * 2};
    cuuint32_t box[2] = {64, 1};
    cuuint32_t estr[2] = {1, 1};
    const CUresult r = enc(&tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<__nv_bfloat16*>(shadow), gdim, gstr, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    RBR_REQUIRE(r == CUDA_SUCCESS, RBR_ECUDA, "conv_fwd[bf16]: cuTensorMapEncodeTiled failed (%d)", (int)r);
    // all-padding documents are cheap to find and need no tensor-core work (short documents only: NARRE's padded review slots)
    a.live = nullptr;
    a.ntl = nullptr;
    a.rowidx = nullptr;
    // Row-index table (written by the pre-pass that reads the ids / masks anyway: the tile-count pass for long documents, the
    // document selection for short ones; a pass of its own otherwise).
    const bool want_ri = ws && ws_bytes >= conv_tc2_workspace_bytes(n_docs, L, K, pad) &&
                         ws_bytes > conv_tc2_select_bytes(n_docs) && (reinterpret_cast<uintptr_t>(ws) & 15) == 0;
    int32_t* ri = want_ri ? reinterpret_cast<int32_t*>(reinterpret_cast<char*>(ws) + conv_tc2_select_bytes(n_docs)) : nullptr;
    if (ws && ws_bytes >= conv_tc2_select_bytes(n_docs) && (mask || ids.mask_ids) && gate_mode == 0 && n_docs >= 64 &&
        n_docs < (1ll << 30)) {
        int32_t* w32 = reinterpret_cast<int32_t*>(ws);
        if (a.p.mode_b) {
            // short documents: drop the all-padding ones.  The list (count at [T2_WS_HDR - 1]) is read as live[0], live[1 + i]
            int32_t* live = w32 + T2_WS_HDR - 1;
            RBR_CUDA(cudaMemsetAsync(live, 0, 4, s));
            // (with the row-index table: one more warp, for the table's all -1 row)
            conv_doc_select_kernel<<<(unsigned)(((n_docs + (want_ri ? 1 : 0)) * 32 + 255) / 256), 256, 0, s>>>(
                ids, mask, n_docs, L, live, bias, H, act, feat, argmax, preact, feat_ld, want_ri ? ri : nullptr, a.p.RS, pad, a.p.Lext, vocab);
            RBR_LAUNCH_CHECK("conv_doc_select_kernel");
            a.live = live;
            if (want_ri) a.rowidx = ri;
        } else if (a.p.tpu > 1) {
            // long documents: skip the tiles that lie entirely in a document's padding tail
            RBR_CUDA(cudaMemsetAsync(w32, 0, T2_WS_HDR * 4, s));
            if (want_ri) {                                   // the row-index pass counts the tiles as it goes
                conv_rowidx_kernel<<<(unsigned)(n_docs + 1 < 148 * 64 ? n_docs + 1 : 148 * 64), 256, 0, s>>>(
                    ids, mask, n_docs, L, pad, a.p.Lext, a.p.RS, vocab, ri, a.p.Lout, w32);
                RBR_LAUNCH_CHECK("conv_rowidx_kernel");
                a.rowidx = ri;
            } else {
                conv_doc_tiles_count_kernel<<<(unsigned)((n_docs * 32 + 255) / 256), 256, 0, s>>>(ids, mask, n_docs, L, a.p.Lout, a.p.pad, w32);
                RBR_LAUNCH_CHECK("conv_doc_tiles_count_kernel");
            }
            conv_doc_tiles_fill_kernel<<<(unsigned)((n_docs + 255) / 256), 256, 0, s>>>(w32, n_docs);
            RBR_LAUNCH_CHECK("conv_doc_tiles_fill_kernel");
            // (live[0] must be the count and live[1 + i] the list: the fill kernel writes the count just below the list)
            a.live = w32 + T2_WS_HDR - 1;
            a.ntl = w32 + T2_WS_HDR + n_docs;
        }
    }
    if (want_ri && !a.rowidx) {
        // short rows (several documents per tile): a thread block of 256 would idle on a 32- or 64-entry row — flat indexing instead
        if (a.p.RS < 128) {
            conv_rowidx_short_kernel<<<(unsigned)(((n_docs + 1) * a.p.RS + 255) / 256), 256, 0, s>>>(ids, mask, n_docs, L, pad, a.p.Lext,
                                                                                                   a.p.RS, vocab, ri);
            RBR_LAUNCH_CHECK("conv_rowidx_short_kernel");
        } else {
            conv_rowidx_kernel<<<(unsigned)(n_docs + 1 < 148 * 64 ? n_docs + 1 : 148 * 64), 256, 0, s>>>(
                ids, mask, n_docs, L, pad, a.p.Lext, a.p.RS, vocab, ri, a.p.Lout, nullptr);
            RBR_LAUNCH_CHECK("conv_rowidx_kernel");
        }
        a.rowidx = ri;
    }
    a.vocab = vocab; a.ids = ids; a.mask = mask; a.n_docs = n_docs; a.wpack = umma_w2; a.bias = bias;
    a.feat = feat; a.argmax = argmax; a.preact = preact; a.gate = gate; a.gate_mode = gate_mode; a.feat_ld = feat_ld;
    const bool wide = a.p.mode_b || a.p.Nb / 16 >= 9 || a.p.nkb <= 2;
    // (Tried and rejected: the column max as a transposed shuffle butterfly (24 shfl.bfly per 16 columns, value + first row carried
    // along) instead of redux.sync + ballot: DeepCoNN conv 299 -> 361 us, NARRE 313 -> 380 us — the redux form is the cheap one.)
    // (Tried and rejected: 20 epilogue warps = five column shares, so that Nb = 160 = 10 chunks splits 2,2,2,2,2 instead of 3,2,3,2 and
    // the per-document finalisation waits less for the slowest warp.  NARRE conv 305 -> 340 us: the extra warps take issue slots
    // from the producer warps, and gather issue is what bounds the kernel.)
#define RBR_T2(KT_) return wide ? tc2_launch<KT_, 16>(tm, a, s) : tc2_launch<KT_, 8>(tm, a, s)
    switch (K) {
        case 1: RBR_T2(1);
        case 2: RBR_T2(2);
        case 3: RBR_T2(3);
        case 4: RBR_T2(4);
        case 5: RBR_T2(5);
        default: RBR_T2(7);
    }
#undef RBR_T2
}

}  // namespace rbr

// Host-side plan of the CTA-pair kernel for a shape, without launching anything (tests of the tiling logic run on CPU).
// out[0..15] = {available, P, Nb, NL, nkb, ksteps, groups, stage_bytes, nst, w_bytes, mode_b, D, S, tpu, smem_bytes, tmem_cols}
extern "C" int rbr_conv_tc2_plan(int64_t emb, int64_t filters, int64_t ksize, int64_t doc_len, int64_t pad, int64_t n_docs,
                                 int64_t* out) {
    RBR_REQUIRE(out, RBR_EINVAL, "rbr_conv_tc2_plan: null pointer");
    rbr::Tc2Plan p{};
    const bool ok = emb > 0 && filters > 0 && ksize > 0 && doc_len > 0 && pad >= 0 &&
                    rbr::tc2_make_plan((int)emb, (int)filters, (int)ksize, (int)doc_len, (int)pad, 0, n_docs, &p);
    const int64_t v[16] = {ok ? 1 : 0, p.P, p.Nb, p.NL, p.nkb, p.ksteps, p.groups, p.stage_bytes, p.nst, p.w_bytes, p.mode_b, p.D, p.S,
                           p.tpu, p.smem_bytes, p.tmem_cols};
    for (int i = 0; i < 16; ++i) out[i] = v[i];
    return RBR_OK;
}

RBR_DEFINE_OOB_ACCESSOR(conv_tc2)
