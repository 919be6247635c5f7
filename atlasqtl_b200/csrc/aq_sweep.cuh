// The CAVI Gauss-Seidel sweep kernel (sm_100a): coreDualLoop (reference src/coreLoop.cpp:38-86) in
// sample space, blocked over SNPs, one persistent CTA per trait tile.
//
// Roles inside a CTA of 16 warps (warp-specialised, no __syncthreads in the steady state).  The fp64 tensor op
// (DMMA) and scalar fp64 math share one pipe per SM sub-partition (SMSP = warp id % 4); the serial chain is
// latency bound and runs ~2-3x slower behind a saturated DMMA stream (ncu: stall_math on the chain warp,
// profiles/r1_ncu_sweep_c4_v1_chain_shares_dmma_pipe.txt).  So SMSPs 0-2 carry four MMA warps each (pipe
// saturated), and SMSP 3 carries the chain, the helper and only TWO MMA warps (pipe half loaded):
//   14 "MMA" warps  hold the tile's residual R^T (traits x samples) in REGISTERS as the accumulator
//                   fragments of the rank-8 update  R^T -= Delta^T X_b^T  (DMMA m8n8k4), and reuse the very
//                   same registers as the A operand of  S^T = R^T X_b  -- the accumulator layout
//                   C[m][2l+e] is an A fragment A[m][l] once the contraction index is read as 2l+e, so the
//                   residual never moves: it is loaded once per tile and stored once per tile.
//                   One lane of the last MMA warp also streams the pre-tiled X blocks (+ Gram band + SNP
//                   ids) into a 3-stage shared-memory ring with 1-D bulk copies (TMA engine) on mbarriers.
//   1 "chain" warp  one lane per trait: resolves the in-block Gauss-Seidel order exactly from the Gram
//                   band (S[u] -= G[t][u] Delta[t]), evaluates mu / gam (annealed logistic) / beta and emits
//                   -Delta.  It is the only serial dependency of the sweep (block b+1 needs Delta_b), so it
//                   touches shared memory only; everything else of a block is done around it by the
//   1 "helper" warp which sums the split-K partials of S, stages the block's beta_old and c (D + cst) in shared memory
//                   (p x q rows fetched by cp.async one block ahead), writes gam / mu back and keeps the per-trait
//                   running sums.
//
// One-block look-ahead hides the serial chain behind the tensor pipe: S'_{b+1} = X_{b+1}' R_{b-1} is formed
// while the chain of block b runs, and corrected by the cross Gram block, S_{b+1} = S'_{b+1} - G_{b+1,b} Delta_b;
// the correction is accumulated inside the chain of block b (independent FMAs that fill its latency bubbles).
#pragma once
#include "aq_common.cuh"
#include "aq_mis.cuh"
#ifdef AQ_TIMING
// development only: per-section cycle sums of the chain (0-3) and helper (4-9) warps of CTA 0, kept in registers and
// written once at the end (a global read-modify-write per probe would put an L2 round trip into every section)
#define AQ_T(i) do { long long t_ = clock64(); tacc[i] += t_ - tlast; tlast = t_; } while (0)
#define AQ_T0() long long tlast = clock64()
#else
#define AQ_T(i) do { } while (0)
#define AQ_T0() do { } while (0)
#endif

namespace aq {

struct SweepParams {
    const int* order;       // [nb * 8] sweep position -> SNP index (-1 for padding slots); same ids as in the tile images
    const double* xtiles;   // nb * ncta tile images, tile_stride doubles apart: image (b, r) at (b * ncta + r)
    size_t tile_stride;
    int nb;                 // number of SNP blocks = p_pad / 8
    int ntiles;             // trait tiles of this launch
    int k_base;             // first trait of this launch: tile i covers traits [k_base + i kT, k_base + (i + 1) kT)
    int q;                  // valid traits
    int q_pad;              // leading dimension of the p x q arrays (trait-contiguous)
    int ld_resid;           // leading dimension of resid (samples per trait row) = ncta * kNPad
    int ncta;               // CTAs per cluster = sample slices (1 for the single-CTA kernel)
    double* resid;          // [q_pad][ld_resid]
    double* gam;            // [p_pad][q_pad]
    double* mu;             // [p_pad][q_pad]
    const double* dtab;     // [p_pad][q_pad]  log(1-Phi) - log(Phi)
    const double* wtab;     // [p_pad][q_pad]  imr1 - imr0
    const double* i0tab;    // [p_pad][q_pad]  imr0
    const double* tau;      // [q_pad]
    const double* log_tau;  // [q_pad]
    const double* sig2_beta;  // [q_pad]
    double c;
    double log_sig2_inv;
    double* cs_gam;         // [q_pad] outputs
    double* cs_gmu2;
    double* cs_b2;
    double* rsq;
    double* cs_z;
    double* rowpart;        // [rowpart_base + tile][p_pad] this tile's part of rowsum_j = sum_k gam W + I0 (NULL: not wanted)
    int rowpart_base;       // first row of this launch in rowpart
    int p_pad;
    int mode;               // 0: sweep;  1: build residual (R -= X beta) + sums from the loaded state
    // Segmented sweep (nseg > 1; single-CTA configurations, cooperative launch): the SNP blocks of every tile are cut into
    // nseg segments of seg_len blocks and the work units (segment s, tile) are dealt round-robin, segment-major, to the
    // persistent CTAs, so a partly filled last round costs 1 / nseg of a round instead of a whole one.  Unit (s, tile)
    // needs (s - 1, tile), which another CTA finished at an EARLIER position of its own list; the hand-off goes through
    // the residual / column sums in global memory and seg_done[tile] (release / acquire at gpu scope).
    int nseg;
    int seg_len;
    int* seg_done;          // [ntiles] segments completed per tile, zeroed before the launch (NULL iff nseg == 1)
    // Missing-response variant (SweepCfg<..., MIS = true>; coreDualMisLoop, src/coreLoop.cpp:91-138): every trait has its own
    // Gram matrix X' diag(mis_k) X.  The residual tile is kept MASKED (zero in the missing rows of its trait), so
    // S = X_b' R needs no mask; the in-block / look-ahead Gram entries come from a per-trait band precomputed once per
    // order (gk), and sig2_beta_vb(j, k) = 1 / (c (X_norm_sq(j, k) + sig2_inv) tau_k) enters through two p x q tables.
    const unsigned long long* mbits;  // [q_pad][mwords] bit i of row k: sample i of trait k is observed
    int mwords;
    const double* xnsq;     // [p_pad][q_pad] X_norm_sq = crossprod(X^2, mis_pat) (R/atlasqtl_global_local_core.R:23)
    const double* atab;     // [p_pad][q_pad] a = c sig2_beta tau = 1 / (X_norm_sq + sig2_inv)          (src/coreLoop.cpp:125)
    const double* ltab;     // [p_pad][q_pad] log sig2_beta_vb(j, k)                                     (:129)
    const double* gk;       // [tile][nb][128][16] per-trait Gram band, entry t * 16 + u as in the tile image's band
    double* mis_out;        // [kMisOutputs][q_pad] per-trait sums of the missing-response path
    long long* timing;      // development only (-DAQ_TIMING): per-section cycle sums of the chain warp
};

constexpr int kMaxCluster = 8;

template <int MT_, int NT_, bool CL_ = false, bool MIS_ = false>
struct SweepCfg {
    static constexpr bool kMis = MIS_;  // missing-response variant
    static constexpr int WS = 14;   // MMA warps, all along samples (split-K of the S GEMM)
    static constexpr int MT = MT_;  // 8-trait M tiles per MMA warp
    static constexpr int NT = NT_;  // 8-sample N tiles per MMA warp
    static constexpr bool kCl = CL_;  // sample-split thread-block cluster variant (n > 1008)
    static constexpr int kMmaWarps = WS;
    static constexpr int kT = MT * 8;                // traits per tile
    static constexpr int kNPad = WS * NT * 8;        // samples per CTA, padded
    static constexpr int kXS = kNPad + ((kNPad % 16 == 0) ? 8 : 0);  // tile row stride == 8 (mod 16) doubles
    static constexpr int kThreads = 16 * 32;  // warps 3 (chain) and 7 (helper) + 14 MMA warps (two of them on SMSP 3)
    static constexpr int kStages = 3;
    // the chain's logistic with two dependent operations less (aq_common.cuh): wins where the serial chain bounds a block
    // (clusters, missing responses, 24- / 32-trait tiles of small n), loses on the tensor-bound 16-trait tiles
    static constexpr bool kShortLogistic = CL_ || MIS_ || MT_ != 2;
    static constexpr size_t kTileDoubles = (size_t)kBlk * kXS + kTileTail;
    // S tiles in shared memory ([trait][8 SNP slots], partials and sums alike): row stride 8 doubles, the four 16-byte
    // pairs of a row XOR-swizzled by (trait >> 1) & 3 (sp_off), so that both the C-fragment stores of the MMA warps (lanes
    // = 2 traits x 4 pairs per quarter-warp) and the row reads of the chain / helper (lanes = 8 consecutive traits, same
    // pair) hit 8 different 16-byte bank groups.  (ncu on the unswizzled stride-10 layout: 2-way conflicts on every
    // partial store, 15 % of the kernel's shared-memory wavefronts.)
    static constexpr int kSps = 8;
    // who sums the split-K partials of S: the chain warp itself (single CTA: one hop less between the tensor work and the
    // recurrence), or the helper warp (clusters: the wait for the other CTAs' slices stays off the serial path)
    static constexpr bool kChainSums = MT > 1;
    // cluster leader: the helper warp sums the other CTAs' S tiles while the chain warp sums this CTA's own partials
    // (n = 5000, 8 CTAs: chain does both 24.99 ms, in parallel 23.74 ms; helper does both, as in round 1: 28.4 ms)
    static constexpr bool kHelperSumsFollowers = kCl && kChainSums;
    static constexpr int kIoPer = kMis ? 4 : 2;        // iobuf entries per (SNP slot, trait)
    static constexpr int kStgArrays = kMis ? 8 : 5;    // p x q arrays staged per block
    static constexpr uint32_t kDeltaBytes = (uint32_t)(kT * kBlk * sizeof(double));  // one -Delta block (or S tile)

    // ---- shared-memory layout: offset and size (doubles) of every region, each starting where the previous one ends (size 0
    // where a configuration has no use for it), then the barrier block.  The kernel carves its pointers from these.
    // [kStages] X tile images: the ring the producer lane fills with bulk copies
    static constexpr size_t kOffTiles = 0, kTilesDoubles = kStages * kTileDoubles;
    // [WS][kT][kSps] split-K partials of S, single-buffered (sfree barrier)
    static constexpr size_t kOffSpart = kOffTiles + kTilesDoubles, kSpartDoubles = (size_t)WS * kT * kSps;
    // [2][kT][kSps] S tile handed from the helper to the chain: the whole sum (8-trait tiles) or the followers' part of it
    static constexpr size_t kOffSsum = kOffSpart + kSpartDoubles,
                            kSsumDoubles = (kChainSums && !kHelperSumsFollowers) ? 0 : (size_t)2 * kT * kSps;
    // [2][kT x kBlk] -Delta (d_off layout)
    static constexpr size_t kOffDbuf = kOffSsum + kSsumDoubles, kDbufDoubles = (size_t)2 * kT * kBlk;
    // [WS][kT] squared norms of the residual, per MMA warp
    static constexpr size_t kOffRsqs = kOffDbuf + kDbufDoubles, kRsqsDoubles = (size_t)WS * kT;
    // [2][kBlk][kIoPer][kT]: in beta_old, c (D + cst) (+ a, bq per pair with missing responses); out gam, mu
    static constexpr size_t kOffIo = kOffRsqs + kRsqsDoubles, kIoDoubles = (size_t)2 * kBlk * kIoPer * kT;
    // [kStgArrays][kBlk][kT]: gam, mu, D, W, I0 (+ X_norm_sq, a, log sig2_beta) rows of the next block
    static constexpr size_t kOffStg = kOffIo + kIoDoubles, kStgDoubles = (size_t)kStgArrays * kBlk * kT;
    // cluster leader: [2][kMaxCluster - 1][kT][kSps] the followers' reduced S tiles
    static constexpr size_t kOffRed = kOffStg + kStgDoubles, kRedDoubles = kCl ? (size_t)2 * (kMaxCluster - 1) * kT * kSps : 0;
    // cluster leader: [kMaxCluster - 1][kT] the followers' squared-norm partials
    static constexpr size_t kOffRsqAll = kOffRed + kRedDoubles, kRsqAllDoubles = kCl ? (size_t)(kMaxCluster - 1) * kT : 0;
    // missing responses: [2][128][kT] per-trait Gram band of a block
    static constexpr size_t kOffGk = kOffRsqAll + kRsqAllDoubles, kGkDoubles = kMis ? (size_t)2 * 128 * kT : 0;
    static constexpr size_t kOffBars = kOffGk + kGkDoubles;
    // barrier block: slot of the first barrier of each family
    static constexpr int kBarFull = 0;                      // [kStages] tile landed (tx bytes)
    static constexpr int kBarEmpty = kBarFull + kStages;    // [kStages] MMA warps released the tile
    static constexpr int kBarDready = kBarEmpty + kStages;  // [2] chain warp published -Delta (in every CTA of the cluster)
    static constexpr int kBarDcons = kBarDready + 2;        // [2] mode 1 only, leader: all MMA warps consumed -Delta buffer
    static constexpr int kBarSred = kBarDcons + 2;          // [2] leader: followers delivered their reduced S tiles
    static constexpr int kBarRsq = kBarSred + 2;            // [1] leader: followers delivered their squared-norm partials
    static constexpr int kBarInready = kBarRsq + 1;         // [2] helper warp staged S and the block's inputs for the chain
    static constexpr int kBarSfree = kBarInready + 2;       // [1] helper / reducer warp has read the S partials of a block
    // [2][4] this CTA's MMA warps wrote their S partials, one barrier per SM sub-partition (the four warps of SMSP 0, 1, 2,
    // the two of SMSP 3): whoever sums the partials takes them group by group as they complete instead of after the last
    static constexpr int kBarSdone = kBarSfree + 1;
    static constexpr int kNumBars = kBarSdone + 8;
    static constexpr int kBarSlots = 24;
    static constexpr size_t kSmemBytes = kOffBars * sizeof(double) + kBarSlots * sizeof(uint64_t);
    static_assert(kNumBars <= kBarSlots, "barrier block");
    static_assert(kT <= 32, "one chain lane per trait");
    static_assert(!kMis || kT == 16, "the missing-response variant uses 16-trait tiles (its Gram band table is laid out for them)");
    static_assert(kXS % 16 == 8, "row stride must be 8 mod 16 doubles");
    static_assert(kSmemBytes <= 232448, "shared memory budget (227 KB)");
};

// offset (doubles) of SNP slot t (even: the pair t, t + 1) of trait row r in an S tile
__device__ __forceinline__ int sp_off(int r, int t) { return r * 8 + ((((t >> 1) ^ (r >> 1)) & 3) << 1) + (t & 1); }
// offset (doubles) of (trait r, SNP slot t) in a -Delta block of kT traits: pair-major [t >> 1][trait][2] with bit 3
// flipped in odd pair planes: the chain's 16-byte stores (lanes = consecutive traits) and the MMA warps' 8-byte loads
// (lane (g, l) reads trait g, slot l and l + 4) are both bank-conflict free (the trait-major [trait][8] layout gave 4-way
// conflicts on both)
template <int kT>
__device__ __forceinline__ int d_off(int r, int t) { return (t >> 1) * 2 * kT + ((2 * r + (t & 1)) ^ (((t >> 1) & 1) << 3)); }

// Sums of N values per lane over a group of G consecutive lanes (G = 4 N), by recursive halving: at every step a lane
// hands half of its values to its partner and keeps the other half.  On return v[0] of lane L is the group total of value
// slot_of(L) = the N-ary digit string of L's upper lane bits (see the caller); fixed order, deterministic.
template <int N>
__device__ __forceinline__ void group_sums(double (&v)[N], int lane, int top_bit) {
    if constexpr (N > 1) {
        const bool up = (lane & top_bit) != 0;
        double w[N / 2];
#pragma unroll
        for (int i = 0; i < N / 2; ++i) {
            const double send = up ? v[i] : v[i + N / 2];
            const double keep = up ? v[i + N / 2] : v[i];
            w[i] = keep + __shfl_xor_sync(0xffffffffu, send, top_bit);
        }
        group_sums<N / 2>(w, lane, top_bit >> 1);
        v[0] = w[0];
    } else {
        v[0] += __shfl_xor_sync(0xffffffffu, v[0], 2);
        v[0] += __shfl_xor_sync(0xffffffffu, v[0], 1);
    }
}

// This CTA's part of S = X_b' R of one block: sums the WS split-K partials of its MMA warps, SM sub-partition by
// sub-partition as their barriers complete.  Lane layout: trait `tsum`, and with <= 16 traits per tile the two half-warps
// split the partials of a trait between them (the caller adds the halves).  Frees the partial buffer when done.
template <class Cfg>
__device__ __forceinline__ void sum_own_partials(double (&s)[kBlk], const double* spart, uint64_t* sdone, uint64_t* sfree,
                                                 long gb, int lane, int tsum) {
    constexpr int WS = Cfg::WS, kT = Cfg::kT;
    static_assert(WS == 14, "MMA warp i sits on SMSP i % 3 for i < 12, warps 12 and 13 on SMSP 3");
    constexpr int kH = (kT <= 16) ? 2 : 1;
    const int half = (kH == 2) ? (lane >> 4) : 0;
    const uint32_t par = (uint32_t)((gb >> 1) & 1);
#pragma unroll
    for (int t = 0; t < kBlk; ++t) s[t] = 0.0;
    auto add = [&](int w) {
#pragma unroll
        for (int t = 0; t < kBlk; t += 2) {
            const double2 v = *reinterpret_cast<const double2*>(spart + w * kT * Cfg::kSps + sp_off(tsum, t));
            s[t] += v.x;
            s[t + 1] += v.y;
        }
    };
    // group order: SMSP 3 first (its two MMA warps share the pipe with nobody and deliver early), then SMSP 0, 1, 2.  Fixed
    // order whatever the arrival times: deterministic.
    mbar_wait(&sdone[(gb & 1) * 4 + 3], par);
    if (kH == 2) add(12 + half);
    else { add(12); add(13); }
#pragma unroll
    for (int g4 = 0; g4 < 3; ++g4) {
        mbar_wait(&sdone[(gb & 1) * 4 + g4], par);
        if (kH == 2) { add(g4 + 6 * half); add(g4 + 6 * half + 3); }
        else { add(g4); add(g4 + 3); add(g4 + 6); add(g4 + 9); }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&sfree[0]);  // the MMA warps may overwrite the partials
}

// Cluster leader: waits until the other CTAs' reduced S tiles of block gb have landed here (st.async, accounted on sred).
template <class Cfg>
__device__ __forceinline__ void wait_follower_tiles(uint64_t* sred, long gb, int ncta, int lane) {
    if (lane == 0) mbar_arrive_expect_tx(&sred[gb & 1], (uint32_t)(ncta - 1) * Cfg::kDeltaBytes);
    mbar_wait(&sred[gb & 1], (uint32_t)((gb >> 1) & 1));
}

// Cluster leader: adds the S tiles of CTA ranks [r0, r1) to the row of trait `tsum`, in rank order.
template <class Cfg>
__device__ __forceinline__ void add_follower_tiles(double (&s)[kBlk], const double* red, long gb, int tsum, int r0, int r1) {
    for (int r2 = r0; r2 < r1; ++r2) {
        const double* rp = red + (size_t)((gb & 1) * (kMaxCluster - 1) + (r2 - 1)) * Cfg::kT * Cfg::kSps;
#pragma unroll
        for (int t = 0; t < kBlk; t += 2) {
            const double2 v = *reinterpret_cast<const double2*>(rp + sp_off(tsum, t));
            s[t] += v.x;
            s[t + 1] += v.y;
        }
    }
}

// Cluster leader: the sum of the S tiles the other CTAs shipped here.  Lane = trait; with <= 16 traits per tile the two
// half-warps split the CTAs and the halves are added at the end.
template <class Cfg>
__device__ __forceinline__ void sum_follower_tiles(double (&s)[kBlk], const double* red, uint64_t* sred, long gb, int ncta,
                                                   int lane, int tsum) {
    constexpr int kH = (Cfg::kT <= 16) ? 2 : 1;
    const int half = (kH == 2) ? (lane >> 4) : 0;
#pragma unroll
    for (int t = 0; t < kBlk; ++t) s[t] = 0.0;
    wait_follower_tiles<Cfg>(sred, gb, ncta, lane);
    const int mid = (kH == 2) ? (ncta + 1) / 2 : ncta;
    add_follower_tiles<Cfg>(s, red, gb, tsum, half == 0 ? 1 : mid, half == 0 ? mid : ncta);
    if (kH == 2) {
#pragma unroll
        for (int t = 0; t < kBlk; ++t) s[t] += __shfl_xor_sync(0xffffffffu, s[t], 16);
    }
}

// S = X_b' R of one block: this CTA's partials and, on a cluster leader, the tiles the other CTAs shipped.
// On return every lane holds the complete S row of its trait.  Called by the chain warp (single CTA) or the helper warp.
template <class Cfg>
__device__ __forceinline__ void sum_s_partials(double (&s)[kBlk], const double* spart, const double* red, uint64_t* sdone,
                                               uint64_t* sfree, uint64_t* sred, long gb, int ncta, int lane, int tsum) {
    constexpr int kT = Cfg::kT;
    constexpr int kH = (kT <= 16) ? 2 : 1;
    const int half = (kH == 2) ? (lane >> 4) : 0;
    sum_own_partials<Cfg>(s, spart, sdone, sfree, gb, lane, tsum);
    if (Cfg::kCl && ncta > 1) {  // + the other sample slices, already reduced (and stored here) by their CTAs
        wait_follower_tiles<Cfg>(sred, gb, ncta, lane);
        if (half == 0) add_follower_tiles<Cfg>(s, red, gb, tsum, 1, ncta);
    }
    if (kH == 2) {
#pragma unroll
        for (int t = 0; t < kBlk; ++t) s[t] += __shfl_xor_sync(0xffffffffu, s[t], 16);
    }
}

// One work unit of a persistent CTA (cluster): SNP blocks [b0, b1) of trait tile `tile` (= all blocks when nseg == 1).
struct Unit {
    int tile, seg, b0, b1;
};
__device__ __forceinline__ Unit unit_of(const SweepParams& P, int group, int ngroups, int ju) {
    const int u = group + ju * ngroups;   // segment-major: (seg, tile) needs (seg - 1, tile) = unit u - ntiles < u
    Unit w;
    w.seg = u / P.ntiles;
    w.tile = u - w.seg * P.ntiles;
    w.b0 = w.seg * P.seg_len;
    w.b1 = min(P.nb, w.b0 + P.seg_len);
    return w;
}
// wait (one lane polls, acquire at gpu scope) until the previous segment of the unit's tile has been handed off
__device__ __forceinline__ void unit_acquire(const SweepParams& P, const Unit& w, int lane) {
    if (w.seg > 0) {
        if (lane == 0) {
            uint32_t spins = 0;
            // (a hand-off normally takes microseconds; 2^23 polls are ~1 s.  If the CTAs of the launch are NOT all resident
            // -- seen under `ncu --set full` with segmented cluster launches -- this traps instead of spinning for minutes)
            while (ld_acquire_gpu(P.seg_done + w.tile) < w.seg) {
                __nanosleep(64);
                if (++spins == (1u << 23)) __trap();
            }
        }
        __syncwarp();
    }
}
// end of a unit (segmented launches only): every warp of the CTA (of every CTA of the cluster) has finished its global
// writes of the unit -> publish.  Executed by ALL warps of all CTAs, whatever their role.
template <class Cfg>
__device__ __forceinline__ void unit_release(const SweepParams& P, const Unit& w) {
    if (P.nseg > 1) {
        __syncwarp();
        if constexpr (Cfg::kCl) cluster_sync_all();
        else asm volatile("bar.sync 2, %0;" ::"n"(Cfg::kThreads) : "memory");
        bool leader = threadIdx.x == 0;
        if constexpr (Cfg::kCl) leader = leader && cluster_ctarank() == 0;
        if (leader) {
            __threadfence();
            st_release_gpu(P.seg_done + w.tile, w.seg + 1);
        }
    }
}

template <class Cfg>
__global__ void __launch_bounds__(Cfg::kThreads, 1) sweep_kernel(const SweepParams P) {
    constexpr int WS = Cfg::WS, MT = Cfg::MT, NT = Cfg::NT, kT = Cfg::kT, XS = Cfg::kXS;
    constexpr int kStages = Cfg::kStages;
    constexpr bool kCl = Cfg::kCl;
    constexpr bool kMis = Cfg::kMis;
    constexpr int kIoPer = Cfg::kIoPer;
    // regions and barriers as SweepCfg lays them out
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double* const smem = reinterpret_cast<double*>(smem_raw);
    double* tiles = smem + Cfg::kOffTiles;
    double* spart = smem + Cfg::kOffSpart;
    double* ssum = smem + Cfg::kOffSsum;
    double* dbuf = smem + Cfg::kOffDbuf;
    double* rsqs = smem + Cfg::kOffRsqs;
    double* iobuf = smem + Cfg::kOffIo;
    double* stg = smem + Cfg::kOffStg;
    double* red = smem + Cfg::kOffRed;
    double* rsq_all = smem + Cfg::kOffRsqAll;
    double* gkbuf = smem + Cfg::kOffGk;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kOffBars);
    uint64_t* full = bars + Cfg::kBarFull;
    uint64_t* empty = bars + Cfg::kBarEmpty;
    uint64_t* dready = bars + Cfg::kBarDready;
    uint64_t* dcons = bars + Cfg::kBarDcons;
    uint64_t* sred = bars + Cfg::kBarSred;
    uint64_t* rsqbar = bars + Cfg::kBarRsq;
    uint64_t* inready = bars + Cfg::kBarInready;
    uint64_t* sfree = bars + Cfg::kBarSfree;
    uint64_t* sdone = bars + Cfg::kBarSdone;

    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
#ifdef AQ_TIMING
    long long tacc[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
#endif
    // role map: SMSPs 0-2 (wid % 4 != 3) host four MMA warps each; SMSP 3 hosts the chain (wid 3), the helper (wid 7)
    // and MMA warps 12, 13 (wid 11, 15)
    const int smsp = wid & 3, quad = wid >> 2;
    const bool is_mma = smsp != 3 || quad >= 2;
    const int mma_idx = smsp != 3 ? quad * 3 + smsp : 12 + (quad - 2);   // 0..13 for MMA warps
    const bool is_chain = smsp == 3 && quad == 0;                          // followers: S reducer
    const bool is_helper = smsp == 3 && quad == 1;
    const bool is_producer = mma_idx == Cfg::kMmaWarps - 1 && is_mma;      // also streams the X tiles
    const int ncta = kCl ? P.ncta : 1;
    const int rank = kCl ? (int)cluster_ctarank() : 0;
    const int group = kCl ? (int)cluster_id_x() : (int)blockIdx.x;         // unit-loop index of this CTA (cluster)
    const int ngroups = kCl ? (int)cluster_count_x() : (int)gridDim.x;
    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], Cfg::kMmaWarps); }
        for (int s = 0; s < 2; ++s) {
            for (int g4 = 0; g4 < 4; ++g4) mbar_init(&sdone[s * 4 + g4], g4 < 3 ? 4 : Cfg::kMmaWarps - 12);
            mbar_init(&dready[s], 1);
            mbar_init(&dcons[s], Cfg::kMmaWarps * ncta);
            mbar_init(&sred[s], 1);
            mbar_init(&inready[s], 1);
        }
        mbar_init(&rsqbar[0], ncta > 1 ? ncta - 1 : 1);
        mbar_init(&sfree[0], 1);
        fence_mbar_init();
    }
    __syncthreads();
    if (kCl) cluster_sync_all();  // every CTA's barriers are initialised before any remote arrive

    const int nunits = P.ntiles * P.nseg;
    const int my_units = (nunits - group + ngroups - 1) / ngroups;
    const uint32_t tile_bytes = (uint32_t)(Cfg::kTileDoubles * sizeof(double));

    if (is_mma) {
        // ------------------------------------------------------------------ MMA warps
        const int ws = mma_idx;
        const int mtid = mma_idx * 32 + lane;
        // producer duty (one lane): the X tiles of this CTA's units, in order, into the ring; (pj, pb) is its cursor
        long total = 0;   // blocks this CTA sweeps
        int pj = 0, pb = 0, pb1 = 0;
        if (is_producer) {
            for (int ju = 0; ju < my_units; ++ju) {
                const Unit w = unit_of(P, group, ngroups, ju);
                total += w.b1 - w.b0;
            }
            if (my_units > 0) {
                const Unit w = unit_of(P, group, ngroups, 0);
                pb = w.b0;
                pb1 = w.b1;
            }
        }
        auto load_next = [&](long it) {
            const int stage = (int)(it % kStages);
            mbar_arrive_expect_tx(&full[stage], tile_bytes);
            bulk_g2s(tiles + stage * Cfg::kTileDoubles, P.xtiles + ((size_t)pb * ncta + rank) * P.tile_stride, tile_bytes, &full[stage]);
            if (++pb == pb1 && ++pj < my_units) {
                const Unit w = unit_of(P, group, ngroups, pj);
                pb = w.b0;
                pb1 = w.b1;
            }
        };
        if (is_producer && lane == 0)
            for (long it = 0; it < kStages && it < total; ++it) load_next(it);
        const int g = lane >> 2, l = lane & 3;
        const int i0 = ws * NT * 8;                       // first sample of this warp inside the CTA's slice
        const int ig = rank * Cfg::kNPad + i0;            // ... and inside the residual row
        // lane-constant shared-memory offsets of the two operand patterns
        const int offS = g * XS + ((i0 + 2 * l) ^ ((g & 2) << 1));         // + nt*8   (16-byte loads)
        const int offU0 = l * XS + ((i0 + g) ^ ((l & 2) << 1));            // ks = 0, + nt*8
        const int offU1 = (l + 4) * XS + ((i0 + g) ^ ((l & 2) << 1));      // ks = 1 (snp l+4 has the same bit 1)
        const int offD = d_off<kT>(g, l);                                  // -Delta[trait g][snp l]; + 16 mt, + 4 kT (snp l + 4)
        const int offP = sp_off(g, 2 * l);                                 // S partial pair; + 64 mt
        uint32_t dcons_leader[2] = {0, 0}, rsqbar_leader = 0, rsq_all_leader = 0;
        if (kCl) {
            dcons_leader[0] = mapa_u32(&dcons[0], 0);
            dcons_leader[1] = mapa_u32(&dcons[1], 0);
            rsqbar_leader = mapa_u32(&rsqbar[0], 0);
            rsq_all_leader = mapa_u32(rsq_all, 0);
        }
        double acc[MT][NT][2];
        long gb = 0;  // global block counter of this CTA (drives ring stage and barrier parity)
        for (int ju = 0; ju < my_units; ++ju) {
            const Unit un = unit_of(P, group, ngroups, ju);
            const int k0 = P.k_base + un.tile * kT;
            unit_acquire(P, un, lane);   // the residual of this tile as the previous segment left it
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    const double2 v = __ldcg(reinterpret_cast<const double2*>(
                        P.resid + (size_t)(k0 + mt * 8 + g) * P.ld_resid + ig + nt * 8 + 2 * l));
                    acc[mt][nt][0] = v.x;
                    acc[mt][nt][1] = v.y;
                }
            constexpr int kSC = (MT >= 4) ? 1 : 2;   // accumulator chains per M tile of the S phase
            double sa[MT][2][2];
            // missing responses: bit 2 nt + e of mb[mt] = this lane's accumulator element (mt, nt, e) belongs to an observed sample
            uint32_t mb[MT];
            if constexpr (kMis) {
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) {
                    const unsigned long long* row = P.mbits + (size_t)(k0 + mt * 8 + g) * P.mwords;
                    uint32_t bits = 0;
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const int smp = ig + nt * 8 + 2 * l + e;
                            bits |= (uint32_t)((__ldg(row + (smp >> 6)) >> (smp & 63)) & 1ull) << (2 * nt + e);
                        }
                    mb[mt] = bits;
                }
            }
            // S phase of block gbi: the split-K DMMAs of S'^T = R^T X_b into the accumulators sa, then the accumulator chains
            // added, the partials stored and the chain warp told
            auto s_phase = [&](long gbi) {
                const int stage = (int)(gbi % kStages);
                AQ_T0();
                mbar_wait(&full[stage], (uint32_t)((gbi / kStages) & 1));
                AQ_T(10);
                const double* xt = tiles + stage * Cfg::kTileDoubles;
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) sa[mt][0][0] = sa[mt][0][1] = sa[mt][1][0] = sa[mt][1][1] = 0.0;
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    const double2 xb = *reinterpret_cast<const double2*>(xt + offS + nt * 8);
                    // (issue order keeps DMMAs on the same accumulator at least MT issue slots apart)
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt) dmma(sa[mt][0][0], sa[mt][0][1], acc[mt][nt][0], xb.x);
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt) dmma(sa[mt][kSC - 1][0], sa[mt][kSC - 1][1], acc[mt][nt][1], xb.y);
                }
                AQ_T(11);
                if (gbi > 0) mbar_wait(&sfree[0], (uint32_t)((gbi - 1) & 1));  // the previous block's partials have been read
                AQ_T(12);
                double* sp = spart + (size_t)ws * kT * Cfg::kSps + offP;
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) {
                    double2 v;  // C fragment: S^T[trait g + 8 mt][snp 2l, 2l + 1]
                    v.x = (kSC == 2) ? sa[mt][0][0] + sa[mt][1][0] : sa[mt][0][0];
                    v.y = (kSC == 2) ? sa[mt][0][1] + sa[mt][1][1] : sa[mt][0][1];
                    *reinterpret_cast<double2*>(sp + mt * 8 * Cfg::kSps) = v;
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&sdone[(gbi & 1) * 4 + smsp]);
                AQ_T(13);
            };
            if (P.mode == 0) s_phase(gb);
            for (int b = un.b0; b < un.b1; ++b, ++gb) {
                if (P.mode == 0 && b + 1 < un.b1) s_phase(gb + 1);
                // ---- rank-8 update with -Delta_b
                const int stage = (int)(gb % kStages);
                AQ_T0();
                if (P.mode != 0) mbar_wait(&full[stage], (uint32_t)((gb / kStages) & 1));  // sweep mode: S phase waited
                // (followers: -Delta arrives by an async bulk copy accounted on this barrier, so a CTA-scope wait is enough;
                // an acquire.cluster wait would invalidate L1 (CCTL.IVALL) on every block)
                mbar_wait(&dready[gb & 1], (uint32_t)((gb >> 1) & 1));
                AQ_T(14);
                const double* xt = tiles + stage * Cfg::kTileDoubles;
                const double* db = dbuf + (size_t)(gb & 1) * kT * kBlk;
                if (kCl && rank == 0) {
                    // leader: forward the kT x 8 block of -Delta to every follower, one 16-byte asynchronous DSMEM store per
                    // lane, accounted on the follower's barrier (armed by its reducer warp)
                    constexpr int kV2 = kT * kBlk / 2;
                    const int nsend = (ncta - 1) * kV2;
                    for (int L = mtid; L < nsend; L += Cfg::kMmaWarps * 32) {
                        const int r2 = 1 + L / kV2, idx = L % kV2;
                        const double2 v = *reinterpret_cast<const double2*>(db + 2 * idx);
                        st_async_v2(mapa_u32(db + 2 * idx, r2), v.x, v.y, mapa_u32(&dready[gb & 1], r2));
                    }
                }
                double nd[MT][2];
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) {
                    nd[mt][0] = db[offD + 16 * mt];
                    nd[mt][1] = db[offD + 16 * mt + 4 * kT];
                }
                if (P.mode != 0) {
                    // no S phase paces the chain in this mode: tell it that -Delta buffer (gb & 1) has been consumed,
                    // otherwise it could run two blocks ahead, overwrite the buffer and alias the barrier phase
                    __syncwarp();
                    if (lane == 0) {
                        if (kCl) mbar_arrive_cluster(dcons_leader[gb & 1]);
                        else mbar_arrive(&dcons[gb & 1]);
                    }
                }
#pragma unroll
                for (int nt = 0; nt < NT; nt += 2) {
                    // two sample tiles at a time: the two K-steps on one accumulator end up 2 MT issue slots apart
                    constexpr int kLast = NT - 1;
                    const int nt1 = nt + 1 < NT ? nt + 1 : kLast;
                    const bool two = nt + 1 < NT;
                    const double x0a = xt[offU0 + nt * 8], x1a = xt[offU1 + nt * 8];
                    const double x0b = xt[offU0 + nt1 * 8], x1b = xt[offU1 + nt1 * 8];
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt) dmma(acc[mt][nt][0], acc[mt][nt][1], nd[mt][0], x0a);
                    if (two) {
#pragma unroll
                        for (int mt = 0; mt < MT; ++mt) dmma(acc[mt][nt1][0], acc[mt][nt1][1], nd[mt][0], x0b);
                    }
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt) dmma(acc[mt][nt][0], acc[mt][nt][1], nd[mt][1], x1a);
                    if (two) {
#pragma unroll
                        for (int mt = 0; mt < MT; ++mt) dmma(acc[mt][nt1][0], acc[mt][nt1][1], nd[mt][1], x1b);
                    }
                }
                if constexpr (kMis) {
                    // keep the residual masked: r_k -= delta (mis_k o x_j)  (src/coreLoop.cpp:132 in sample space)
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                        for (int nt = 0; nt < NT; ++nt) {
                            if (!((mb[mt] >> (2 * nt)) & 1u)) acc[mt][nt][0] = 0.0;
                            if (!((mb[mt] >> (2 * nt + 1)) & 1u)) acc[mt][nt][1] = 0.0;
                        }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[stage]);
                AQ_T(15);
                if (is_producer) {  // refill the stage once every MMA warp has released it
                    if (lane == 0 && gb + kStages < total) {
                        mbar_wait(&empty[stage], (uint32_t)((gb / kStages) & 1));
                        load_next(gb + kStages);
                    }
                    __syncwarp();
                }
            }
            // ---- unit epilogue: store the residual; after the last segment of the tile, the per-trait squared norms
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
                double ss = 0.0;
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    double2 v;
                    v.x = acc[mt][nt][0];
                    v.y = acc[mt][nt][1];
                    ss = fma(v.x, v.x, ss);
                    ss = fma(v.y, v.y, ss);
                    *reinterpret_cast<double2*>(P.resid + (size_t)(k0 + mt * 8 + g) * P.ld_resid + ig + nt * 8 + 2 * l) = v;
                }
                ss += __shfl_xor_sync(0xffffffffu, ss, 1);
                ss += __shfl_xor_sync(0xffffffffu, ss, 2);
                if (l == 0) rsqs[ws * kT + mt * 8 + g] = ss;
            }
            const bool last_seg = un.seg == P.nseg - 1;
            asm volatile("bar.sync 1, %0;" ::"n"(Cfg::kMmaWarps * 32) : "memory");
            if (mtid < 32 * ((kT + 31) / 32)) {  // whole warps, so that the elected arrive below is warp-uniform
                double ss = 0.0;
                if (mtid < kT) {
#pragma unroll
                    for (int w2 = 0; w2 < WS; ++w2) ss += rsqs[w2 * kT + mtid];
                }
                if (!kCl) {
                    if (last_seg && mtid < kT && k0 + mtid < P.q) P.rsq[k0 + mtid] = ss;
                } else if (rank != 0) {
                    if (mtid < kT) st_cluster_f64(rsq_all_leader + (uint32_t)(((rank - 1) * kT + mtid) * sizeof(double)), ss);
                    // release.cluster arrive below is cumulative over the stores ordered before it by __syncwarp
                    __syncwarp();
                    if (mtid == 0) mbar_arrive_cluster(rsqbar_leader);
                } else {
                    if (ncta > 1) mbar_wait_cluster(&rsqbar[0], (uint32_t)(ju & 1));
                    if (mtid < kT) {
                        for (int r2 = 1; r2 < ncta; ++r2) ss += rsq_all[(r2 - 1) * kT + mtid];  // fixed order: deterministic
                        if (last_seg && k0 + mtid < P.q) P.rsq[k0 + mtid] = ss;
                    }
                }
            }
            asm volatile("bar.sync 1, %0;" ::"n"(Cfg::kMmaWarps * 32) : "memory");
            unit_release<Cfg>(P, un);
        }
    } else if (is_chain && rank != 0) {
        // ------------------------------------------------------------------ follower CTA: S-tile reducer warp
        // Arms this CTA's -Delta barrier for every block (the leader's asynchronous stores complete it) and, in sweep
        // mode, sums this CTA's WS split-K partials and ships the kT x 8 tile into the leader's shared memory with
        // st.async (fire-and-forget DSMEM stores whose bytes are accounted on the leader's barrier: no remote arrive,
        // no fence).  With <= 16 traits per tile the two half-warps split the work.
        constexpr int kH = (kT <= 16) ? 2 : 1;
        constexpr int kTP = kBlk / kH;
        const int half = (kH == 2) ? (lane >> 4) : 0;
        const int tl = (kH == 2) ? (lane & 15) : lane;
        const bool active = tl < kT;
        const int tls = active ? tl : 0;
        const uint32_t red_leader = mapa_u32(red, 0);
        const uint32_t sred_leader[2] = {mapa_u32(&sred[0], 0), mapa_u32(&sred[1], 0)};
        long gb = 0;
        for (int ju = 0; ju < my_units; ++ju) {
            const Unit un = unit_of(P, group, ngroups, ju);
            for (int b = un.b0; b < un.b1; ++b, ++gb) {
                if (gb >= 2) mbar_wait(&dready[gb & 1], (uint32_t)(((gb >> 1) - 1) & 1));  // the phase of block gb - 2 is over
                if (lane == 0) mbar_arrive_expect_tx(&dready[gb & 1], Cfg::kDeltaBytes);
                if (P.mode != 0) continue;
                double s[kBlk];
                sum_own_partials<Cfg>(s, spart, sdone, sfree, gb, lane, tls);
                if (kH == 2) {
#pragma unroll
                    for (int t = 0; t < kBlk; ++t) s[t] += __shfl_xor_sync(0xffffffffu, s[t], 16);
                }
                if (active) {
                    const uint32_t dst = red_leader + (uint32_t)((((gb & 1) * (kMaxCluster - 1)) + (rank - 1)) * kT *
                                                                 Cfg::kSps * sizeof(double));
#pragma unroll
                    for (int i = 0; i < kTP; i += 2) {
                        const int t = half * kTP + i;
                        st_async_v2(dst + (uint32_t)sp_off(tl, t) * (uint32_t)sizeof(double), s[t], s[t + 1], sred_leader[gb & 1]);
                    }
                }
            }
            unit_release<Cfg>(P, un);
        }
    } else if (is_helper) {
        // ------------------------------------------------------------------ helper warp (leader CTA, sweep mode)
        // Everything of a block that is NOT the serial recurrence.  Before the chain needs them, the block's inputs
        // beta_old and c (D + cst) are staged in shared memory (their p x q rows arrive by asynchronous copies issued
        // one block earlier, so no HBM / L2 latency sits between "S is complete" and "the chain may start") and the
        // split-K partials of S are summed; after the chain, gam / mu go back to HBM and the per-trait running sums
        // are accumulated.  With <= 16 traits per tile the two half-warps split the work.
        constexpr int kH = (kT <= 16) ? 2 : 1;
        constexpr int kTP = kBlk / kH;           // SNP slots per lane
        // W / I0 of a block: staged with the other rows when a lane handles 4 SNP slots; with 8 slots per lane (T > 16)
        // the extra asynchronous copies cost more than they hide, and W / I0 are requested directly one block ahead
        constexpr bool kStageWI = (kH == 2);
        const int half = (kH == 2) ? (lane >> 4) : 0;
        const int tl = (kH == 2) ? (lane & 15) : lane;
        const bool active = tl < kT;
        const int tls = active ? tl : 0;
        const int t0 = half * kTP;
        const bool work = P.mode == 0 && rank == 0;
        int idn[kTP], idc[kTP];
        double wn[kTP], in[kTP];   // W, I0 of the block being prepared: consumed after its chain
        long gb = 0;
        for (int ju = 0; ju < my_units; ++ju) {
            const Unit un = unit_of(P, group, ngroups, ju);
            if (work) {
                const int tile = un.tile;
                const int k = P.k_base + tile * kT + tls;
                const bool valid = active && k < P.q;
                // src/coreLoop.cpp:56; with missing responses :108 (log sig2_beta_vb(j, k) enters per pair, :129)
                double cst;
                if constexpr (kMis) cst = -(P.log_tau[k] + P.log_sig2_inv) / 2;
                else cst = -(P.log_tau[k] + P.log_sig2_inv + log(P.sig2_beta[k])) / 2;
                const double ctau = P.c * P.tau[k], inv_ctau = 1.0 / ctau;   // (missing responses) sig2_beta = a / (c tau)
                double sg = 0.0, sgm2 = 0.0, sb2 = 0.0, sz = 0.0;
                double ss2g = 0.0, sxgm2 = 0.0, sxs2g = 0.0, sxb2 = 0.0, sgl = 0.0;   // missing-response sums (aq_mis.cuh)
                double xnn[kTP], s2n[kTP], lsn[kTP];   // X_norm_sq, sig2_beta, log sig2_beta of the block being prepared
                double* rowrow = P.rowpart ? P.rowpart + (size_t)(P.rowpart_base + tile) * P.p_pad : nullptr;
                // asynchronous copies (LDGSTS) of this lane's gam / mu / D / W / I0 elements of block `blk` into the staging
                // buffer: issued a whole block ahead, so neither preparing a block nor finishing it ever waits on HBM or L2
                auto stage_rows = [&](int blk) {
                    // 16-byte copies: a row of kT traits is kT / 2 lanes wide, so one instruction covers 64 / kT rows
                    constexpr int kLanesPerRow = kT / 2, kRowsPerInst = 32 / kLanesPerRow;
                    constexpr int kArrays = kMis ? 8 : (kStageWI ? 5 : 3);
                    static_assert(!kMis || kStageWI, "the missing-response variant stages all its rows");
                    const int idr = __ldg(P.order + (size_t)blk * kBlk + (lane & 7));
                    const int rsub = lane / kLanesPerRow, csub = 2 * (lane % kLanesPerRow);
                    const size_t kcol = (size_t)P.k_base + (size_t)tile * kT + csub;
#pragma unroll
                    for (int r0 = 0; r0 < kArrays * kBlk; r0 += kRowsPerInst) {
                        const int row = r0 + rsub;                       // (array, SNP slot) = (row / 8, row % 8)
                        const int a = row / kBlk, t = row % kBlk;
                        const int idt = __shfl_sync(0xffffffffu, idr, t);
                        if (row < kArrays * kBlk) {
                            const double* base = a == 0 ? P.gam : a == 1 ? P.mu : a == 2 ? P.dtab : a == 3 ? P.wtab :
                                                 a == 4 ? P.i0tab : a == 5 ? P.xnsq : a == 6 ? P.atab : P.ltab;
                            cp_async16(stg + (size_t)row * kT + csub, base + (size_t)(idt < 0 ? 0 : idt) * P.q_pad + kcol);
                        }
                    }
                    cp_async_commit();
                };
                // missing responses: the per-trait Gram band of block `blk` (16 KB) -> buffer g & 1, 32 copies per lane
                auto stage_gk = [&](long g, int blk) {
                    if constexpr (kMis) {
                        const double* src = P.gk + (((size_t)(P.k_base / kT + tile) * P.nb + blk) * 128) * kT;
                        double* dst = gkbuf + (size_t)(g & 1) * 128 * kT;
                        for (int i = lane; i < 128 * kT / 2; i += 32) cp_async16(dst + 2 * i, src + 2 * i);
                        cp_async_commit();
                    }
                };
                auto pre = [&](long g, int blk) {
                    AQ_T0();
                    double* io = iobuf + (size_t)(g & 1) * kBlk * kIoPer * kT;
                    cp_async_wait_all();  // issued a whole block earlier
                    __syncwarp();         // (each lane waited for its own copies; the rows are read by other lanes)
#pragma unroll
                    for (int i = 0; i < kTP; ++i) {
                        const int t = t0 + i;
                        idn[i] = __ldg(P.order + (size_t)blk * kBlk + t);
                        const double go = stg[(0 * kBlk + t) * kT + tls], mo = stg[(1 * kBlk + t) * kT + tls];
                        const double dd = stg[(2 * kBlk + t) * kT + tls];
                        if (kStageWI) {
                            wn[i] = stg[(3 * kBlk + t) * kT + tls];
                            in[i] = stg[(4 * kBlk + t) * kT + tls];
                        }
                        if constexpr (kMis) {
                            const double xn = stg[(5 * kBlk + t) * kT + tls], aa = stg[(6 * kBlk + t) * kT + tls];
                            const double ls = stg[(7 * kBlk + t) * kT + tls];
                            xnn[i] = xn;
                            s2n[i] = aa * inv_ctau;        // sig2_beta_vb(j, k), update_sig2_beta_vb_ R/update_vb.R:47
                            lsn[i] = ls;
                            if (active) {
                                io[(t * kIoPer + 0) * kT + tl] = idn[i] >= 0 ? go * mo : 0.0;
                                io[(t * kIoPer + 1) * kT + tl] = P.c * (dd - 0.5 * ls + cst);   // :127-129 without the mu^2 term
                                io[(t * kIoPer + 2) * kT + tl] = aa;                            // mu = a s              (:125)
                                io[(t * kIoPer + 3) * kT + tl] = 0.5 * P.c * aa * ctau;         // c mu^2 / (2 sig2_beta) = bq s^2
                            }
                        } else if (active) {
                            io[(t * kIoPer + 0) * kT + tl] = idn[i] >= 0 ? go * mo : 0.0;  // beta_old (0 for padding slots)
                            io[(t * kIoPer + 1) * kT + tl] = P.c * (dd + cst);              // :75-77 without the mu^2 term
                        }
                    }
                    if (blk + 1 < un.b1) stage_rows(blk + 1);
                    if constexpr (Cfg::kHelperSumsFollowers) {
                        // the other CTAs' S tiles, summed here while the chain warp sums this CTA's own partials
                        if (ncta > 1) {
                            double s[kBlk];
                            sum_follower_tiles<Cfg>(s, red, sred, g, ncta, lane, tls);
                            if (half == 0 && active) {
#pragma unroll
                                for (int t = 0; t < kBlk; t += 2) {
                                    double2 v;
                                    v.x = s[t];
                                    v.y = s[t + 1];
                                    *reinterpret_cast<double2*>(ssum + (size_t)(g & 1) * kT * Cfg::kSps + sp_off(tl, t)) = v;
                                }
                            }
                        }
                    }
                    if (!Cfg::kChainSums) {
                        AQ_T(4);
                        double s[kBlk];
                        sum_s_partials<Cfg>(s, spart, red, sdone, sfree, sred, g, ncta, lane, tls);
                        if (half == 0 && active) {
#pragma unroll
                            for (int t = 0; t < kBlk; t += 2) {
                                double2 v;
                                v.x = s[t];
                                v.y = s[t + 1];
                                *reinterpret_cast<double2*>(ssum + (size_t)(g & 1) * kT * Cfg::kSps + sp_off(tl, t)) = v;
                            }
                        }
                    }
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&inready[g & 1]);
                    AQ_T(7);
                };
                auto post = [&](long g, int blk, const double (&ww)[kTP], const double (&ii)[kTP], const double (&xc)[kTP],
                                const double (&s2c)[kTP], const double (&lsc)[kTP]) {
                    AQ_T0();
                    mbar_wait(&dready[g & 1], (uint32_t)((g >> 1) & 1));
                    AQ_T(8);
                    if (blk + 2 < un.b1) stage_gk(g + 2, blk + 2);   // the chain is through with buffer g & 1
                    const double* io = iobuf + (size_t)(g & 1) * kBlk * kIoPer * kT;
                    double zrow[kTP];
#pragma unroll
                    for (int i = 0; i < kTP; ++i) {
                        const int t = t0 + i;
                        const double gm = io[(t * kIoPer + 0) * kT + tls];
                        const double m = io[(t * kIoPer + 1) * kT + tls];
                        zrow[i] = 0.0;
                        if (idc[i] >= 0) {
                            const double bn = gm * m;  // :79
                            const double z = fma(gm, ww[i], ii[i]);
                            sg += gm;
                            sgm2 = fma(bn, m, sgm2);
                            sb2 = fma(bn, bn, sb2);
                            sz += z;
                            if constexpr (kMis) {
                                ss2g = fma(s2c[i], gm, ss2g);
                                sxgm2 = fma(xc[i] * bn, m, sxgm2);
                                sxs2g = fma(xc[i] * s2c[i], gm, sxs2g);
                                sxb2 = fma(xc[i] * bn, bn, sxb2);
                                sgl = fma(gm, lsc[i], sgl);
                            }
                            if (valid) {
                                const size_t off = (size_t)idc[i] * P.q_pad + k;
                                P.gam[off] = gm;
                                P.mu[off] = m;
                                if (!kCl) zrow[i] = z;
                            }
                        }
                    }
                    if (!kCl && P.rowpart) {  // (never requested from a clustered launch)
                        // this tile's share of rowSums(Z) (update_theta_vb_, R/update_vb.R:179): the products are here anyway,
                        // so the p x q arrays are not read a second time for them.  Lanes of a half-warp (a warp if kT > 16)
                        // hold the traits; after the halving sums lane L owns SNP slot (L >> 2) & (kTP - 1) of its half.
                        group_sums<kTP>(zrow, lane, kH == 2 ? 8 : 16);
                        const int slot = (lane >> 2) & (kTP - 1);
                        int ids = idc[0];
#pragma unroll
                        for (int i = 1; i < kTP; ++i) ids = slot == i ? idc[i] : ids;
                        if ((lane & 3) == 0 && ids >= 0) rowrow[ids] = zrow[0];
                    }
                    AQ_T(9);
                };
                stage_gk(gb, un.b0);
                if (un.b0 + 1 < un.b1) stage_gk(gb + 1, un.b0 + 1);
                stage_rows(un.b0);
                pre(gb, un.b0);
                for (int b = un.b0; b < un.b1; ++b, ++gb) {
                    double ww[kTP], ii[kTP], xc[kTP], s2c[kTP], lsc[kTP];
#pragma unroll
                    for (int i = 0; i < kTP; ++i) {
                        idc[i] = idn[i];
                        xc[i] = xnn[i];
                        s2c[i] = s2n[i];
                        lsc[i] = lsn[i];
                        if (kStageWI) {
                            ww[i] = wn[i];
                            ii[i] = in[i];
                        } else {  // requested before the next block is prepared, consumed after the chain
                            const size_t off = (size_t)(idc[i] < 0 ? 0 : idc[i]) * P.q_pad + k;
                            ww[i] = P.wtab[off];
                            ii[i] = P.i0tab[off];
                        }
                    }
                    if (b + 1 < un.b1) pre(gb + 1, b + 1);
                    post(gb, b, ww, ii, xc, s2c, lsc);
                }
                if (kH == 2) {
                    sg += __shfl_xor_sync(0xffffffffu, sg, 16);
                    sgm2 += __shfl_xor_sync(0xffffffffu, sgm2, 16);
                    sb2 += __shfl_xor_sync(0xffffffffu, sb2, 16);
                    sz += __shfl_xor_sync(0xffffffffu, sz, 16);
                    if constexpr (kMis) {
                        ss2g += __shfl_xor_sync(0xffffffffu, ss2g, 16);
                        sxgm2 += __shfl_xor_sync(0xffffffffu, sxgm2, 16);
                        sxs2g += __shfl_xor_sync(0xffffffffu, sxs2g, 16);
                        sxb2 += __shfl_xor_sync(0xffffffffu, sxb2, 16);
                        sgl += __shfl_xor_sync(0xffffffffu, sgl, 16);
                    }
                }
                unit_acquire(P, un, lane);   // the column sums of the earlier segments (fixed order: deterministic)
                if constexpr (kMis) {   // (never segmented: one unit per tile)
                    if (valid && half == 0) {
                        double* o = P.mis_out + k;
                        o[(size_t)kMisGam * P.q_pad] = sg;
                        o[(size_t)kMisGamMu2 * P.q_pad] = sgm2;
                        o[(size_t)kMisS2Gam * P.q_pad] = ss2g;
                        o[(size_t)kMisXnGamMu2 * P.q_pad] = sxgm2;
                        o[(size_t)kMisXnS2Gam * P.q_pad] = sxs2g;
                        o[(size_t)kMisXnBeta2 * P.q_pad] = sxb2;
                        o[(size_t)kMisZ * P.q_pad] = sz;
                        o[(size_t)kMisGamLogS2 * P.q_pad] = sgl;
                    }
                } else if (valid && half == 0) {
                    if (un.seg > 0) {
                        sg += __ldcg(P.cs_gam + k);
                        sgm2 += __ldcg(P.cs_gmu2 + k);
                        sb2 += __ldcg(P.cs_b2 + k);
                        sz += __ldcg(P.cs_z + k);
                    }
                    P.cs_gam[k] = sg;
                    P.cs_gmu2[k] = sgm2;
                    P.cs_b2[k] = sb2;
                    P.cs_z[k] = sz;
                }
            }
            unit_release<Cfg>(P, un);
        }
    } else if (is_chain) {
        // ------------------------------------------------------------------ chain warp (one lane per trait; leader CTA)
        const int tl = lane;
        const bool active = tl < kT;
        const int tls = active ? tl : 0;  // inactive lanes shadow trait 0 without side effects
        // summation of the S partials: lanes 16-31 take the second half of the partials of trait (lane & 15) when kT <= 16;
        // they then shadow that trait through the recurrence, still without side effects
        const int tsum0 = (kT <= 16) ? (lane & 15) : lane;
        const int tsum = tsum0 < kT ? tsum0 : 0;
        // -Delta leaves for this CTA's MMA warps (which forward it to the other CTAs of a cluster): this warp never issues
        // a remote operation, they would sit in its load/store queue on the serial path
        auto publish = [&](long gb, const double (&nd)[kBlk]) {
            double* dblk = dbuf + (size_t)(gb & 1) * kT * kBlk;
            if (active) {
#pragma unroll
                for (int t = 0; t < kBlk; t += 2) {
                    double2 v;
                    v.x = nd[t];
                    v.y = nd[t + 1];
                    *reinterpret_cast<double2*>(dblk + d_off<kT>(tl, t)) = v;
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&dready[gb & 1]);
        };
        long gb = 0;
        for (int ju = 0; ju < my_units; ++ju) {
            const Unit un = unit_of(P, group, ngroups, ju);
            const int k = P.k_base + un.tile * kT + tls;
            const bool valid = active && k < P.q;
            if (P.mode == 0) {
                // ---- sweep: only the serial recurrence lives here; inputs arrive through shared memory (helper warp)
                double a = 0.0, bq = 0.0;   // (missing responses: per pair, through shared memory with the other inputs)
                if constexpr (!kMis) {
                    const double sig2 = P.sig2_beta[k];
                    a = P.c * sig2 * P.tau[k];                      // src/coreLoop.cpp:73:  mu = a * s
                    bq = P.c * a * a / (2.0 * sig2);                // :76  c * mu^2 / (2 sig2_beta) = bq * s^2
                }
                double corr[kBlk];  // look-ahead correction of the NEXT block, accumulated while this one is resolved
#pragma unroll
                for (int t = 0; t < kBlk; ++t) corr[t] = 0.0;
                for (int b = un.b0; b < un.b1; ++b, ++gb) {
                    AQ_T0();
                    const int stage = (int)(gb % kStages);
                    mbar_wait(&full[stage], (uint32_t)((gb / kStages) & 1));
                    // Gram band of the block, entry (t, u) at gband[(t * 16 + u) * gstride]: the tile image's band, shared by
                    // all traits -- or, with missing responses, this lane's column of the per-trait band the helper fetched
                    const double* gband = kMis ? gkbuf + (size_t)(gb & 1) * 128 * kT + tsum
                                               : tiles + stage * Cfg::kTileDoubles + kBlk * XS;
                    constexpr int gstride = kMis ? kT : 1;
                    double* io = iobuf + (size_t)(gb & 1) * kBlk * kIoPer * kT;
                    double s[kBlk], bo[kBlk], ap[kBlk], nd[kBlk], av[kMis ? kBlk : 1], bv[kMis ? kBlk : 1];
                    if constexpr (Cfg::kHelperSumsFollowers) {
                        // clusters: this CTA's partials first (they only need the MMA warps), then the inputs and the other
                        // CTAs' part of S, both prepared by the helper warp meanwhile
                        AQ_T(0);
                        sum_own_partials<Cfg>(s, spart, sdone, sfree, gb, lane, tsum);
                        if (kT <= 16) {
#pragma unroll
                            for (int t = 0; t < kBlk; ++t) s[t] += __shfl_xor_sync(0xffffffffu, s[t], 16);
                        }
                    }
                    mbar_wait(&inready[gb & 1], (uint32_t)((gb >> 1) & 1));   // beta_old, c (D + cst): staged a block ahead
#pragma unroll
                    for (int t = 0; t < kBlk; ++t) {
                        bo[t] = io[(t * kIoPer + 0) * kT + tsum];
                        ap[t] = io[(t * kIoPer + 1) * kT + tsum];
                        if constexpr (kMis) {
                            av[t] = io[(t * kIoPer + 2) * kT + tsum];
                            bv[t] = io[(t * kIoPer + 3) * kT + tsum];
                        }
                    }
                    if constexpr (Cfg::kHelperSumsFollowers) {
                        if (ncta > 1) {
                            const double* sp0 = ssum + (size_t)(gb & 1) * kT * Cfg::kSps;
#pragma unroll
                            for (int t = 0; t < kBlk; t += 2) {
                                const double2 v = *reinterpret_cast<const double2*>(sp0 + sp_off(tsum, t));
                                s[t] += v.x;
                                s[t + 1] += v.y;
                            }
                        }
                    } else if (Cfg::kChainSums) {
                        // S = X_b' R: this warp sums the split-K partials itself the moment the MMA warps have delivered
                        // them; no other warp sits between the tensor work and the recurrence
                        AQ_T(0);
                        sum_s_partials<Cfg>(s, spart, red, sdone, sfree, sred, gb, ncta, lane, tsum);
                    } else {
                        AQ_T(0);
                        const double* sp0 = ssum + (size_t)(gb & 1) * kT * Cfg::kSps;
#pragma unroll
                        for (int t = 0; t < kBlk; t += 2) {
                            const double2 v = *reinterpret_cast<const double2*>(sp0 + sp_off(tsum, t));
                            s[t] = v.x;
                            s[t + 1] = v.y;
                        }
                    }
#pragma unroll
                    for (int t = 0; t < kBlk; ++t) {
                        // S was formed before the previous block's update was applied (corr); leave-one-out: + beta_old |X_t|^2
                        s[t] = fma(bo[t], gband[(t * 16 + 8 + t) * gstride], s[t] + corr[t]);
                        corr[t] = 0.0;
                    }
                    AQ_T(1);
#pragma unroll
                    for (int t = 0; t < kBlk; ++t) {
                        const double st = s[t];
                        const double m = (kMis ? av[kMis ? t : 0] : a) * st;                        // :73  (:125)
                        const double x = fma(st * st, -(kMis ? bv[kMis ? t : 0] : bq), ap[t]);      // :75-77  (:127-129)
                        const double gm = logistic_neg<Cfg::kShortLogistic>(x);   // 1/(1+e^x) == exp(-log1pexp(x))
                        const double dlt = fma(gm, m, -bo[t]);               // :79 beta_new - beta_old (0 for padding slots)
                        const double* grow = gband + t * 16 * gstride;       // row t: [next block | this block]
#pragma unroll
                        for (int u = t + 1; u < kBlk; ++u) s[u] = fma(-grow[(8 + u) * gstride], dlt, s[u]);
#pragma unroll
                        for (int u = 0; u < kBlk; ++u) corr[u] = fma(-grow[u * gstride], dlt, corr[u]);
                        nd[t] = -dlt;
                        if (active) {
                            io[(t * kIoPer + 0) * kT + tl] = gm;
                            io[(t * kIoPer + 1) * kT + tl] = m;
                        }
                    }
                    AQ_T(2);
                    publish(gb, nd);
                    AQ_T(3);
                }
            } else {
                // ---- mode 1: R = Y - X beta from the loaded state, and its per-trait sums
                double sg = 0.0, sgm2 = 0.0, sb2 = 0.0, sxg = 0.0, sxgm2 = 0.0, sxb2 = 0.0;
                for (int b = un.b0; b < un.b1; ++b, ++gb) {
                    const int stage = (int)(gb % kStages);
                    mbar_wait(&full[stage], (uint32_t)((gb / kStages) & 1));
                    const int* ids = reinterpret_cast<const int*>(tiles + stage * Cfg::kTileDoubles + kBlk * XS + 128);
                    double nd[kBlk];
#pragma unroll
                    for (int t = 0; t < kBlk; ++t) {
                        const int idt = ids[t];
                        const size_t off = (size_t)(idt < 0 ? 0 : idt) * P.q_pad + k;
                        const double go = P.gam[off], mo = P.mu[off];
                        const double bo = idt >= 0 ? go * mo : 0.0;
                        if (idt >= 0) {
                            sg += go;
                            sgm2 = fma(bo, mo, sgm2);
                            sb2 = fma(bo, bo, sb2);
                            if constexpr (kMis) {
                                const double xn = P.xnsq[off];
                                sxg = fma(xn, go, sxg);
                                sxgm2 = fma(xn * bo, mo, sxgm2);
                                sxb2 = fma(xn * bo, bo, sxb2);
                            }
                        }
                        nd[t] = -bo;
                    }
                    if (gb >= 2) {  // -Delta buffer (gb & 1) free again in every CTA
                        if (kCl) mbar_wait_cluster(&dcons[gb & 1], (uint32_t)(((gb >> 1) - 1) & 1));
                        else mbar_wait(&dcons[gb & 1], (uint32_t)(((gb >> 1) - 1) & 1));
                    }
                    publish(gb, nd);
                }
                unit_acquire(P, un, lane);
                if constexpr (kMis) {   // rows as mis_sweep_kernel's mode 1 leaves them (aq_mis.cuh)
                    if (valid) {
                        double* o = P.mis_out + k;
                        o[(size_t)kMisGam * P.q_pad] = sg;
                        o[(size_t)kMisGamMu2 * P.q_pad] = sgm2;
                        o[(size_t)kMisS2Gam * P.q_pad] = sb2;
                        o[(size_t)kMisXnGamMu2 * P.q_pad] = sxgm2;
                        o[(size_t)kMisXnS2Gam * P.q_pad] = sxg;
                        o[(size_t)kMisXnBeta2 * P.q_pad] = sxb2;
                    }
                } else if (valid) {
                    if (un.seg > 0) {
                        sg += __ldcg(P.cs_gam + k);
                        sgm2 += __ldcg(P.cs_gmu2 + k);
                        sb2 += __ldcg(P.cs_b2 + k);
                    }
                    P.cs_gam[k] = sg;
                    P.cs_gmu2[k] = sgm2;
                    P.cs_b2[k] = sb2;
                }
            }
            unit_release<Cfg>(P, un);
        }
    }
#ifdef AQ_TIMING
    if (blockIdx.x == 0 && lane == 0 && P.timing && (is_chain || is_helper || wid == 0))
        for (int i = 0; i < 16; ++i)
            if (tacc[i]) atomicAdd(reinterpret_cast<unsigned long long*>(P.timing) + i, (unsigned long long)tacc[i]);
#endif
    if (kCl) {
        __syncwarp();
        cluster_sync_all();  // keep every CTA's shared memory alive until all remote stores / arrives have landed
    }
}

}  // namespace aq
