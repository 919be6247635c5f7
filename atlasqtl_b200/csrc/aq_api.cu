// C ABI of atlasqtl_b200 (include/atlasqtl_b200.h): context management, host <-> device layout
// conversion and kernel launches.  No torch, no CPU fallback: every entry point either runs the CUDA
// path or returns an error code.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <string>
#include <vector>

#include "../../include/atlasqtl_b200.h"
#include "aq_internal.h"
#include "aq_mis.cuh"
#include "aq_prep.cuh"
#include "aq_select.cuh"
#include "aq_stream.cuh"
#include "aq_sweep.cuh"

using namespace aq;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

#define AQ_CUDA(expr)                                                                                   \
    do {                                                                                                \
        cudaError_t e_ = (expr);                                                                        \
        if (e_ != cudaSuccess) {                                                                        \
            cudaGetLastError();                                                                         \
            return fail(e_ == cudaErrorMemoryAllocation ? AQ_ENOMEM : AQ_ECUDA,                         \
                        std::string(#expr) + ": " + cudaGetErrorString(e_));                            \
        }                                                                                               \
    } while (0)

// ---- kernel configurations (SweepCfg<MT, NT, clustered, missing>): picked by n and q at aq_create time, and again by
// aq_set_missing for the missing-response variant.  14 MMA warps split a CTA's samples (112 NT of them); each holds MT
// 8-trait tiles: MT * NT * 2 accumulator doubles (<= 42: the 16-warp CTA leaves 128 registers per thread).  n <= 1008: one
// CTA per trait tile.  n > 1008: a thread-block cluster of 2, 3, 4, 6 or 8 CTAs splits the samples (up to n = 7168).
// Traits / tile = 8 MT: 16, 24 or 32.  Beyond 16 the helper warp handles one trait per lane (no half-warp split), which the
// extra DSMEM hop of the clustered variant cannot afford at 7 sample tiles per warp.
constexpr int mt_of_nt(int nt, bool cl) { return nt >= (cl ? 7 : 8) ? 2 : (nt >= 6 ? 3 : 4); }
template <int NT, bool CL>
using CfgOf = SweepCfg<mt_of_nt(NT, CL), NT, CL>;
// Missing responses: 16-trait tiles, and fewer sample tiles per warp than the dense kernel so that the per-trait Gram band
// buffers (32 KB) fit beside the X tile ring.
template <int NT, bool CL>
using CfgMis = SweepCfg<2, NT, CL, true>;
// One compiled configuration (an entry of kSweepKernels).
struct SweepKernel {
    bool mis, cl;                     // missing-response variant; sample-split cluster variant
    int nt, n_pad, xs, kT, threads;   // n_pad: samples per CTA (slice), padded
    size_t smem, tile_doubles;
    int (*launch)(aq_ctx*, const SweepParams&);   // one sweep (mode 0) or residual set-up (mode 1) of a context
};
// the configuration a context runs: an entry of kSweepKernels and its number of CTAs per cluster (sample slices)
struct CfgInfo {
    const SweepKernel* k = nullptr;
    int ncta = 1;
};

// Test and development overrides, read from the environment once, when a context is created, so that no other thread's
// setenv can change the plan of a context while it sweeps:
//   AQ_NO_TAIL               (any value) leftover traits go through full-size tiles, never the 8-trait tail variant
//   AQ_NO_SEG                (any value) the SNP blocks of a tile are never cut into segments
//   AQ_NSEG=S                S segments per tile whenever the tiles outnumber one round of the persistent grid
//   AQ_FORCE_CLUSTER=c       c CTAs per cluster (1..8) wherever the samples fit
//   AQ_MIS_KERNEL=warp|tile  the kernel aq_set_missing chooses for missing responses
struct DevOverrides {
    bool no_tail = false, no_seg = false;
    int nseg = 0, force_cluster = 0;      // 0: not forced
    bool mis_warp = false, mis_tile = false;
};
DevOverrides read_overrides() {
    DevOverrides o;
    o.no_tail = std::getenv("AQ_NO_TAIL") != nullptr;
    o.no_seg = std::getenv("AQ_NO_SEG") != nullptr;
    if (const char* v = std::getenv("AQ_NSEG")) o.nseg = std::max(1, std::atoi(v));   // (< 2: no segment count matches)
    if (const char* v = std::getenv("AQ_FORCE_CLUSTER")) o.force_cluster = std::atoi(v);
    if (const char* v = std::getenv("AQ_MIS_KERNEL")) {
        o.mis_warp = std::strcmp(v, "warp") == 0;
        o.mis_tile = std::strcmp(v, "tile") == 0;
    }
    return o;
}

}  // namespace

struct aq_ctx {
    int device = 0, n = 0, p = 0, q = 0;
    int p_pad = 0, q_pad = 0, nb = 0, ntiles = 0, sm_count = 0, ld_resid = 0;
    CfgInfo cfg{};
    DevOverrides ov;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;  // sweep kernel
    cudaEvent_t evr0 = nullptr, evr1 = nullptr, evt0 = nullptr, evt1 = nullptr;  // rowsums / tables kernels
    float last_rows_ms = 0.f, last_tables_ms = 0.f;
    double *xraw = nullptr, *xtiles = nullptr, *ymat = nullptr, *resid = nullptr;
    double *gam = nullptr, *mu = nullptr, *dtab = nullptr, *wtab = nullptr, *i0tab = nullptr;
    double *tvec = nullptr;     // 3 x q_pad: tau, log_tau, sig2_beta
    double *ovec = nullptr;     // 5 x q_pad: cs_gam, cs_gmu2, cs_b2, rsq, cs_z
    double *theta = nullptr, *zeta = nullptr, *rowsum = nullptr, *partials = nullptr, *scalar = nullptr;
    double *stage = nullptr;    // transposition staging: stage_cols x p doubles
    int stage_cols = 0;
    size_t n_partials = 0;
    int* order_dev = nullptr;
    // missing responses (aq_set_missing): bit masks, X_norm_sq, per-trait observation counts and the sums of the NA kernels
    unsigned long long* mask = nullptr;
    double *xnsq = nullptr, *n_obs = nullptr, *mis_out = nullptr;
    double* sig2tab = nullptr;  // explicit p x q sig2_beta_vb (stateless coreDualMisLoop entry only)
    // tile-structured missing-response path (aq_sweep.cuh, MIS variant): observed-sample bit matrix, CSR lists of the
    // missing samples per trait, per-trait Gram band table, the two per-sweep p x q tables
    bool mis_tile = false;
    unsigned long long* mbits = nullptr;
    int mwords = 0;
    int *mis_off_dev = nullptr, *mis_idx_dev = nullptr;
    double *gk = nullptr, *atab = nullptr, *ltab = nullptr;
    bool has_mis = false;
    double* rowpart = nullptr;      // [rowpart_cap][p_pad] per-tile row sums of gam W + I0 left by the last aq_sweep
    int rowpart_cap = 0, rowpart_rows = 0;   // rows allocated / rows the last sweep wrote (0: not valid)
    int rowpart_k_tail = -1;                 // first trait NOT covered by those rows (-1: all are)
    bool rowpart_tried = false;
    // launch attributes of the context's two kernel configurations (0: main, 1: 8-trait tail variant), set on first use
    bool attr_done[2] = {false, false};
    int max_groups[2] = {0, 0};       // tiles one round of the persistent grid processes (SMs, or schedulable clusters)
    int* seg_done = nullptr;          // segmented sweeps: per-tile hand-off counters
    int last_nseg = 1;                // SNP segments per tile of the last sweep launch
    // asynchronous state hand-off (aq_snapshot / aq_snapshot_fetch): device copies of gam / mu, a second staging buffer,
    // a copy stream and the event that orders it after the snapshot
    double *snap_gam = nullptr, *snap_mu = nullptr, *stage2 = nullptr;
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_snap = nullptr;
    bool have_snap = false;
    double* sel_partial = nullptr;  // scratch of the selection kernels: 2 x kSelBlocks partials + 2 results
    std::vector<int32_t> order, order_pad;
    std::vector<double> hbuf;   // pinned-size-agnostic host scratch
    bool have_state = false, have_tables = false;
    int64_t launches = 0;
    float last_ms = 0.f;
};

// Pre-processed predictors (aq_prep_x / aq_prep_geno): the raw input stays on the device until a context has
// materialised the kept, standardised columns from it.
struct aq_prep {
    int device = 0, n = 0, p_raw = 0, p_kept = 0;
    bool geno = false;
    int bytes_per_col = 0;
    double* xd = nullptr;
    uint8_t* gd = nullptr;
    ColStats* st = nullptr;
    int* kept_dev = nullptr;
    cudaStream_t stream = nullptr;
    std::vector<ColStats> hst;
    std::vector<uint8_t> status;    // 0 kept, 1 constant, 2 duplicate of dup_of[j]
    std::vector<int32_t> dup_of, kept;
    int64_t launches = 0;
};

namespace {

int build_gk(aq_ctx* c);   // (missing-response tile path, defined with aq_set_missing)

// Launch configuration of kernel configuration C on the context's stream: clusters of cfg.ncta CTAs for the clustered
// variant and, with `cooperative`, all CTAs resident at the same time.  lc.attrs points into `attr`.
template <class C>
cudaLaunchConfig_t launch_config(const aq_ctx* c, unsigned grid, bool cooperative, cudaLaunchAttribute (&attr)[2]) {
    cudaLaunchConfig_t lc{};
    lc.gridDim = dim3(grid);
    lc.blockDim = dim3(C::kThreads);
    lc.dynamicSmemBytes = C::kSmemBytes;
    lc.stream = c->stream;
    lc.attrs = attr;
    lc.numAttrs = 0;
    if (C::kCl) {
        attr[lc.numAttrs].id = cudaLaunchAttributeClusterDimension;
        attr[lc.numAttrs].val.clusterDim.x = c->cfg.ncta;
        attr[lc.numAttrs].val.clusterDim.y = 1;
        attr[lc.numAttrs].val.clusterDim.z = 1;
        lc.numAttrs++;
    }
    if (cooperative) {
        attr[lc.numAttrs].id = cudaLaunchAttributeCooperative;
        attr[lc.numAttrs].val.cooperative = 1;
        lc.numAttrs++;
    }
    return lc;
}

// Launch attributes of one kernel configuration on this context's device: set once per context (not in function statics:
// the cluster size is a run-time value of the same template instance, and contexts live on several devices / threads).
template <class C>
int prepare_sweep_t(aq_ctx* c, int slot) {
    if (c->attr_done[slot]) return AQ_OK;
    const int ncta = c->cfg.ncta;
    AQ_CUDA(cudaFuncSetAttribute(sweep_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::kSmemBytes));
    c->max_groups[slot] = c->sm_count;
    if (C::kCl) {
        cudaLaunchAttribute attr[2];
        const cudaLaunchConfig_t lc = launch_config<C>(c, c->sm_count / ncta * ncta, false, attr);
        int nc = 0;
        AQ_CUDA(cudaOccupancyMaxActiveClusters(&nc, sweep_kernel<C>, &lc));
        if (nc < 1) return fail(AQ_EUNSUPPORTED, "no thread-block cluster of the required size can be scheduled");
        c->max_groups[slot] = nc;
    } else {
        int per_sm = 0;
        AQ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sweep_kernel<C>, C::kThreads, C::kSmemBytes));
        if (per_sm < 1) return fail(AQ_EUNSUPPORTED, "the sweep kernel does not fit on this device");
    }
    c->attr_done[slot] = true;
    return AQ_OK;
}

// One launch of configuration C (slot 0: the context's main configuration, 1: its 8-trait tail variant) over `ntiles`
// trait tiles starting at trait k_base, each cut into P.nseg SNP segments.
template <class C>
int launch_sweep_t(aq_ctx* c, int slot, SweepParams P, int ntiles, int k_base) {
    int rc = prepare_sweep_t<C>(c, slot);
    if (rc != AQ_OK) return rc;
    if (ntiles <= 0) return AQ_OK;
    P.ntiles = ntiles;
    P.k_base = k_base;
    const long nunits = (long)ntiles * P.nseg;
    // (segmented: CTAs hand trait tiles over to one another inside the launch, so all of them must be resident at once)
    cudaLaunchAttribute attr[2];
    const cudaLaunchConfig_t lc =
        launch_config<C>(c, (unsigned)std::min<long>(nunits, c->max_groups[slot]) * c->cfg.ncta, P.nseg > 1, attr);
    AQ_CUDA(cudaLaunchKernelEx(&lc, sweep_kernel<C>, P));
    AQ_CUDA(cudaGetLastError());
    c->launches++;
    return AQ_OK;
}

// How the trait tiles are spread over the persistent grid.  A grid of G CTAs (clusters) processes G tiles per round and
// a partly filled last round costs as much as a full one.  Two remedies, whichever the block-count model below prefers:
//  (a) segmented sweep: the SNP blocks of every tile are cut into S segments and the
//      (segment, tile) units dealt round-robin, so the last round costs 1 / S of a round; a unit costs its blocks plus
//      ~kSegOverheadBlocks (pipeline fill / drain, residual reload);
//  (b) leftover traits that fit into one round of 8-trait tiles are swept by the MT = 1 variant of the configuration
//      (an 8-trait tile is bound by the serial chain and takes ~0.68 of a full tile).
struct SweepPlan {
    int nseg = 1, seg_len = 0;
    int n_main = 0, n_tail = 0, k_tail = 0;
};
constexpr double kSegOverheadBlocks = 4.0, kTailTileCost = 0.68;

SweepPlan plan_sweep(const aq_ctx* c, int G, int kT, bool has_tail_variant) {
    SweepPlan pl;
    const int ntiles = c->ntiles, nb = c->nb;
    pl.n_main = ntiles;
    pl.seg_len = nb;
    const int rem = ntiles % G;
    double best = (double)((ntiles + G - 1) / G) * (nb + kSegOverheadBlocks);
    if (has_tail_variant && rem != 0 && !c->ov.no_tail) {
        const int k_tail = (ntiles - rem) * kT;
        const int tail_tiles = (c->q - k_tail + 7) / 8;
        if (tail_tiles <= G) {
            const double cost = (ntiles / G + kTailTileCost) * (nb + kSegOverheadBlocks);
            if (cost < best) {
                best = cost;
                pl.n_main = ntiles - rem;
                pl.n_tail = tail_tiles;
                pl.k_tail = k_tail;
            }
        }
    }
    if (ntiles > G && !c->ov.no_seg) {
        const int force = c->ov.nseg;
        for (int S = 2; S <= 64 && nb / S >= 16; ++S) {
            if (force && S != force) continue;
            const int len = (nb + S - 1) / S;
            const int S2 = (nb + len - 1) / len;   // segments actually needed at this length
            const long slots = std::max<long>(S2, ((long)ntiles * S2 + G - 1) / G);
            const double cost = (double)slots * (len + kSegOverheadBlocks);
            if (cost < best * 0.995 || force) {
                best = cost;
                pl = SweepPlan{};
                pl.nseg = S2;
                pl.seg_len = len;
                pl.n_main = ntiles;
            }
        }
    }
    return pl;
}

template <int NT, bool CL>
int launch_sweep_cfg(aq_ctx* c, const SweepParams& P) {
    using Main = CfgOf<NT, CL>;
    using Tail = SweepCfg<1, NT, CL>;
    int rc = prepare_sweep_t<Main>(c, 0);
    if (rc != AQ_OK) return rc;
    const int G = c->max_groups[0];
    const int ntiles = c->ntiles;
    const SweepPlan pl = plan_sweep(c, G, Main::kT, Main::MT > 1);
    SweepParams Pm = P, Pt = P;
    Pm.nseg = pl.nseg;
    Pm.seg_len = pl.seg_len;
    Pt.seg_len = c->nb;
    if (pl.nseg > 1) {
        if (!c->seg_done) AQ_CUDA(cudaMalloc((void**)&c->seg_done, sizeof(int) * (size_t)ntiles));
        AQ_CUDA(cudaMemsetAsync(c->seg_done, 0, sizeof(int) * (size_t)ntiles, c->stream));
        Pm.seg_done = c->seg_done;
    }
    c->last_nseg = pl.nseg;
    c->rowpart_rows = 0;
    if (P.mode == 0 && !CL) {
        // per-tile row sums of gam W + I0 ride along with the sweep (aq_rowsums_zpart reduces them); without the scratch
        // buffer the streaming row-sum kernel is used instead
        if (!c->rowpart && !c->rowpart_tried) {
            c->rowpart_tried = true;
            c->rowpart_cap = ntiles + 1;
            if (cudaMalloc((void**)&c->rowpart, sizeof(double) * (size_t)c->rowpart_cap * c->p_pad) != cudaSuccess) {
                cudaGetLastError();
                c->rowpart = nullptr;
            }
        }
        // (measured: +0.5-1 % on a tensor-bound tile, +2.5 % on the chain-bound 8-trait tail tiles and cluster tiles, whose
        // helper warp sits closer to the serial path; the streaming pass costs 24 B per update, i.e. 2-6 % of a sweep for
        // n <= 1008 and < 1 % beyond.  So: full-size single-CTA tiles only; the tail's traits get one streamed extra row.)
        if (c->rowpart && pl.n_main > 0 && pl.n_main + 1 <= c->rowpart_cap) {
            Pm.rowpart = c->rowpart;
            Pm.rowpart_base = 0;
            c->rowpart_rows = pl.n_main;
            c->rowpart_k_tail = pl.n_tail > 0 ? pl.k_tail : -1;
        }
    }
    AQ_CUDA(cudaEventRecord(c->ev0, c->stream));
    rc = launch_sweep_t<Main>(c, 0, Pm, pl.n_main, 0);
    if (rc == AQ_OK && pl.n_tail > 0) rc = launch_sweep_t<Tail>(c, 1, Pt, pl.n_tail, pl.k_tail);
    if (rc != AQ_OK) {
        c->rowpart_rows = 0;
        return rc;
    }
    AQ_CUDA(cudaEventRecord(c->ev1, c->stream));
    return AQ_OK;
}

// Missing-response variant: one launch, one unit per 16-trait tile (no segments, no 8-trait tail variant).
template <int NT, bool CL>
int launch_sweep_mis_cfg(aq_ctx* c, const SweepParams& P) {
    using Main = CfgMis<NT, CL>;
    int rc = prepare_sweep_t<Main>(c, 0);
    if (rc != AQ_OK) return rc;
    c->last_nseg = 1;
    c->rowpart_rows = 0;
    AQ_CUDA(cudaEventRecord(c->ev0, c->stream));
    rc = launch_sweep_t<Main>(c, 0, P, c->ntiles, 0);
    if (rc != AQ_OK) return rc;
    AQ_CUDA(cudaEventRecord(c->ev1, c->stream));
    return AQ_OK;
}

// ---- the compiled configurations.  A dense entry launches SweepCfg<1, NT, CL> as its 8-trait tail variant.
template <class C>
constexpr SweepKernel entry(int (*launch)(aq_ctx*, const SweepParams&)) {
    return SweepKernel{C::kMis, C::kCl, C::NT, C::kNPad, C::kXS, C::kT, C::kThreads, C::kSmemBytes, C::kTileDoubles, launch};
}
template <int NT, bool CL>
constexpr SweepKernel dense() { return entry<CfgOf<NT, CL>>(launch_sweep_cfg<NT, CL>); }
template <int NT, bool CL>
constexpr SweepKernel mis() { return entry<CfgMis<NT, CL>>(launch_sweep_mis_cfg<NT, CL>); }
constexpr SweepKernel kSweepKernels[] = {
    // dense, one CTA: NT 1-9 (n <= 1008)
    dense<1, false>(), dense<2, false>(), dense<3, false>(), dense<4, false>(), dense<5, false>(), dense<6, false>(),
    dense<7, false>(), dense<8, false>(), dense<9, false>(),
    // dense, clustered: NT 1-8 (the leader also buffers the followers' S tiles: n <= ncta * 896)
    dense<1, true>(), dense<2, true>(), dense<3, true>(), dense<4, true>(), dense<5, true>(), dense<6, true>(),
    dense<7, true>(), dense<8, true>(),
    // missing responses, one CTA: NT 1-7 (n <= 784)
    mis<1, false>(), mis<2, false>(), mis<3, false>(), mis<4, false>(), mis<5, false>(), mis<6, false>(), mis<7, false>(),
    // missing responses, clustered: NT 1-6 (n <= ncta * 672)
    mis<1, true>(), mis<2, true>(), mis<3, true>(), mis<4, true>(), mis<5, true>(), mis<6, true>(),
};

const SweepKernel* find_kernel(bool missing, bool cl, int nt) {
    for (const SweepKernel& k : kSweepKernels)
        if (k.mis == missing && k.cl == cl && k.nt == nt) return &k;
    return nullptr;
}

// Which cluster size?  A cluster of c CTAs holds ceil(n / (112 c)) sample tiles per warp; smaller slices mean wider trait
// tiles (more traits per serial chain step) but more CTAs to synchronise per block and fewer clusters per GPU.  Model,
// fitted to sweeps timed on B200 (gpurun_out/r2_*.log: n = 1500 / 3000 / 5000, 2..8 CTAs):
//   cycles per 8-SNP block  =  256 MT NT (tensor pipe: 4 warps per sub-partition x 4 MT NT DMMAs x 16 cycles)
//                              + 1500 (S reduction -> chain -> -Delta hand-off across the cluster; + 500 for 8 CTAs)
//   clusters resident at once on 148 SMs:  74 / 49 / 33 / 22 / 15  for  2 / 3 / 4 / 6 / 8 CTAs  (5 and 7 place badly)
//   cost  =  rounds of the persistent grid x cycles per block  =  ceil(tiles / clusters) x ...
// and the cheapest candidate wins: the choice depends on q_local through the number of rounds (C3 on one GPU, n = 3000,
// q = 1500: 4 CTAs, 3 rounds of 16-trait tiles; C5 on 8 GPUs, n = 5000, q_local = 2500: 6 CTAs).
int clusters_resident(int ncta, int sm_count) {
    const int on148 = ncta == 1 ? 148 : ncta == 2 ? 74 : ncta == 3 ? 49 : ncta == 4 ? 33 : ncta == 6 ? 22 : 15;
    return std::max(1, (int)((long)on148 * sm_count / 148));
}
// The dense or missing-response configuration for n samples and q traits; `forced` (1..8) fixes the cluster size.  No
// entry (k == NULL) when n is beyond every configuration of the kind.
CfgInfo pick_cfg(int n, int q, int sm_count, bool missing, int forced) {
    double best = 0.0;
    CfgInfo pick;
    for (int c : {1, 2, 3, 4, 6, 8}) {
        if (forced >= 1 && forced <= kMaxCluster && c != forced) continue;
        const SweepKernel* k = find_kernel(missing, c > 1, (n + 112 * c - 1) / (112 * c));
        if (!k) continue;
        const int mt = k->kT / 8, nt = k->nt;
        const long tiles = (q + 8 * mt - 1) / (8 * mt);
        const long rounds = (tiles + clusters_resident(c, sm_count) - 1) / clusters_resident(c, sm_count);
        const double cost = (double)rounds * (256.0 * mt * nt + (c == 1 ? 600.0 : 1500.0) + (c == 8 ? 500.0 : 0.0));
        if (c == 1) { pick = CfgInfo{k, 1}; break; }   // one CTA whenever the samples fit: no cluster traffic at all
        if (!pick.k || cost < best) { best = cost; pick = CfgInfo{k, c}; }
    }
    if (forced >= 2 && forced <= kMaxCluster && !pick.k) {   // a forced size outside the candidate list (5, 7)
        const SweepKernel* k = find_kernel(missing, true, (n + 112 * forced - 1) / (112 * forced));
        if (k) pick = CfgInfo{k, forced};
    }
    return pick;
}

int launch_sweep(aq_ctx* c, int mode, double cc, double log_sig2_inv) {
    SweepParams P;
    P.order = c->order_dev;
    P.xtiles = c->xtiles;
    P.tile_stride = c->cfg.k->tile_doubles;
    P.nb = c->nb;
    P.ntiles = c->ntiles;
    P.k_base = 0;
    P.q = c->q;
    P.q_pad = c->q_pad;
    P.ld_resid = c->ld_resid;
    P.ncta = c->cfg.ncta;
    P.resid = c->resid;
    P.gam = c->gam;
    P.mu = c->mu;
    P.dtab = c->dtab;
    P.wtab = c->wtab;
    P.i0tab = c->i0tab;
    P.tau = c->tvec;
    P.log_tau = c->tvec + c->q_pad;
    P.sig2_beta = c->tvec + 2 * (size_t)c->q_pad;
    P.c = cc;
    P.log_sig2_inv = log_sig2_inv;
    P.cs_gam = c->ovec;
    P.cs_gmu2 = c->ovec + c->q_pad;
    P.cs_b2 = c->ovec + 2 * (size_t)c->q_pad;
    P.rsq = c->ovec + 3 * (size_t)c->q_pad;
    P.cs_z = c->ovec + 4 * (size_t)c->q_pad;
    P.rowpart = nullptr;
    P.rowpart_base = 0;
    P.p_pad = c->p_pad;
    P.mbits = c->mbits;
    P.mwords = c->mwords;
    P.xnsq = c->xnsq;
    P.atab = c->atab;
    P.ltab = c->ltab;
    P.gk = c->gk;
    P.mis_out = c->mis_out;
    if (c->mis_tile) P.rsq = c->mis_out + (size_t)kMisRsq * c->q_pad;
    P.mode = mode;
    P.nseg = 1;
    P.seg_len = c->nb;
    P.seg_done = nullptr;
    P.timing = nullptr;
#ifdef AQ_TIMING
    {
        static long long* tbuf = nullptr;
        if (!tbuf) { cudaMalloc(&tbuf, 16 * sizeof(long long)); }
        long long h[16];
        cudaMemcpy(h, tbuf, sizeof(h), cudaMemcpyDeviceToHost);
        if (mode == 0) { fprintf(stderr, "[timing of previous sweep, cycles/block]"); for (int i = 0; i < 16; ++i) fprintf(stderr, " t%d=%lld", i, h[i] / (c->nb > 0 ? c->nb : 1)); fprintf(stderr, "\n"); }
        cudaMemset(tbuf, 0, 16 * sizeof(long long));
        P.timing = tbuf;
    }
#endif
    return c->cfg.k->launch(c, P);
}

int upload_pxq(aq_ctx* c, const double* host, double* dev) {
    // host: p x q column-major.  Staged in chunks of stage_cols traits, transposed on the device.
    c->rowpart_rows = 0;  // gam or a table changes: the last sweep's row-sum partials no longer describe the state
    for (int k0 = 0; k0 < c->q; k0 += c->stage_cols) {
        const int kc = std::min(c->stage_cols, c->q - k0);
        AQ_CUDA(cudaMemcpyAsync(c->stage, host + (size_t)k0 * c->p, sizeof(double) * (size_t)kc * c->p,
                                cudaMemcpyHostToDevice, c->stream));
        dim3 grid((c->p + 31) / 32, (kc + 31) / 32), block(32, 8);
        cm_to_dev_kernel<<<grid, block, 0, c->stream>>>(c->stage, c->p, kc, k0, c->q_pad, dev);
        AQ_CUDA(cudaGetLastError());
        c->launches++;
    }
    return AQ_OK;
}

int download_pxq(aq_ctx* c, const double* a, const double* b, int op, double* host) {
    for (int k0 = 0; k0 < c->q; k0 += c->stage_cols) {
        const int kc = std::min(c->stage_cols, c->q - k0);
        dim3 grid((c->p + 31) / 32, (kc + 31) / 32), block(32, 8);
        dev_to_cm_kernel<<<grid, block, 0, c->stream>>>(a, b, op, c->p, kc, k0, c->q_pad, c->stage);
        AQ_CUDA(cudaGetLastError());
        c->launches++;
        AQ_CUDA(cudaMemcpyAsync(host + (size_t)k0 * c->p, c->stage, sizeof(double) * (size_t)kc * c->p,
                                cudaMemcpyDeviceToHost, c->stream));
        AQ_CUDA(cudaStreamSynchronize(c->stream));
    }
    return AQ_OK;
}

int fetch_outputs(aq_ctx* c, double* o0, double* o1, double* o2, double* o3, double* o4) {
    double* outs[5] = {o0, o1, o2, o3, o4};
    bool any = false;
    for (double* o : outs) any = any || (o != nullptr);
    if (!any) return AQ_OK;
    c->hbuf.resize(5 * (size_t)c->q_pad);
    AQ_CUDA(cudaMemcpyAsync(c->hbuf.data(), c->ovec, sizeof(double) * 5 * (size_t)c->q_pad, cudaMemcpyDeviceToHost,
                            c->stream));
    AQ_CUDA(cudaStreamSynchronize(c->stream));
    for (int i = 0; i < 5; ++i)
        if (outs[i]) std::memcpy(outs[i], c->hbuf.data() + (size_t)i * c->q_pad, sizeof(double) * c->q);
    return AQ_OK;
}

int retile(aq_ctx* c) {
    c->order_pad.assign(c->p_pad, -1);  // padding slots of the last block carry -1, as in the tile images
    std::copy(c->order.begin(), c->order.end(), c->order_pad.begin());
    AQ_CUDA(cudaMemcpyAsync(c->order_dev, c->order_pad.data(), sizeof(int32_t) * c->p_pad, cudaMemcpyHostToDevice, c->stream));
    build_tiles_kernel<<<dim3(c->nb, c->cfg.ncta), 256, 0, c->stream>>>(c->xraw, c->order_dev, c->n, c->p, c->cfg.k->xs,
                                                                         c->cfg.k->n_pad, c->cfg.k->tile_doubles, c->xtiles);
    AQ_CUDA(cudaGetLastError());
    gram_band_kernel<<<c->nb, 128, 0, c->stream>>>(c->xtiles, c->cfg.k->n_pad, c->cfg.ncta, c->cfg.k->xs, c->cfg.k->tile_doubles);
    AQ_CUDA(cudaGetLastError());
    c->launches += 2;
    return AQ_OK;
}

}  // namespace

namespace aq {

int internal_load_state(aq_ctx* c, const double* gam_vb, const double* mu_beta_vb) {
    if (!c || !gam_vb || !mu_beta_vb) return fail(AQ_EINVAL, "internal_load_state: NULL argument");
    AQ_CUDA(cudaSetDevice(c->device));
    int rc = upload_pxq(c, gam_vb, c->gam);
    if (rc != AQ_OK) return rc;
    rc = upload_pxq(c, mu_beta_vb, c->mu);
    if (rc != AQ_OK) return rc;
    AQ_CUDA(cudaMemcpyAsync(c->resid, c->ymat, sizeof(double) * (size_t)c->q_pad * c->ld_resid, cudaMemcpyDeviceToDevice,
                            c->stream));
    AQ_CUDA(cudaStreamSynchronize(c->stream));
    c->have_state = true;
    return AQ_OK;
}

int internal_load_dtab(aq_ctx* c, const double* d_host) {
    if (!c || !d_host) return fail(AQ_EINVAL, "internal_load_dtab: NULL argument");
    AQ_CUDA(cudaSetDevice(c->device));
    int rc = upload_pxq(c, d_host, c->dtab);
    if (rc != AQ_OK) return rc;
    const size_t pq = (size_t)c->p_pad * c->q_pad;
    AQ_CUDA(cudaMemsetAsync(c->wtab, 0, sizeof(double) * pq, c->stream));
    AQ_CUDA(cudaMemsetAsync(c->i0tab, 0, sizeof(double) * pq, c->stream));
    AQ_CUDA(cudaStreamSynchronize(c->stream));
    c->have_tables = true;
    return AQ_OK;
}

int internal_load_sig2(aq_ctx* c, const double* s2_host) {
    if (!c || !s2_host) return fail(AQ_EINVAL, "internal_load_sig2: NULL argument");
    AQ_CUDA(cudaSetDevice(c->device));
    if (!c->sig2tab) AQ_CUDA(cudaMalloc((void**)&c->sig2tab, sizeof(double) * (size_t)c->p_pad * c->q_pad));
    AQ_CUDA(cudaMemsetAsync(c->sig2tab, 0, sizeof(double) * (size_t)c->p_pad * c->q_pad, c->stream));
    int rc = upload_pxq(c, s2_host, c->sig2tab);
    if (rc != AQ_OK) return rc;
    AQ_CUDA(cudaStreamSynchronize(c->stream));
    return AQ_OK;
}

int internal_fail(int code, const char* msg) { return fail(code, msg); }

}  // namespace aq

extern "C" {

const char* aq_last_error(void) { return g_err.c_str(); }
int aq_version(void) { return 100; }

int aq_device_info(int device, int* sm_count, int64_t* free_bytes, int64_t* total_bytes) {
    int ndev = 0;
    AQ_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(AQ_EINVAL, "device index out of range");
    AQ_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    AQ_CUDA(cudaGetDeviceProperties(&prop, device));
    size_t fr = 0, tot = 0;
    AQ_CUDA(cudaMemGetInfo(&fr, &tot));
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (free_bytes) *free_bytes = (int64_t)fr;
    if (total_bytes) *total_bytes = (int64_t)tot;
    return AQ_OK;
}

int aq_destroy(aq_ctx* c) {
    if (!c) return AQ_OK;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    double* bufs[] = {c->xraw, c->xtiles, c->ymat, c->resid, c->gam, c->mu, c->dtab, c->wtab, c->i0tab, c->tvec,
                      c->ovec, c->theta, c->zeta, c->rowsum, c->partials, c->scalar, c->stage};
    for (double* b : bufs)
        if (b) cudaFree(b);
    if (c->order_dev) cudaFree(c->order_dev);
    if (c->seg_done) cudaFree(c->seg_done);
    if (c->mask) cudaFree(c->mask);
    if (c->mbits) cudaFree(c->mbits);
    if (c->mis_off_dev) cudaFree(c->mis_off_dev);
    if (c->mis_idx_dev) cudaFree(c->mis_idx_dev);
    for (double* b : {c->gk, c->atab, c->ltab})
        if (b) cudaFree(b);
    if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
    for (double* b : {c->sig2tab, c->xnsq, c->n_obs, c->mis_out, c->sel_partial, c->rowpart, c->snap_gam, c->snap_mu, c->stage2})
        if (b) cudaFree(b);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    for (cudaEvent_t e : {c->evr0, c->evr1, c->evt0, c->evt1})
        if (e) cudaEventDestroy(e);
    if (c->ev_snap) cudaEventDestroy(c->ev_snap);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return AQ_OK;
}

}  // extern "C"

namespace {
// X != NULL: standardised predictors from the host (aq_create).  prep != NULL: the kept columns are standardised on the
// device from the raw input, Y is centred over its observed entries there and n_obs (may be NULL) receives their counts.
int create_impl(aq_ctx** out, int device, int n, int p, int q_local, const double* X, const aq_prep* prep, const double* Y,
                double* n_obs) {
    if (n < 2 || p < 1 || q_local < 1) return fail(AQ_EINVAL, "aq_create: need n >= 2, p >= 1, q >= 1");
    int sm = 0;
    int rc = aq_device_info(device, &sm, nullptr, nullptr);
    if (rc != AQ_OK) return rc;
    const DevOverrides ov = read_overrides();
    const CfgInfo cfg = pick_cfg(n, q_local, sm, false, ov.force_cluster);
    if (!cfg.k)
        return fail(AQ_EUNSUPPORTED, "aq_create: n > 7168 is beyond the 8-CTA sample-split cluster kernel");
    aq_ctx* c = new aq_ctx();
    c->device = device;
    c->n = n;
    c->p = p;
    c->q = q_local;
    c->cfg = cfg;
    c->ov = ov;
    c->sm_count = sm;
    c->p_pad = (p + kBlk - 1) / kBlk * kBlk;
    // leading dimension of the p x q arrays: a multiple of every tile width (16 / 24 / 32 traits, 96 = their lcm), so that a
    // context can change its kernel configuration (missing responses use 16-trait tiles) without re-laying them out
    c->q_pad = (q_local + 95) / 96 * 96;
    c->nb = c->p_pad / kBlk;
    c->ld_resid = cfg.k->n_pad * cfg.ncta;
    c->ntiles = (q_local + cfg.k->kT - 1) / cfg.k->kT;
    const size_t pq = (size_t)c->p_pad * c->q_pad;
    c->stage_cols = (int)std::max<size_t>(1, std::min<size_t>((size_t)q_local, ((size_t)256 << 20) / (sizeof(double) * (size_t)p)));
    c->n_partials = (size_t)((c->q + 255) / 256) * tab_row_blocks(c->p);   // one per CTA of the table pass
#define AQ_ALLOC(ptr, count)                                                              \
    do {                                                                                  \
        cudaError_t e_ = cudaMalloc((void**)&(ptr), sizeof(*(ptr)) * (size_t)(count));    \
        if (e_ != cudaSuccess) {                                                          \
            cudaGetLastError();                                                           \
            aq_destroy(c);                                                                \
            return fail(AQ_ENOMEM, std::string("cudaMalloc ") + #ptr + ": " + cudaGetErrorString(e_)); \
        }                                                                                 \
    } while (0)
    AQ_ALLOC(c->xraw, (size_t)n * p);
    AQ_ALLOC(c->xtiles, (size_t)c->nb * cfg.ncta * cfg.k->tile_doubles);
    AQ_ALLOC(c->ymat, (size_t)c->q_pad * c->ld_resid);
    AQ_ALLOC(c->resid, (size_t)c->q_pad * c->ld_resid);
    AQ_ALLOC(c->gam, pq);
    AQ_ALLOC(c->mu, pq);
    AQ_ALLOC(c->dtab, pq);
    AQ_ALLOC(c->wtab, pq);
    AQ_ALLOC(c->i0tab, pq);
    AQ_ALLOC(c->tvec, 3 * (size_t)c->q_pad);
    AQ_ALLOC(c->ovec, 5 * (size_t)c->q_pad);
    AQ_ALLOC(c->theta, c->p_pad);
    AQ_ALLOC(c->zeta, c->q_pad);
    AQ_ALLOC(c->rowsum, c->p_pad);
    AQ_ALLOC(c->partials, c->n_partials);
    AQ_ALLOC(c->scalar, 8);
    AQ_ALLOC(c->stage, (size_t)c->stage_cols * p);
    AQ_ALLOC(c->order_dev, c->p_pad);
#undef AQ_ALLOC
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev1);
    if (e == cudaSuccess) e = cudaEventCreate(&c->evr0);
    if (e == cudaSuccess) e = cudaEventCreate(&c->evr1);
    if (e == cudaSuccess) e = cudaEventCreate(&c->evt0);
    if (e == cudaSuccess) e = cudaEventCreate(&c->evt1);
    if (e == cudaSuccess) e = cudaMemsetAsync(c->ymat, 0, sizeof(double) * (size_t)c->q_pad * c->ld_resid, c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(c->gam, 0, sizeof(double) * pq, c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(c->mu, 0, sizeof(double) * pq, c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(c->dtab, 0, sizeof(double) * pq, c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(c->wtab, 0, sizeof(double) * pq, c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(c->i0tab, 0, sizeof(double) * pq, c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(c->ovec, 0, sizeof(double) * 5 * (size_t)c->q_pad, c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(c->rowsum, 0, sizeof(double) * c->p_pad, c->stream);
    if (e == cudaSuccess && X) e = cudaMemcpyAsync(c->xraw, X, sizeof(double) * (size_t)n * p, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess && prep) {
        if (prep->geno)
            materialise_kernel<<<p, 256, 0, c->stream>>>(SrcGeno{prep->gd, prep->bytes_per_col}, n, prep->st, prep->kept_dev, p, c->xraw);
        else
            materialise_kernel<<<p, 256, 0, c->stream>>>(SrcDouble{prep->xd, n}, n, prep->st, prep->kept_dev, p, c->xraw);
        e = cudaGetLastError();
        c->launches++;
    }
    // Y: n x q column-major -> [q_pad][n_pad] rows (same orientation, padded leading dimension)
    if (e == cudaSuccess)
        e = cudaMemcpy2DAsync(c->ymat, sizeof(double) * c->ld_resid, Y, sizeof(double) * n, sizeof(double) * n, q_local,
                              cudaMemcpyHostToDevice, c->stream);
    std::vector<int> n_mis;
    if (e == cudaSuccess && prep) {
        // scale(Y, center = TRUE, scale = FALSE) (R/prepare_atlasqtl.R:83); the counts go through the (still unused) order buffer
        int* n_mis_dev = c->order_dev;
        if (q_local > c->p_pad) e = cudaMalloc((void**)&n_mis_dev, sizeof(int) * (size_t)q_local);
        if (e == cudaSuccess) {
            center_y_kernel<<<(q_local + 7) / 8, 256, 0, c->stream>>>(c->ymat, n, q_local, c->ld_resid, n_mis_dev);
            e = cudaGetLastError();
            c->launches++;
        }
        n_mis.resize(q_local);
        if (e == cudaSuccess) e = cudaMemcpyAsync(n_mis.data(), n_mis_dev, sizeof(int) * (size_t)q_local, cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (n_mis_dev != c->order_dev) cudaFree(n_mis_dev);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        aq_destroy(c);
        return fail(AQ_ECUDA, std::string("aq_create: ") + cudaGetErrorString(e));
    }
    for (int k = 0; k < (int)n_mis.size(); ++k) {
        if (n_mis[k] >= n) {
            aq_destroy(c);
            return fail(AQ_EINVAL, "aq_create_prepared: a column of Y has no observed value");
        }
        if (n_obs) n_obs[k] = (double)(n - n_mis[k]);
    }
    // benign per-trait constants for padding traits
    fill_kernel<<<64, 256, 0, c->stream>>>(c->tvec, 3 * (size_t)c->q_pad, 1.0);
    c->launches++;
    c->order.resize(p);
    for (int j = 0; j < p; ++j) c->order[j] = j;
    rc = retile(c);
    if (rc == AQ_OK && cudaStreamSynchronize(c->stream) != cudaSuccess) rc = fail(AQ_ECUDA, "aq_create: sync failed");
    if (rc != AQ_OK) {
        aq_destroy(c);
        return rc;
    }
    *out = c;
    return AQ_OK;
}
}  // namespace

extern "C" {

int aq_create(aq_ctx** out, int device, int n, int p, int q_local, const double* X, const double* Y) {
    if (!out || !X || !Y) return fail(AQ_EINVAL, "aq_create: NULL argument");
    return create_impl(out, device, n, p, q_local, X, nullptr, Y, nullptr);
}

int aq_create_prepared(aq_ctx** out, const aq_prep* prep, int q_local, const double* Y_raw, double* n_obs) {
    if (!out || !prep || !Y_raw) return fail(AQ_EINVAL, "aq_create_prepared: NULL argument");
    if (prep->p_kept < 1) return fail(AQ_EINVAL, "There must be at least 1 non-constant candidate predictor stored in X.");
    return create_impl(out, prep->device, prep->n, prep->p_kept, q_local, nullptr, prep, Y_raw, n_obs);
}

int aq_get_x(aq_ctx* c, double* X) {
    if (!c || !X) return fail(AQ_EINVAL, "aq_get_x: NULL argument");
    if (!c->xraw) return fail(AQ_ESTATE, "aq_get_x after aq_release_x");
    AQ_CUDA(cudaSetDevice(c->device));
    AQ_CUDA(cudaMemcpyAsync(X, c->xraw, sizeof(double) * (size_t)c->n * c->p, cudaMemcpyDeviceToHost, c->stream));
    AQ_CUDA(cudaStreamSynchronize(c->stream));
    return AQ_OK;
}

int aq_release_x(aq_ctx* c) {
    if (!c) return fail(AQ_EINVAL, "NULL context");
    if (c->has_mis) return fail(AQ_ESTATE, "aq_release_x: the missing-response kernel reads the untiled X");
    AQ_CUDA(cudaSetDevice(c->device));
    AQ_CUDA(cudaStreamSynchronize(c->stream));
    if (c->xraw) AQ_CUDA(cudaFree(c->xraw));
    c->xraw = nullptr;
    return AQ_OK;
}

int aq_get_y(aq_ctx* c, double* Y) {
    if (!c || !Y) return fail(AQ_EINVAL, "aq_get_y: NULL argument");
    AQ_CUDA(cudaSetDevice(c->device));
    AQ_CUDA(cudaMemcpy2DAsync(Y, sizeof(double) * c->n, c->ymat, sizeof(double) * c->ld_resid, sizeof(double) * c->n, c->q,
                              cudaMemcpyDeviceToHost, c->stream));
    AQ_CUDA(cudaStreamSynchronize(c->stream));
    return AQ_OK;
}

// ---------------------------------------------------------------- pre-processing of the predictors
int aq_prep_destroy(aq_prep* P) {
    if (!P) return AQ_OK;
    cudaSetDevice(P->device);
    if (P->stream) cudaStreamSynchronize(P->stream);
    if (P->xd) cudaFree(P->xd);
    if (P->gd) cudaFree(P->gd);
    if (P->st) cudaFree(P->st);
    if (P->kept_dev) cudaFree(P->kept_dev);
    if (P->stream) cudaStreamDestroy(P->stream);
    delete P;
    return AQ_OK;
}

}  // extern "C"

namespace {
template <class Src>
int prep_verify(aq_prep* P, Src src, const std::vector<int32_t>& pairs, std::vector<int>& differs) {
    const int npairs = (int)(pairs.size() / 2);
    differs.assign(npairs, 0);
    if (!npairs) return AQ_OK;
    int *pairs_dev = nullptr, *diff_dev = nullptr;
    AQ_CUDA(cudaMalloc((void**)&pairs_dev, sizeof(int) * pairs.size()));
    cudaError_t e = cudaMalloc((void**)&diff_dev, sizeof(int) * (size_t)npairs);
    if (e == cudaSuccess) e = cudaMemcpyAsync(pairs_dev, pairs.data(), sizeof(int) * pairs.size(), cudaMemcpyHostToDevice, P->stream);
    if (e == cudaSuccess) {
        verify_dups_kernel<<<(npairs + 7) / 8, 256, 0, P->stream>>>(src, P->n, P->st, pairs_dev, npairs, diff_dev);
        e = cudaGetLastError();
        P->launches++;
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(differs.data(), diff_dev, sizeof(int) * (size_t)npairs, cudaMemcpyDeviceToHost, P->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(P->stream);
    cudaFree(pairs_dev);
    if (diff_dev) cudaFree(diff_dev);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(AQ_ECUDA, std::string("aq_prep: ") + cudaGetErrorString(e));
    }
    return AQ_OK;
}

// moments + fingerprints are on the device: classify the columns (constant / duplicate / kept)
template <class Src>
int prep_classify(aq_prep* P, Src src) {
    const int p = P->p_raw;
    P->hst.resize(p);
    AQ_CUDA(cudaMemcpyAsync(P->hst.data(), P->st, sizeof(ColStats) * (size_t)p, cudaMemcpyDeviceToHost, P->stream));
    AQ_CUDA(cudaStreamSynchronize(P->stream));
    P->status.assign(p, 0);
    P->dup_of.assign(p, -1);
    std::vector<int32_t> cand;
    cand.reserve(p);
    for (int j = 0; j < p; ++j) {
        if (P->hst[j].bad)
            return fail(AQ_EINVAL, P->geno ? "aq_prep_geno: invalid genotype call (code 3) in column " + std::to_string(j)
                                           : "aq_prep_x: X must not contain missing / non-finite values (column " + std::to_string(j) + ")");
        if (!(P->hst[j].sd > 0.0)) P->status[j] = 1;   // scale() made it NaN: rm_constant_ (R/utils.R:278)
        else cand.push_back(j);
    }
    // duplicated(mat, MARGIN = 2) (R/utils.R:305): equal fingerprints are suspects, the first of a group is its representative
    std::sort(cand.begin(), cand.end(), [&](int a, int b) {
        const ColStats &x = P->hst[a], &y = P->hst[b];
        if (x.h1 != y.h1) return x.h1 < y.h1;
        if (x.h2 != y.h2) return x.h2 < y.h2;
        return a < b;
    });
    std::vector<std::vector<int32_t>> groups;   // each: representative first, then its suspects (ascending)
    for (size_t i = 0; i < cand.size();) {
        size_t e = i + 1;
        while (e < cand.size() && P->hst[cand[e]].h1 == P->hst[cand[i]].h1 && P->hst[cand[e]].h2 == P->hst[cand[i]].h2) ++e;
        if (e - i > 1) groups.emplace_back(cand.begin() + i, cand.begin() + e);
        i = e;
    }
    while (!groups.empty()) {
        std::vector<int32_t> pairs;
        for (const auto& g : groups)
            for (size_t i = 1; i < g.size(); ++i) {
                pairs.push_back(g[i]);
                pairs.push_back(g[0]);
            }
        std::vector<int> differs;
        int rc = prep_verify(P, src, pairs, differs);
        if (rc != AQ_OK) return rc;
        // a suspect that differs value by value (fingerprint collision) starts / joins a new group, verified next round
        std::vector<std::vector<int32_t>> next;
        size_t m = 0;
        for (const auto& g : groups) {
            std::vector<int32_t> rest;
            for (size_t i = 1; i < g.size(); ++i, ++m) {
                if (differs[m]) rest.push_back(g[i]);
                else {
                    P->status[g[i]] = 2;
                    P->dup_of[g[i]] = g[0];
                }
            }
            if (rest.size() > 1) next.push_back(std::move(rest));
        }
        groups.swap(next);
    }
    P->kept.clear();
    for (int j = 0; j < p; ++j)
        if (P->status[j] == 0) P->kept.push_back(j);
    P->p_kept = (int)P->kept.size();
    if (P->p_kept) {
        AQ_CUDA(cudaMalloc((void**)&P->kept_dev, sizeof(int) * (size_t)P->p_kept));
        AQ_CUDA(cudaMemcpyAsync(P->kept_dev, P->kept.data(), sizeof(int) * (size_t)P->p_kept, cudaMemcpyHostToDevice, P->stream));
        AQ_CUDA(cudaStreamSynchronize(P->stream));
    }
    return AQ_OK;
}

int prep_impl(aq_prep** out, int device, int n, int p_raw, const double* X_raw, const uint8_t* geno, int64_t bytes_per_col,
              int* p_kept) {
    if (!out || (!X_raw && !geno)) return fail(AQ_EINVAL, "aq_prep: NULL argument");
    if (n < 2 || p_raw < 1) return fail(AQ_EINVAL, "aq_prep: need n >= 2, p >= 1");
    if (geno && (bytes_per_col < (n + 3) / 4 || bytes_per_col > (int64_t)1 << 30))
        return fail(AQ_EINVAL, "aq_prep_geno: bytes_per_col must be at least ceil(n / 4)");
    int rc = aq_device_info(device, nullptr, nullptr, nullptr);
    if (rc != AQ_OK) return rc;
    aq_prep* P = new aq_prep();
    P->device = device;
    P->n = n;
    P->p_raw = p_raw;
    P->geno = geno != nullptr;
    P->bytes_per_col = (int)bytes_per_col;
    cudaError_t e = cudaStreamCreateWithFlags(&P->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMalloc((void**)&P->st, sizeof(ColStats) * (size_t)p_raw);
    if (e == cudaSuccess) {
        if (geno) {
            e = cudaMalloc((void**)&P->gd, (size_t)bytes_per_col * p_raw);
            if (e == cudaSuccess) e = cudaMemcpyAsync(P->gd, geno, (size_t)bytes_per_col * p_raw, cudaMemcpyHostToDevice, P->stream);
        } else {
            e = cudaMalloc((void**)&P->xd, sizeof(double) * (size_t)n * p_raw);
            if (e == cudaSuccess) e = cudaMemcpyAsync(P->xd, X_raw, sizeof(double) * (size_t)n * p_raw, cudaMemcpyHostToDevice, P->stream);
        }
    }
    if (e == cudaSuccess) {
        if (geno) col_stats_geno_kernel<<<(p_raw + 7) / 8, 256, 0, P->stream>>>(SrcGeno{P->gd, P->bytes_per_col}, n, p_raw, P->st);
        else col_stats_double_kernel<<<(p_raw + 7) / 8, 256, 0, P->stream>>>(SrcDouble{P->xd, n}, p_raw, P->st);
        e = cudaGetLastError();
        P->launches++;
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        aq_prep_destroy(P);
        return fail(e == cudaErrorMemoryAllocation ? AQ_ENOMEM : AQ_ECUDA, std::string("aq_prep: ") + cudaGetErrorString(e));
    }
    rc = geno ? prep_classify(P, SrcGeno{P->gd, P->bytes_per_col}) : prep_classify(P, SrcDouble{P->xd, n});
    if (rc != AQ_OK) {
        aq_prep_destroy(P);
        return rc;
    }
    if (p_kept) *p_kept = P->p_kept;
    *out = P;
    return AQ_OK;
}
}  // namespace

extern "C" {

int aq_prep_x(aq_prep** out, int device, int n, int p_raw, const double* X_raw, int* p_kept) {
    if (!X_raw) return fail(AQ_EINVAL, "aq_prep_x: NULL argument");
    return prep_impl(out, device, n, p_raw, X_raw, nullptr, 0, p_kept);
}

int aq_prep_geno(aq_prep** out, int device, int n, int p_raw, const uint8_t* geno, int64_t bytes_per_col, int* p_kept) {
    if (!geno) return fail(AQ_EINVAL, "aq_prep_geno: NULL argument");
    return prep_impl(out, device, n, p_raw, nullptr, geno, bytes_per_col, p_kept);
}

int aq_prep_result(const aq_prep* P, uint8_t* status, int32_t* dup_of, double* mean, double* sd) {
    if (!P) return fail(AQ_EINVAL, "aq_prep_result: NULL argument");
    for (int j = 0; j < P->p_raw; ++j) {
        if (status) status[j] = P->status[j];
        if (dup_of) dup_of[j] = P->dup_of[j];
        if (mean) mean[j] = P->hst[j].mean;
        if (sd) sd[j] = P->hst[j].sd;
    }
    return AQ_OK;
}

int aq_prep_dims(const aq_prep* P, int* n, int* p_raw, int* p_kept) {
    if (!P) return fail(AQ_EINVAL, "aq_prep_dims: NULL argument");
    if (n) *n = P->n;
    if (p_raw) *p_raw = P->p_raw;
    if (p_kept) *p_kept = P->p_kept;
    return AQ_OK;
}

int64_t aq_prep_launch_count(const aq_prep* P) { return P ? P->launches : 0; }

int aq_dims(const aq_ctx* c, int* n, int* p, int* q_local, int* p_pad, int* q_pad) {
    if (!c) return fail(AQ_EINVAL, "NULL context");
    if (n) *n = c->n;
    if (p) *p = c->p;
    if (q_local) *q_local = c->q;
    if (p_pad) *p_pad = c->p_pad;
    if (q_pad) *q_pad = c->q_pad;
    return AQ_OK;
}

int aq_set_order(aq_ctx* c, const int32_t* shuffled_ind) {
    if (!c) return fail(AQ_EINVAL, "NULL context");
    AQ_CUDA(cudaSetDevice(c->device));
    std::vector<int32_t> ord(c->p);
    if (shuffled_ind) {
        std::vector<char> seen(c->p, 0);
        for (int b = 0; b < c->p; ++b) {
            const int32_t j = shuffled_ind[b];
            if (j < 0 || j >= c->p || seen[j]) return fail(AQ_EINVAL, "aq_set_order: shuffled_ind is not a permutation of 0..p-1");
            seen[j] = 1;
            ord[b] = j;
        }
    } else {
        for (int j = 0; j < c->p; ++j) ord[j] = j;
    }
    if (ord == c->order) return AQ_OK;
    if (!c->xraw) return fail(AQ_ESTATE, "aq_set_order: a new order needs the untiled X, which aq_release_x freed");
    c->order.swap(ord);
    int rc = retile(c);
    if (rc == AQ_OK && c->mis_tile) rc = build_gk(c);   // the per-trait Gram band follows the blocks of the order
    if (rc != AQ_OK) return rc;
    AQ_CUDA(cudaStreamSynchronize(c->stream));
    return AQ_OK;
}

int aq_set_state(aq_ctx* c, const double* gam_vb, const double* mu_beta_vb, double* colsum_gam, double* colsum_gam_mu2,
                 double* colsum_beta2, double* resid_sq) {
    if (!c || !gam_vb || !mu_beta_vb) return fail(AQ_EINVAL, "aq_set_state: NULL argument");
    if (c->has_mis) return fail(AQ_ESTATE, "aq_set_state: this context has missing responses, use aq_set_state_mis");
    AQ_CUDA(cudaSetDevice(c->device));
    int rc = upload_pxq(c, gam_vb, c->gam);
    if (rc != AQ_OK) return rc;
    rc = upload_pxq(c, mu_beta_vb, c->mu);
    if (rc != AQ_OK) return rc;
    AQ_CUDA(cudaMemcpyAsync(c->resid, c->ymat, sizeof(double) * (size_t)c->q_pad * c->ld_resid, cudaMemcpyDeviceToDevice,
                            c->stream));
    rc = launch_sweep(c, /*mode=*/1, 1.0, 0.0);
    if (rc != AQ_OK) return rc;
    c->have_state = true;
    rc = fetch_outputs(c, colsum_gam, colsum_gam_mu2, colsum_beta2, resid_sq, nullptr);
    if (rc != AQ_OK) return rc;
    AQ_CUDA(cudaStreamSynchronize(c->stream));
    return AQ_OK;
}

int aq_get_state(aq_ctx* c, double* gam_vb, double* mu_beta_vb, double* beta_vb) {
    if (!c) return fail(AQ_EINVAL, "NULL context");
    if (!c->have_state) return fail(AQ_ESTATE, "aq_get_state before aq_set_state");
    AQ_CUDA(cudaSetDevice(c->device));
    int rc = AQ_OK;
    if (gam_vb && (rc = download_pxq(c, c->gam, nullptr, 0, gam_vb)) != AQ_OK) return rc;
    if (mu_beta_vb && (rc = download_pxq(c, c->mu, nullptr, 0, mu_beta_vb)) != AQ_OK) return rc;
    if (beta_vb && (rc = download_pxq(c, c->gam, c->mu, 1, beta_vb)) != AQ_OK) return rc;
    return AQ_OK;
}

int aq_snapshot(aq_ctx* c) {
    if (!c) return fail(AQ_EINVAL, "NULL context");
    if (!c->have_state) return fail(AQ_ESTATE, "aq_snapshot before aq_set_state");
    AQ_CUDA(cudaSetDevice(c->device));
    const size_t pq = (size_t)c->p_pad * c->q_pad;
    // (each resource on its own: a call that failed half-way leaves nothing to leak or to allocate twice)
    if (!c->snap_gam) AQ_CUDA(cudaMalloc((void**)&c->snap_gam, sizeof(double) * pq));
    if (!c->snap_mu) AQ_CUDA(cudaMalloc((void**)&c->snap_mu, sizeof(double) * pq));
    if (!c->stage2) AQ_CUDA(cudaMalloc((void**)&c->stage2, sizeof(double) * (size_t)c->stage_cols * c->p));
    if (!c->ev_snap) AQ_CUDA(cudaEventCreateWithFlags(&c->ev_snap, cudaEventDisableTiming));
    if (!c->copy_stream) AQ_CUDA(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    AQ_CUDA(cudaStreamSynchronize(c->copy_stream));   // a fetch of the previous snapshot has finished reading it
    AQ_CUDA(cudaMemcpyAsync(c->snap_gam, c->gam, sizeof(double) * pq, cudaMemcpyDeviceToDevice, c->stream));
    AQ_CUDA(cudaMemcpyAsync(c->snap_mu, c->mu, sizeof(double) * pq, cudaMemcpyDeviceToDevice, c->stream));
    AQ_CUDA(cudaEventRecord(c->ev_snap, c->stream));
    c->have_snap = true;
    return AQ_OK;
}

int aq_snapshot_fetch(aq_ctx* c, double* gam_vb, double* mu_beta_vb, double* beta_vb) {
    if (!c) return fail(AQ_EINVAL, "NULL context");
    if (!c->have_snap) return fail(AQ_ESTATE, "aq_snapshot_fetch before aq_snapshot");
    AQ_CUDA(cudaSetDevice(c->device));
    AQ_CUDA(cudaStreamWaitEvent(c->copy_stream, c->ev_snap, 0));
    // touches the snapshot, the second staging buffer and the copy stream only: may run on another host thread while
    // the owner of the context keeps sweeping
    double* outs[3] = {gam_vb, mu_beta_vb, beta_vb};
    for (int which = 0; which < 3; ++which) {
        if (!outs[which]) continue;
        const double* a = which == 1 ? c->snap_mu : c->snap_gam;
        const double* b = which == 2 ? c->snap_mu : nullptr;
        for (int k0 = 0; k0 < c->q; k0 += c->stage_cols) {
            const int kc = std::min(c->stage_cols, c->q - k0);
            dim3 grid((c->p + 31) / 32, (kc + 31) / 32), block(32, 8);
            dev_to_cm_kernel<<<grid, block, 0, c->copy_stream>>>(a, b, which == 2 ? 1 : 0, c->p, kc, k0, c->q_pad, c->stage2);
            AQ_CUDA(cudaGetLastError());
            AQ_CUDA(cudaMemcpyAsync(outs[which] + (size_t)k0 * c->p, c->stage2, sizeof(double) * (size_t)kc * c->p,
                                    cudaMemcpyDeviceToHost, c->copy_stream));
            AQ_CUDA(cudaStreamSynchronize(c->copy_stream));
        }
    }
    return AQ_OK;
}

int aq_get_residual(aq_ctx* c, double* resid) {
    if (!c || !resid) return fail(AQ_EINVAL, "NULL argument");
    if (!c->have_state) return fail(AQ_ESTATE, "aq_get_residual before aq_set_state");
    AQ_CUDA(cudaSetDevice(c->device));
    AQ_CUDA(cudaMemcpy2DAsync(resid, sizeof(double) * c->n, c->resid, sizeof(double) * c->ld_resid, sizeof(double) * c->n,
                              c->q, cudaMemcpyDeviceToHost, c->stream));
    AQ_CUDA(cudaStreamSynchronize(c->stream));
    return AQ_OK;
}

int aq_get_tables(aq_ctx* c, double* D, double* W, double* I0) {
    if (!c) return fail(AQ_EINVAL, "NULL context");
    if (!c->have_tables) return fail(AQ_ESTATE, "aq_get_tables before aq_refresh_tables");
    AQ_CUDA(cudaSetDevice(c->device));
    int rc = AQ_OK;
    if (D && (rc = download_pxq(c, c->dtab, nullptr, 0, D)) != AQ_OK) return rc;
    if (W && (rc = download_pxq(c, c->wtab, nullptr, 0, W)) != AQ_OK) return rc;
    if (I0 && (rc = download_pxq(c, c->i0tab, nullptr, 0, I0)) != AQ_OK) return rc;
    return AQ_OK;
}

int aq_refresh_tables(aq_ctx* c, const double* theta_vb, const double* zeta_vb, double c_next, double* elbo_b_part) {
    if (!c || !theta_vb || !zeta_vb) return fail(AQ_EINVAL, "aq_refresh_tables: NULL argument");
    if (!(c_next > 0.0)) return fail(AQ_EINVAL, "aq_refresh_tables: c_next must be positive");
    if (elbo_b_part && !c->have_state) return fail(AQ_ESTATE, "aq_refresh_tables: ELBO part needs a state");
    AQ_CUDA(cudaSetDevice(c->device));
    c->rowpart_rows = 0;  // W / I0 change
    AQ_CUDA(cudaMemcpyAsync(c->theta, theta_vb, sizeof(double) * c->p, cudaMemcpyHostToDevice, c->stream));
    AQ_CUDA(cudaMemcpyAsync(c->zeta, zeta_vb, sizeof(double) * c->q, cudaMemcpyHostToDevice, c->stream));
    const int c_is_one = std::fabs(c_next - 1.0) < 1.5e-8;  // isTRUE(all.equal(c, 1)), R/update_vb.R:219
    const int row_blocks = tab_row_blocks(c->p);
    AQ_CUDA(cudaEventRecord(c->evt0, c->stream));
    for (int rb0 = 0; rb0 < row_blocks; rb0 += kTabMaxGridRows) {   // (one launch for p <= 524,280)
        dim3 grid((c->q + 255) / 256, std::min(row_blocks - rb0, kTabMaxGridRows));
        const int j0 = rb0 * kTabRowsPerBlock;
        const size_t off = (size_t)j0 * c->q_pad;
        tables_kernel<<<grid, 256, 0, c->stream>>>(c->theta + j0, c->zeta, c->p - j0, c->q, c->q_pad,
                                                   c_is_one ? 1.0 : std::sqrt(c_next), c_is_one, c->gam + off, c->dtab + off,
                                                   c->wtab + off, c->i0tab + off, elbo_b_part ? 1 : 0,
                                                   c->partials + (size_t)rb0 * grid.x);
        AQ_CUDA(cudaGetLastError());
        c->launches++;
    }
    if (elbo_b_part) {
        sum_partials_kernel<<<1, 1024, 0, c->stream>>>(c->partials, c->n_partials, c->scalar);
        AQ_CUDA(cudaGetLastError());
        c->launches++;
        AQ_CUDA(cudaMemcpyAsync(elbo_b_part, c->scalar, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    }
    AQ_CUDA(cudaEventRecord(c->evt1, c->stream));
    AQ_CUDA(cudaStreamSynchronize(c->stream));
    AQ_CUDA(cudaEventElapsedTime(&c->last_tables_ms, c->evt0, c->evt1));
    c->have_tables = true;
    return AQ_OK;
}

int aq_sweep(aq_ctx* c, double cc, double log_sig2_inv_vb, const double* tau_vb, const double* log_tau_vb,
             const double* sig2_beta_vb, double* colsum_gam, double* colsum_gam_mu2, double* colsum_beta2,
             double* resid_sq, double* colsum_zpart) {
    if (!c || !tau_vb || !log_tau_vb || !sig2_beta_vb) return fail(AQ_EINVAL, "aq_sweep: NULL argument");
    if (c->has_mis) return fail(AQ_ESTATE, "aq_sweep: this context has missing responses, use aq_sweep_mis");
    if (!c->have_state) return fail(AQ_ESTATE, "aq_sweep before aq_set_state");
    if (!c->have_tables) return fail(AQ_ESTATE, "aq_sweep before aq_refresh_tables");
    if (!(cc > 0.0)) return fail(AQ_EINVAL, "aq_sweep: c must be positive");
    AQ_CUDA(cudaSetDevice(c->device));
    AQ_CUDA(cudaMemcpyAsync(c->tvec, tau_vb, sizeof(double) * c->q, cudaMemcpyHostToDevice, c->stream));
    AQ_CUDA(cudaMemcpyAsync(c->tvec + c->q_pad, log_tau_vb, sizeof(double) * c->q, cudaMemcpyHostToDevice, c->stream));
    AQ_CUDA(cudaMemcpyAsync(c->tvec + 2 * (size_t)c->q_pad, sig2_beta_vb, sizeof(double) * c->q, cudaMemcpyHostToDevice,
                            c->stream));
    int rc = launch_sweep(c, /*mode=*/0, cc, log_sig2_inv_vb);
    if (rc != AQ_OK) return rc;
    rc = fetch_outputs(c, colsum_gam, colsum_gam_mu2, colsum_beta2, resid_sq, colsum_zpart);
    if (rc != AQ_OK) return rc;
    AQ_CUDA(cudaStreamSynchronize(c->stream));
    AQ_CUDA(cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1));
    return AQ_OK;
}

int aq_rowsums_zpart_dev(aq_ctx* c, double** rowsum_zpart_dev) {
    if (!c || !rowsum_zpart_dev) return fail(AQ_EINVAL, "NULL argument");
    if (!c->have_state || !c->have_tables) return fail(AQ_ESTATE, "aq_rowsums_zpart before state/tables");
    AQ_CUDA(cudaSetDevice(c->device));
    AQ_CUDA(cudaEventRecord(c->evr0, c->stream));
    if (c->rowpart_rows > 0) {  // the last sweep left per-tile partial sums: no second pass over the p x q arrays
        int rows = c->rowpart_rows;
        if (c->rowpart_k_tail >= 0) {  // traits swept by the 8-trait tail launch: streamed into one more row
            const int kt = c->rowpart_k_tail;
            rowsums_kernel<<<(c->p + 7) / 8, 256, 0, c->stream>>>(c->gam + kt, c->wtab + kt, c->i0tab + kt, c->p, c->q - kt,
                                                                  c->q_pad, c->rowpart + (size_t)rows * c->p_pad);
            AQ_CUDA(cudaGetLastError());
            c->launches++;
            ++rows;
        }
        rowpart_reduce_kernel<<<(c->p + 31) / 32, dim3(32, 8), 0, c->stream>>>(c->rowpart, rows, c->p, c->p_pad, c->rowsum);
    } else
        rowsums_kernel<<<(c->p + 7) / 8, 256, 0, c->stream>>>(c->gam, c->wtab, c->i0tab, c->p, c->q, c->q_pad, c->rowsum);
    AQ_CUDA(cudaGetLastError());
    c->launches++;
    AQ_CUDA(cudaEventRecord(c->evr1, c->stream));
    AQ_CUDA(cudaStreamSynchronize(c->stream));
    AQ_CUDA(cudaEventElapsedTime(&c->last_rows_ms, c->evr0, c->evr1));
    *rowsum_zpart_dev = c->rowsum;
    return AQ_OK;
}

int aq_rowsums_zpart(aq_ctx* c, double* rowsum_zpart) {
    if (!rowsum_zpart) return fail(AQ_EINVAL, "NULL argument");
    double* dev = nullptr;
    int rc = aq_rowsums_zpart_dev(c, &dev);
    if (rc != AQ_OK) return rc;
    AQ_CUDA(cudaMemcpy(rowsum_zpart, dev, sizeof(double) * c->p, cudaMemcpyDeviceToHost));
    return AQ_OK;
}

// ---------------------------------------------------------------- missing responses (coreDualMisLoop)
namespace {
int launch_mis(aq_ctx* c, int mode, double cc, double log_sig2_inv, double sig2_inv) {
    MisParams P;
    P.xraw = c->xraw;
    P.order = c->order_dev;
    P.mask = c->mask;
    P.n = c->n;
    P.p_pad = c->p_pad;
    P.q = c->q;
    P.q_pad = c->q_pad;
    P.ld_resid = c->ld_resid;
    P.resid = c->resid;
    P.gam = c->gam;
    P.mu = c->mu;
    P.dtab = c->dtab;
    P.wtab = c->wtab;
    P.i0tab = c->i0tab;
    P.xnsq = c->xnsq;
    P.sig2tab = c->sig2tab;
    P.tau = c->tvec;
    P.log_tau = c->tvec + c->q_pad;
    P.c = cc;
    P.log_sig2_inv = log_sig2_inv;
    P.sig2_inv = sig2_inv;
    P.out = c->mis_out;
    P.mode = mode;
    c->rowpart_rows = 0;
    const int warps = 4, grid = (c->q + warps - 1) / warps;
    const int M = (c->n + 31) / 32;
    AQ_CUDA(cudaEventRecord(c->ev0, c->stream));
    if (M <= 4) mis_sweep_kernel<4><<<grid, warps * 32, 0, c->stream>>>(P);
    else if (M <= 8) mis_sweep_kernel<8><<<grid, warps * 32, 0, c->stream>>>(P);
    else if (M <= 16) mis_sweep_kernel<16><<<grid, warps * 32, 0, c->stream>>>(P);
    else if (M <= 32) mis_sweep_kernel<32><<<grid, warps * 32, 0, c->stream>>>(P);
    else mis_sweep_kernel<64><<<grid, warps * 32, 0, c->stream>>>(P);
    AQ_CUDA(cudaGetLastError());
    AQ_CUDA(cudaEventRecord(c->ev1, c->stream));
    c->launches++;
    return AQ_OK;
}

int fetch_mis(aq_ctx* c, const int* rows, double* const* outs, int nout) {
    c->hbuf.resize((size_t)kMisOutputs * c->q_pad);
    AQ_CUDA(cudaMemcpyAsync(c->hbuf.data(), c->mis_out, sizeof(double) * kMisOutputs * (size_t)c->q_pad,
                            cudaMemcpyDeviceToHost, c->stream));
    AQ_CUDA(cudaStreamSynchronize(c->stream));
    for (int i = 0; i < nout; ++i)
        if (outs[i]) std::memcpy(outs[i], c->hbuf.data() + (size_t)rows[i] * c->q_pad, sizeof(double) * c->q);
    return AQ_OK;
}
}  // namespace

}  // extern "C"

namespace {
// (Re)build the per-trait Gram band table and X_norm_sq of the tile path: depends on the masks and on the sweep order.
int build_gk(aq_ctx* c) {
    const int ntiles = c->ntiles;
    AQ_CUDA(cudaMemsetAsync(c->xnsq, 0, sizeof(double) * (size_t)c->p_pad * c->q_pad, c->stream));
    gk_build_kernel<<<dim3(c->nb, ntiles), 128, 0, c->stream>>>(c->xtiles, c->nb, c->cfg.ncta, c->cfg.k->n_pad, c->cfg.k->xs,
                                                                c->cfg.k->tile_doubles, c->mis_off_dev, c->mis_idx_dev, c->q,
                                                                c->q_pad, c->gk, c->xnsq);
    AQ_CUDA(cudaGetLastError());
    c->launches++;
    return AQ_OK;
}

// Tile-structured missing-response path: switch the context to the MIS kernel configuration for its n (16-trait tiles,
// smaller sample tiles: the X tile images, Y and the residual are laid out again), build the observed-sample bit matrix,
// the CSR lists of missing samples and the per-trait Gram band table.
int set_missing_tile(aq_ctx* c, const CfgInfo& cfgm, const double* mis_pat, double* n_obs) {
    const size_t pq = (size_t)c->p_pad * c->q_pad;
    const int n = c->n, q = c->q;
    if (cfgm.k != c->cfg.k || cfgm.ncta != c->cfg.ncta) {
        const int ld_new = cfgm.k->n_pad * cfgm.ncta;
        double *y_new = nullptr, *r_new = nullptr, *t_new = nullptr;
        AQ_CUDA(cudaStreamSynchronize(c->stream));
        AQ_CUDA(cudaFree(c->xtiles));
        c->xtiles = nullptr;
        AQ_CUDA(cudaFree(c->resid));
        c->resid = nullptr;
        AQ_CUDA(cudaMalloc((void**)&y_new, sizeof(double) * (size_t)c->q_pad * ld_new));
        AQ_CUDA(cudaMemsetAsync(y_new, 0, sizeof(double) * (size_t)c->q_pad * ld_new, c->stream));
        AQ_CUDA(cudaMemcpy2DAsync(y_new, sizeof(double) * ld_new, c->ymat, sizeof(double) * c->ld_resid, sizeof(double) * n, q,
                                  cudaMemcpyDeviceToDevice, c->stream));
        AQ_CUDA(cudaStreamSynchronize(c->stream));
        AQ_CUDA(cudaFree(c->ymat));
        c->ymat = y_new;
        AQ_CUDA(cudaMalloc((void**)&r_new, sizeof(double) * (size_t)c->q_pad * ld_new));
        c->resid = r_new;
        AQ_CUDA(cudaMalloc((void**)&t_new, sizeof(double) * (size_t)c->nb * cfgm.ncta * cfgm.k->tile_doubles));
        c->xtiles = t_new;
        c->cfg = cfgm;
        c->ld_resid = ld_new;
        c->ntiles = (q + cfgm.k->kT - 1) / cfgm.k->kT;
        c->attr_done[0] = c->attr_done[1] = false;
        if (c->seg_done) { cudaFree(c->seg_done); c->seg_done = nullptr; }
        if (c->rowpart) { cudaFree(c->rowpart); c->rowpart = nullptr; }
        c->rowpart_tried = true;   // (the tile path of the missing-response sweep streams the row sums)
        int rc = retile(c);
        if (rc != AQ_OK) return rc;
    }
    c->mwords = (c->ld_resid + 63) / 64;
    if (c->mbits) { cudaFree(c->mbits); c->mbits = nullptr; }
    AQ_CUDA(cudaMalloc((void**)&c->mbits, sizeof(unsigned long long) * (size_t)c->q_pad * c->mwords));
    AQ_CUDA(cudaMemsetAsync(c->mbits, 0, sizeof(unsigned long long) * (size_t)c->q_pad * c->mwords, c->stream));
    if (!c->xnsq) AQ_CUDA(cudaMalloc((void**)&c->xnsq, sizeof(double) * pq));
    if (!c->atab) AQ_CUDA(cudaMalloc((void**)&c->atab, sizeof(double) * pq));
    if (!c->ltab) AQ_CUDA(cudaMalloc((void**)&c->ltab, sizeof(double) * pq));
    if (!c->n_obs) AQ_CUDA(cudaMalloc((void**)&c->n_obs, sizeof(double) * c->q_pad));
    if (!c->mis_out) AQ_CUDA(cudaMalloc((void**)&c->mis_out, sizeof(double) * kMisOutputs * (size_t)c->q_pad));
    AQ_CUDA(cudaMemsetAsync(c->atab, 0, sizeof(double) * pq, c->stream));
    AQ_CUDA(cudaMemsetAsync(c->ltab, 0, sizeof(double) * pq, c->stream));
    AQ_CUDA(cudaMemsetAsync(c->mis_out, 0, sizeof(double) * kMisOutputs * (size_t)c->q_pad, c->stream));
    // the n x q pattern goes through the residual buffer (same [q][ld] orientation, ld >= n), which is rebuilt by set_state
    double* tmp = c->resid;
    AQ_CUDA(cudaMemcpyAsync(tmp, mis_pat, sizeof(double) * (size_t)n * q, cudaMemcpyHostToDevice, c->stream));
    pack_bits_kernel<<<(q + 7) / 8, 256, 0, c->stream>>>(tmp, n, q, c->mwords, c->ld_resid, c->mbits, c->ymat, c->n_obs);
    AQ_CUDA(cudaGetLastError());
    c->launches++;
    // CSR lists of the missing samples of every trait (rows of padding traits are empty)
    std::vector<int32_t> off((size_t)c->q_pad + 1, 0), idx;
    for (int k = 0; k < q; ++k) {
        const double* col = mis_pat + (size_t)k * n;
        for (int i = 0; i < n; ++i)
            if (col[i] == 0.0) idx.push_back(i);
        off[k + 1] = (int32_t)idx.size();
    }
    for (int k = q; k < c->q_pad; ++k) off[k + 1] = off[q];
    if (c->mis_off_dev) { cudaFree(c->mis_off_dev); c->mis_off_dev = nullptr; }
    if (c->mis_idx_dev) { cudaFree(c->mis_idx_dev); c->mis_idx_dev = nullptr; }
    AQ_CUDA(cudaMalloc((void**)&c->mis_off_dev, sizeof(int32_t) * off.size()));
    AQ_CUDA(cudaMalloc((void**)&c->mis_idx_dev, sizeof(int32_t) * std::max<size_t>(idx.size(), 1)));
    AQ_CUDA(cudaMemcpyAsync(c->mis_off_dev, off.data(), sizeof(int32_t) * off.size(), cudaMemcpyHostToDevice, c->stream));
    if (!idx.empty())
        AQ_CUDA(cudaMemcpyAsync(c->mis_idx_dev, idx.data(), sizeof(int32_t) * idx.size(), cudaMemcpyHostToDevice, c->stream));
    if (c->gk) { cudaFree(c->gk); c->gk = nullptr; }
    AQ_CUDA(cudaMalloc((void**)&c->gk, sizeof(double) * (size_t)c->ntiles * c->nb * 128 * 16));
    c->has_mis = true;
    c->mis_tile = true;
    c->have_state = false;
    int rc = build_gk(c);
    if (rc != AQ_OK) return rc;
    if (n_obs) AQ_CUDA(cudaMemcpyAsync(n_obs, c->n_obs, sizeof(double) * q, cudaMemcpyDeviceToHost, c->stream));
    AQ_CUDA(cudaStreamSynchronize(c->stream));   // (off / idx are host vectors: the copies must be through before they go)
    return AQ_OK;
}
}  // namespace

extern "C" {

int aq_set_missing(aq_ctx* c, const double* mis_pat, double* n_obs) {
    if (!c || !mis_pat) return fail(AQ_EINVAL, "aq_set_missing: NULL argument");
    if (!c->xraw) return fail(AQ_ESTATE, "aq_set_missing after aq_release_x");
    if (c->has_mis) return fail(AQ_ESTATE, "aq_set_missing: the missing-value pattern of a context is set once");
    AQ_CUDA(cudaSetDevice(c->device));
    const size_t pq = (size_t)c->p_pad * c->q_pad;
    // Two kernels serve coreDualMisLoop: the tile-structured one (the blocked tensor-core sweep with masked accumulators
    // and a per-trait Gram band table of 128 B per SNP x trait pair, n <= 5376) and the warp-per-trait one (no table,
    // n <= 2048, ~8x slower).  The tile path is taken whenever its table fits beside the rest; AQ_MIS_KERNEL=warp|tile forces.
    const CfgInfo cfgm = c->ov.mis_warp ? CfgInfo{} : pick_cfg(c->n, c->q, c->sm_count, true, c->ov.force_cluster);
    bool tile_ok = cfgm.k != nullptr;
    if (tile_ok) {
        size_t fr = 0, tot = 0;
        AQ_CUDA(cudaMemGetInfo(&fr, &tot));
        const size_t ntiles16 = (size_t)(c->q + 15) / 16;
        const double need = 8.0 * (double)ntiles16 * c->nb * 128 * 16 + 3.0 * 8.0 * (double)pq +
                            8.0 * (double)c->nb * cfgm.ncta * (double)cfgm.k->tile_doubles +
                            16.0 * (double)c->q_pad * cfgm.k->n_pad * cfgm.ncta + (double)((size_t)256 << 20);
        const double freed = 8.0 * (double)c->nb * c->cfg.ncta * (double)c->cfg.k->tile_doubles + 16.0 * (double)c->q_pad * c->ld_resid;
        if (need > (double)fr + freed) tile_ok = false;
    }
    if (tile_ok) return set_missing_tile(c, cfgm, mis_pat, n_obs);
    if (c->ov.mis_tile) return fail(AQ_EUNSUPPORTED, "aq_set_missing: the tile-structured kernel needs n <= 5376 and 128 B per SNP x trait pair");
    if (c->n > 2048)
        return fail(AQ_EUNSUPPORTED, "aq_set_missing: no room for the tile kernel's Gram band table (128 B per SNP x trait pair) "
                                     "and the warp-per-trait kernel covers n <= 2048 only");
    if (!c->mask) AQ_CUDA(cudaMalloc((void**)&c->mask, sizeof(unsigned long long) * 32 * (size_t)c->q_pad));
    if (!c->xnsq) AQ_CUDA(cudaMalloc((void**)&c->xnsq, sizeof(double) * pq));
    if (!c->n_obs) AQ_CUDA(cudaMalloc((void**)&c->n_obs, sizeof(double) * c->q_pad));
    if (!c->mis_out) AQ_CUDA(cudaMalloc((void**)&c->mis_out, sizeof(double) * kMisOutputs * (size_t)c->q_pad));
    AQ_CUDA(cudaMemsetAsync(c->xnsq, 0, sizeof(double) * pq, c->stream));
    AQ_CUDA(cudaMemsetAsync(c->mask, 0, sizeof(unsigned long long) * 32 * (size_t)c->q_pad, c->stream));
    // the n x q pattern goes through the residual buffer (same [q][ld] orientation, ld >= n), which is rebuilt by set_state
    double* tmp = c->resid;
    AQ_CUDA(cudaMemcpyAsync(tmp, mis_pat, sizeof(double) * (size_t)c->n * c->q, cudaMemcpyHostToDevice, c->stream));
    pack_mask_kernel<<<(c->q + 7) / 8, 256, 0, c->stream>>>(tmp, c->n, c->q, c->ld_resid, c->mask, c->ymat, c->n_obs);
    AQ_CUDA(cudaGetLastError());
    c->launches++;
    c->has_mis = true;
    c->have_state = false;
    int rc = launch_mis(c, /*mode=*/2, 1.0, 0.0, 0.0);   // X_norm_sq = crossprod(X^2, mis_pat)
    if (rc != AQ_OK) return rc;
    if (n_obs) AQ_CUDA(cudaMemcpyAsync(n_obs, c->n_obs, sizeof(double) * c->q, cudaMemcpyDeviceToHost, c->stream));
    AQ_CUDA(cudaStreamSynchronize(c->stream));
    return AQ_OK;
}

int aq_set_state_mis(aq_ctx* c, const double* gam_vb, const double* mu_beta_vb, double* colsum_gam,
                     double* colsum_gam_mu2, double* colsum_beta2, double* resid_sq, double* colsum_xn_gam,
                     double* colsum_xn_gam_mu2, double* colsum_xn_beta2) {
    if (!c || !gam_vb || !mu_beta_vb) return fail(AQ_EINVAL, "aq_set_state_mis: NULL argument");
    if (!c->has_mis) return fail(AQ_ESTATE, "aq_set_state_mis before aq_set_missing");
    AQ_CUDA(cudaSetDevice(c->device));
    int rc = upload_pxq(c, gam_vb, c->gam);
    if (rc != AQ_OK) return rc;
    rc = upload_pxq(c, mu_beta_vb, c->mu);
    if (rc != AQ_OK) return rc;
    AQ_CUDA(cudaMemcpyAsync(c->resid, c->ymat, sizeof(double) * (size_t)c->q_pad * c->ld_resid, cudaMemcpyDeviceToDevice,
                            c->stream));
    rc = c->mis_tile ? launch_sweep(c, /*mode=*/1, 1.0, 0.0) : launch_mis(c, /*mode=*/1, 1.0, 0.0, 0.0);
    if (rc != AQ_OK) return rc;
    c->have_state = true;
    const int rows[7] = {kMisGam, kMisGamMu2, kMisS2Gam, kMisRsq, kMisXnS2Gam, kMisXnGamMu2, kMisXnBeta2};
    double* outs[7] = {colsum_gam, colsum_gam_mu2, colsum_beta2, resid_sq, colsum_xn_gam, colsum_xn_gam_mu2, colsum_xn_beta2};
    return fetch_mis(c, rows, outs, 7);
}

int aq_sweep_mis(aq_ctx* c, double cc, double log_sig2_inv_vb, double sig2_inv_vb, const double* tau_vb,
                 const double* log_tau_vb, double* colsum_gam, double* colsum_gam_mu2, double* colsum_sig2b_gam,
                 double* colsum_xn_gam_mu2, double* colsum_xn_sig2b_gam, double* colsum_xn_beta2, double* resid_sq,
                 double* colsum_zpart, double* colsum_gam_logsig2b) {
    if (!c || !tau_vb || !log_tau_vb) return fail(AQ_EINVAL, "aq_sweep_mis: NULL argument");
    if (!c->has_mis) return fail(AQ_ESTATE, "aq_sweep_mis before aq_set_missing");
    if (!c->have_state) return fail(AQ_ESTATE, "aq_sweep_mis before aq_set_state_mis");
    if (!c->have_tables) return fail(AQ_ESTATE, "aq_sweep_mis before aq_refresh_tables");
    if (!(cc > 0.0) || !(sig2_inv_vb > 0.0)) return fail(AQ_EINVAL, "aq_sweep_mis: c and sig2_inv_vb must be positive");
    AQ_CUDA(cudaSetDevice(c->device));
    AQ_CUDA(cudaMemcpyAsync(c->tvec, tau_vb, sizeof(double) * c->q, cudaMemcpyHostToDevice, c->stream));
    AQ_CUDA(cudaMemcpyAsync(c->tvec + c->q_pad, log_tau_vb, sizeof(double) * c->q, cudaMemcpyHostToDevice, c->stream));
    int rc;
    if (c->mis_tile) {
        // sig2_beta_vb(j, k) of this sweep, as a = c sig2_beta tau and log sig2_beta (one streaming pass, 24 B per pair)
        mis_prep_kernel<<<dim3((c->q + 255) / 256, std::min(c->p, 4096)), 256, 0, c->stream>>>(
            c->xnsq, c->sig2tab, c->tvec, c->p, c->q, c->q_pad, cc, sig2_inv_vb, c->atab, c->ltab);
        AQ_CUDA(cudaGetLastError());
        c->launches++;
        rc = launch_sweep(c, /*mode=*/0, cc, log_sig2_inv_vb);
    } else {
        rc = launch_mis(c, /*mode=*/0, cc, log_sig2_inv_vb, sig2_inv_vb);
    }
    if (rc != AQ_OK) return rc;
    const int rows[9] = {kMisGam, kMisGamMu2, kMisS2Gam, kMisXnGamMu2, kMisXnS2Gam, kMisXnBeta2, kMisRsq, kMisZ, kMisGamLogS2};
    double* outs[9] = {colsum_gam, colsum_gam_mu2, colsum_sig2b_gam, colsum_xn_gam_mu2, colsum_xn_sig2b_gam,
                       colsum_xn_beta2, resid_sq, colsum_zpart, colsum_gam_logsig2b};
    rc = fetch_mis(c, rows, outs, 9);
    if (rc != AQ_OK) return rc;
    AQ_CUDA(cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1));
    return AQ_OK;
}

// ---------------------------------------------------------------- selection sets (R/summarise_output.R:99-106, :207-223)
namespace {
int sel_scratch(aq_ctx* c) {
    if (!c->have_state) return fail(AQ_ESTATE, "selection before aq_set_state");
    AQ_CUDA(cudaSetDevice(c->device));
    if (!c->sel_partial) AQ_CUDA(cudaMalloc((void**)&c->sel_partial, sizeof(double) * (2 * kSelBlocks + 2)));
    return AQ_OK;
}
}  // namespace

int aq_ppi_count_sum(aq_ctx* c, double t, double* count, double* sum) {
    if (!c || !count || !sum) return fail(AQ_EINVAL, "aq_ppi_count_sum: NULL argument");
    int rc = sel_scratch(c);
    if (rc != AQ_OK) return rc;
    double* res = c->sel_partial + 2 * kSelBlocks;
    ppi_count_sum_kernel<<<kSelBlocks, 256, 0, c->stream>>>(c->gam, c->p, c->q, c->q_pad, t, c->sel_partial);
    ppi_finish_kernel<<<1, 256, 0, c->stream>>>(c->sel_partial, kSelBlocks, 0, res);
    AQ_CUDA(cudaGetLastError());
    c->launches += 2;
    double h[2];
    AQ_CUDA(cudaMemcpyAsync(h, res, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    AQ_CUDA(cudaStreamSynchronize(c->stream));
    *count = h[0];
    *sum = h[1];
    return AQ_OK;
}

int aq_ppi_next_above(aq_ctx* c, double t, double* next) {
    if (!c || !next) return fail(AQ_EINVAL, "aq_ppi_next_above: NULL argument");
    int rc = sel_scratch(c);
    if (rc != AQ_OK) return rc;
    double* res = c->sel_partial + 2 * kSelBlocks;
    ppi_next_kernel<<<kSelBlocks, 256, 0, c->stream>>>(c->gam, c->p, c->q, c->q_pad, t, c->sel_partial);
    ppi_finish_kernel<<<1, 256, 0, c->stream>>>(c->sel_partial, kSelBlocks, 1, res);
    AQ_CUDA(cudaGetLastError());
    c->launches += 2;
    AQ_CUDA(cudaMemcpyAsync(next, res, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    AQ_CUDA(cudaStreamSynchronize(c->stream));
    return AQ_OK;
}

int aq_ppi_collect(aq_ctx* c, int mode, double lo, double hi, int64_t capacity, int32_t* out_j, int32_t* out_k,
                   double* out_gam, int64_t* n_found) {
    if (!c || !n_found) return fail(AQ_EINVAL, "aq_ppi_collect: NULL argument");
    if (mode != 0 && mode != 1) return fail(AQ_EINVAL, "aq_ppi_collect: mode must be 0 (1 - PPI in (lo, hi]) or 1 (PPI > lo)");
    if (capacity < 0 || (capacity > 0 && (!out_j || !out_k || !out_gam))) return fail(AQ_EINVAL, "aq_ppi_collect: bad output buffers");
    int rc = sel_scratch(c);
    if (rc != AQ_OK) return rc;
    int *dj = nullptr, *dk = nullptr;
    double* dg = nullptr;
    unsigned long long* cnt = reinterpret_cast<unsigned long long*>(c->sel_partial);
    const size_t cap = (size_t)std::max<int64_t>(capacity, 1);
    cudaError_t e = cudaMalloc((void**)&dj, sizeof(int) * cap);
    if (e == cudaSuccess) e = cudaMalloc((void**)&dk, sizeof(int) * cap);
    if (e == cudaSuccess) e = cudaMalloc((void**)&dg, sizeof(double) * cap);
    if (e == cudaSuccess) e = cudaMemsetAsync(cnt, 0, sizeof(unsigned long long), c->stream);
    unsigned long long found = 0;
    if (e == cudaSuccess) {
        ppi_collect_kernel<<<kSelBlocks, 256, 0, c->stream>>>(c->gam, c->p, c->q, c->q_pad, mode, lo, hi, (long long)capacity,
                                                               dj, dk, dg, cnt);
        e = cudaGetLastError();
        c->launches++;
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(&found, cnt, sizeof(found), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    const size_t ncopy = (size_t)std::min<unsigned long long>(found, (unsigned long long)capacity);
    if (e == cudaSuccess && ncopy) e = cudaMemcpy(out_j, dj, sizeof(int) * ncopy, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && ncopy) e = cudaMemcpy(out_k, dk, sizeof(int) * ncopy, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && ncopy) e = cudaMemcpy(out_gam, dg, sizeof(double) * ncopy, cudaMemcpyDeviceToHost);
    cudaFree(dj);
    cudaFree(dk);
    cudaFree(dg);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(e == cudaErrorMemoryAllocation ? AQ_ENOMEM : AQ_ECUDA, std::string("aq_ppi_collect: ") + cudaGetErrorString(e));
    }
    *n_found = (int64_t)found;
    return AQ_OK;
}

int64_t aq_launch_count(const aq_ctx* c) { return c ? c->launches : 0; }

int aq_sweep_plan(const aq_ctx* c, int* traits_per_tile, int* ntiles, int* groups, int* nseg) {
    if (!c) return fail(AQ_EINVAL, "NULL context");
    if (traits_per_tile) *traits_per_tile = c->cfg.k->kT;
    if (ntiles) *ntiles = c->ntiles;
    if (groups) *groups = c->max_groups[0];
    if (nseg) *nseg = c->last_nseg;
    return AQ_OK;
}

namespace {
__global__ void test_logistic_kernel(const double* __restrict__ x, double* __restrict__ out, int n, int variant) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = variant ? aq::logistic_neg<true>(x[i]) : aq::logistic_neg<false>(x[i]);
}
}  // namespace

int aq_test_logistic(int device, int variant, const double* x, double* out, int n) {
    if (!x || !out || n < 0 || (variant != 0 && variant != 1)) return fail(AQ_EINVAL, "aq_test_logistic: bad argument");
    if (n == 0) return AQ_OK;
    int rc = aq_device_info(device, nullptr, nullptr, nullptr);
    if (rc != AQ_OK) return rc;
    double *dx = nullptr, *dout = nullptr;
    AQ_CUDA(cudaMalloc((void**)&dx, sizeof(double) * (size_t)n));
    cudaError_t e = cudaMalloc((void**)&dout, sizeof(double) * (size_t)n);
    if (e == cudaSuccess) e = cudaMemcpy(dx, x, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        test_logistic_kernel<<<(n + 255) / 256, 256>>>(dx, dout, n, variant);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(out, dout, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost);
    cudaFree(dx);
    if (dout) cudaFree(dout);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(AQ_ECUDA, std::string("aq_test_logistic: ") + cudaGetErrorString(e));
    }
    return AQ_OK;
}

int aq_last_sweep_ms(const aq_ctx* c, float* ms) {
    if (!c || !ms) return fail(AQ_EINVAL, "NULL argument");
    *ms = c->last_ms;
    return AQ_OK;
}

int aq_last_ms(const aq_ctx* c, int which, float* ms) {
    if (!c || !ms) return fail(AQ_EINVAL, "NULL argument");
    if (which == 0) *ms = c->last_ms;
    else if (which == 1) *ms = c->last_rows_ms;
    else if (which == 2) *ms = c->last_tables_ms;
    else return fail(AQ_EINVAL, "aq_last_ms: which must be 0 (sweep), 1 (row sums) or 2 (tables)");
    return AQ_OK;
}

int aq_sync(aq_ctx* c) {
    if (!c) return fail(AQ_EINVAL, "NULL context");
    AQ_CUDA(cudaSetDevice(c->device));
    AQ_CUDA(cudaStreamSynchronize(c->stream));
    return AQ_OK;
}

}  // extern "C"
