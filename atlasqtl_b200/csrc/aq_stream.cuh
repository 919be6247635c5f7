// Streaming / set-up kernels around the sweep: X tiling + Gram band, layout transposes, the
// log-normal-CDF table pass (with ELBO term B), and the row sums of Z.
#pragma once
#include "aq_common.cuh"

namespace aq {

// ---------------------------------------------------------------- X tiles (one CTA per SNP block x sample slice)
// xraw: [p][n] (column j of the R matrix X contiguous).  order: sweep position -> SNP index.
// Slice r = blockIdx.y holds samples [r * n_pad_c, (r + 1) * n_pad_c); image (b, r) sits at (b * nslice + r) * tile_stride.
__global__ void build_tiles_kernel(const double* __restrict__ xraw, const int* __restrict__ order, int n, int p,
                                   int xs, int n_pad_c, size_t tile_stride, double* __restrict__ tiles) {
    const int b = blockIdx.x, r = blockIdx.y, nslice = gridDim.y;
    double* tile = tiles + ((size_t)b * nslice + r) * tile_stride;
    for (int t = 0; t < kBlk; ++t) {
        const int pos = b * kBlk + t;
        const int j = pos < p ? order[pos] : -1;
        for (int i = threadIdx.x; i < xs; i += blockDim.x) {
            // physical slot i holds logical sample swz(i, t) (the XOR is an involution) of this slice
            const int li = swz(i, t);
            const int gi = r * n_pad_c + li;
            tile[t * xs + i] = (j >= 0 && li < n_pad_c && gi < n) ? xraw[(size_t)j * n + gi] : 0.0;
        }
        if (threadIdx.x == 0) reinterpret_cast<int*>(tile + kBlk * xs + 128)[t] = j;
    }
    if (threadIdx.x < 8) reinterpret_cast<int*>(tile + kBlk * xs + 128)[8 + threadIdx.x] = 0;
}

// Gram band of block b: g[t][u] = X_t' X_u for u in block b+1 (u = 0..7; zero for the last block) and in block b
// (u = 8..15), over ALL sample slices; written into every slice's image.  128 threads, one (t, u) pair each; reads the
// freshly built tiles.
__global__ void gram_band_kernel(double* __restrict__ tiles, int n_pad_c, int nslice, int xs, size_t tile_stride) {
    const int b = blockIdx.x;
    const int t = threadIdx.x >> 4, u = threadIdx.x & 15;
    double acc = 0.0;
    if (u >= 8 || b + 1 < (int)gridDim.x) {
        const int uu = u & 7;
        const int bo = (u >= 8) ? b : b + 1;
        for (int r = 0; r < nslice; ++r) {
            const double* xt = tiles + ((size_t)b * nslice + r) * tile_stride + t * xs;
            const double* xu = tiles + ((size_t)bo * nslice + r) * tile_stride + uu * xs;
            for (int i = 0; i < n_pad_c; ++i) acc = fma(xt[swz(i, t)], xu[swz(i, uu)], acc);
        }
    }
    for (int r = 0; r < nslice; ++r) tiles[((size_t)b * nslice + r) * tile_stride + kBlk * xs + t * 16 + u] = acc;
}

// ---------------------------------------------------------------- layout transposes (32 x 32 smem tiles)
// src: kc columns of an R matrix, column-major with leading dimension p  (src[kk * p + j])
// dst: device layout [p_pad][q_pad], trait-contiguous                    (dst[j * q_pad + k_first + kk])
__global__ void cm_to_dev_kernel(const double* __restrict__ src, int p, int kc, int k_first, int q_pad,
                                 double* __restrict__ dst) {
    __shared__ double tile[32][33];
    const int j0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int kk = c0 + r, j = j0 + threadIdx.x;
        tile[r][threadIdx.x] = (kk < kc && j < p) ? src[(size_t)kk * p + j] : 0.0;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int j = j0 + r, kk = c0 + threadIdx.x;
        if (j < p && kk < kc) dst[(size_t)j * q_pad + k_first + kk] = tile[threadIdx.x][r];
    }
}
// inverse; op: 0 copy a, 1 product a * b (beta_vb = gam_vb * mu_beta_vb)
__global__ void dev_to_cm_kernel(const double* __restrict__ a, const double* __restrict__ b2, int op, int p, int kc,
                                 int k_first, int q_pad, double* __restrict__ dst) {
    __shared__ double tile[32][33];
    const int j0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int j = j0 + r, kk = c0 + threadIdx.x;
        double v = 0.0;
        if (j < p && kk < kc) {
            const size_t off = (size_t)j * q_pad + k_first + kk;
            v = a[off];
            if (op == 1) v *= b2[off];
        }
        tile[r][threadIdx.x] = v;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int kk = c0 + r, j = j0 + threadIdx.x;
        if (kk < kc && j < p) dst[(size_t)kk * p + j] = tile[threadIdx.x][r];
    }
}

__global__ void fill_kernel(double* __restrict__ x, size_t nelem, double v) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < nelem; i += (size_t)gridDim.x * blockDim.x) x[i] = v;
}

// ---------------------------------------------------------------- table pass (K1)
// For every (j, k): u = theta_j + zeta_k; lp = log Phi(u); lq = log Phi(-u);
//   D = lq - lp;  at U = sqrt(c) u:  imr1 = phi(U)/Phi(U) (>= -U), imr0 = -phi(U)/(1 - Phi(U)) (<= -U)
//   W = imr1 - imr0;  I0 = imr0.                             (R/utils.R:172-191, R/update_vb.R:217-234)
// Optional ELBO-B part (R/elbo.R:19-26): sum gam lp + (1-gam) lq - gam log(gam+eps) - (1-gam) log(1-gam+eps).
// Grid: blockIdx.y strides over rows j, blockIdx.x * blockDim.x covers traits k (coalesced); one ELBO partial per CTA.
// gridDim.y is capped at 65,535, so for p > 524,280 the host launches the pass on slices of at most kTabMaxGridRows row
// blocks, with theta, the p x q arrays and the partials offset to the slice (one launch below that).
constexpr int kTabRowsPerBlock = 8;
constexpr int kTabMaxGridRows = 65535;

// row blocks of the table pass: with the 256-trait column blocks, the number of CTAs over all launches and of ELBO partials
inline int tab_row_blocks(int p) { return (p + kTabRowsPerBlock - 1) / kTabRowsPerBlock; }

// Everything the table pass needs about the standard normal at one point u, from ONE erfcx, ONE exp, one log and
// one log1p:  with a = |u|/sqrt2, E = erfcx(a), e2 = exp(-u^2/2):  Q = E e2 / 2 is the tail mass beyond |u|,
//   log Q = log(E/2) - u^2/2,  log(1-Q) = log1p(-Q),  phi/Q = sqrt(2/pi)/E  (no exp),  phi/(1-Q) = e2/(sqrt(2 pi)(1-Q)).
// 1 / d for d in [2^-100, 2^100]: hardware seed (20 bits) times (1 + e + e^2), relative error e^3 < 1e-18 plus one rounding.
// The IEEE division costs ~4x as many fp64 operations, and this pass is bound by exactly those.
__device__ __forceinline__ double fast_rcp(double d) {
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
    const double e0 = fma(-d, y, 1.0);
    return fma(y, fma(e0, e0, e0), y);
}

struct NormalPoint {
    double log_tail, log_body;  // log Q, log(1 - Q)
    double r_tail, r_body;      // phi / Q, phi / (1 - Q)
};
__device__ __forceinline__ NormalPoint normal_point(double u, bool want_logs, bool want_ratios) {
    const double kRs2 = 0.70710678118654752440, kSqrt2OverPi = 0.79788456080286535588, kInvSqrt2Pi = 0.39894228040143267794;
    NormalPoint o;
    const double a = fabs(u) * kRs2;
    const double E = erfcx(a);
    const double e2 = exp(-0.5 * u * u);
    const double Q = 0.5 * E * e2;
    if (want_logs) {
        o.log_tail = log(0.5 * E) - 0.5 * u * u;
        o.log_body = log1p(-Q);
    }
    if (want_ratios) {   // E in (0, 1] falls off like 0.8 / |u|: inside fast_rcp's [2^-100, 2^100] for |u| < 2^99.
                         // 1 - Q in [0.5, 1]
        o.r_tail = kSqrt2OverPi * fast_rcp(E);
        o.r_body = kInvSqrt2Pi * e2 * fast_rcp(1.0 - Q);
    }
    return o;
}

// The same point when only the log-odds of the tail are wanted (no ELBO on this iteration): one log instead of log + log1p,
// log(Q / (1 - Q)) = log(E / (2 (1 - Q))) - u^2 / 2, and the reciprocal of 1 - Q is shared with phi / (1 - Q).
// (exp underflows beyond |u| = 38.6: Q = 0 there and the expression degrades to log(E / 2) - u^2 / 2, still exact.)
__device__ __forceinline__ double normal_point_logodds(double u, bool want_ratios, double& r_tail, double& r_body) {
    const double kRs2 = 0.70710678118654752440, kSqrt2OverPi = 0.79788456080286535588, kInvSqrt2Pi = 0.39894228040143267794;
    const double a = fabs(u) * kRs2;
    const double E = erfcx(a);
    const double e2 = exp(-0.5 * u * u);
    const double Q = 0.5 * E * e2;
    const double inv = fast_rcp(1.0 - Q);
    if (want_ratios) {
        r_tail = kSqrt2OverPi * fast_rcp(E);
        r_body = kInvSqrt2Pi * e2 * inv;
    }
    return log(0.5 * E * inv) - 0.5 * u * u;
}

__global__ void __launch_bounds__(256) tables_kernel(const double* __restrict__ theta, const double* __restrict__ zeta, int p,
                                                     int q, int q_pad, double sqrt_c, int c_is_one,
                                                     const double* __restrict__ gam, double* __restrict__ dtab,
                                                     double* __restrict__ wtab, double* __restrict__ i0tab, int want_elbo,
                                                     double* __restrict__ partials) {
    const double eps = 1.8189894035458565e-12;  // .Machine$double.eps^0.75 (R/elbo.R:15)
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    double part = 0.0;
    if (k < q) {
        const double zk = zeta[k];
        const int j0 = blockIdx.y * kTabRowsPerBlock;
#pragma unroll 1
        for (int r = 0; r < kTabRowsPerBlock; ++r) {
            const int j = j0 + r;
            if (j >= p) break;
            const size_t off = (size_t)j * q_pad + k;
            const double u = theta[j] + zk;
            double lp = 0.0, lq = 0.0, U = u, r_tail = 0.0, r_body = 0.0;
            if (want_elbo) {
                const NormalPoint nu = normal_point(u, true, c_is_one != 0);
                lp = (u >= 0.0) ? nu.log_body : nu.log_tail;  // log Phi(u)
                lq = (u >= 0.0) ? nu.log_tail : nu.log_body;  // log(1 - Phi(u))
                dtab[off] = lq - lp;
                r_tail = nu.r_tail;
                r_body = nu.r_body;
            } else {
                const double lo = normal_point_logodds(u, c_is_one != 0, r_tail, r_body);  // log(tail / body)
                dtab[off] = (u >= 0.0) ? lo : -lo;
            }
            if (!c_is_one) {  // update_Z_ evaluates the CDFs at sqrt(c) (theta + zeta) while annealing (R/update_vb.R:219-224)
                U = sqrt_c * u;
                const NormalPoint nU = normal_point(U, false, true);
                r_tail = nU.r_tail;
                r_body = nU.r_body;
            }
            double m1 = (U >= 0.0) ? r_body : r_tail;    // phi(U) / Phi(U)
            double m0 = -((U >= 0.0) ? r_tail : r_body); // -phi(U) / (1 - Phi(U))
            if (m1 < -U) m1 = -U;                        // R/utils.R:179, :184
            if (m0 > -U) m0 = -U;
            wtab[off] = m1 - m0;
            i0tab[off] = m0;
            if (want_elbo) {
                const double gm = gam[off];
                part += gm * lp + (1.0 - gm) * lq - gm * log(gm + eps) - (1.0 - gm) * log(1.0 - gm + eps);
            }
        }
    }
    if (want_elbo) {
        __shared__ double red[8];
        part = warp_sum(part);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
        __syncthreads();
        if (threadIdx.x == 0) {
            double s = 0.0;
            for (int w = 0; w < 8; ++w) s += red[w];
            partials[(size_t)blockIdx.y * gridDim.x + blockIdx.x] = s;
        }
    }
}

// deterministic sum of `n` doubles by one block of 1024 threads
__global__ void sum_partials_kernel(const double* __restrict__ x, size_t n, double* __restrict__ out) {
    __shared__ double red[32];
    double s = 0.0;
    for (size_t i = threadIdx.x; i < n; i += blockDim.x) s += x[i];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
        double v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.0;
        v = warp_sum(v);
        if (threadIdx.x == 0) *out = v;
    }
}

// ---------------------------------------------------------------- row sums of the Z part (K3)
// rowsum[j] = sum_k gam[j][k] * W[j][k] + I0[j][k]; one warp per row, fixed summation order.
__global__ void __launch_bounds__(256) rowsums_kernel(const double* __restrict__ gam, const double* __restrict__ wtab,
                                                      const double* __restrict__ i0tab, int p, int q, int q_pad,
                                                      double* __restrict__ rowsum) {
    const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (j >= p) return;
    const int lane = threadIdx.x & 31;
    const size_t base = (size_t)j * q_pad;
    double s0 = 0.0, s1 = 0.0;
    const int q2 = q & ~1;
    for (int k = 2 * lane; k < q2; k += 64) {
        const double2 g = *reinterpret_cast<const double2*>(gam + base + k);
        const double2 w = *reinterpret_cast<const double2*>(wtab + base + k);
        const double2 i0 = *reinterpret_cast<const double2*>(i0tab + base + k);
        s0 += fma(g.x, w.x, i0.x);
        s1 += fma(g.y, w.y, i0.y);
    }
    if (lane == 0 && q2 < q) s0 += fma(gam[base + q2], wtab[base + q2], i0tab[base + q2]);
    const double s = warp_sum(s0 + s1);
    if (lane == 0) rowsum[j] = s;
}

// rowsum[j] = sum over the sweep's trait tiles of their partial row sums (rowpart [nrows][p_pad], written by the helper
// warps of the sweep kernel): 0.5 GB instead of the 24 GB of the three p x q arrays at C2.  Block = 32 SNPs x 8 row
// lanes; fixed order.
__global__ void __launch_bounds__(256) rowpart_reduce_kernel(const double* __restrict__ rowpart, int nrows, int p, int p_pad,
                                                             double* __restrict__ rowsum) {
    __shared__ double red[8][33];
    const int j = blockIdx.x * 32 + threadIdx.x;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    if (j < p) {
        const double* col = rowpart + j;
        int r = threadIdx.y;
        for (; r + 24 < nrows; r += 32) {
            s0 += col[(size_t)r * p_pad];
            s1 += col[(size_t)(r + 8) * p_pad];
            s2 += col[(size_t)(r + 16) * p_pad];
            s3 += col[(size_t)(r + 24) * p_pad];
        }
        for (; r < nrows; r += 8) s0 += col[(size_t)r * p_pad];
    }
    red[threadIdx.y][threadIdx.x] = (s0 + s1) + (s2 + s3);
    __syncthreads();
    if (threadIdx.y == 0 && j < p) {
        double s = 0.0;
#pragma unroll
        for (int y = 0; y < 8; ++y) s += red[y][threadIdx.x];
        rowsum[j] = s;
    }
}

}  // namespace aq
