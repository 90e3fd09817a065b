// txh_da.cu -- data-assimilation kernels for sm_100a.
//
// Device form of KalmanFilter.filter (tx_fast_hydrology/da.py:91-136).  The dense contractions
// of the update -- innovation covariance, ensemble transform, gain application, and the
// covariance products of the dense filter -- run on the FP64 tensor cores (mma.sync m8n8k4,
// DMMA in SASS); everything else (means, gathers, the small SPD solve) is plain FP64.
// Matrices are row-major.  State matrices are the routing layout: one row per reach (schedule
// order), members contiguous, `ld` doubles per row.
// For ensembles of up to 64 members with a diagonal observation-error covariance the whole ensemble-space system --
// gauge gather, split-K product, reduction, Cholesky solve, W -- is ONE launch of a 16-CTA thread-block cluster
// (enkf_small_system_kernel: distributed shared memory for the reduce-scatter and the exchange of the solution).
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <cstdlib>

#include "txh_kernels.cuh"

namespace txh {

void count_launch();

namespace {

// D(8x8) += A(8x4) * B(4x8), FP64.  Fragment ownership (lane = 4*g + t):
//   a = A[g][t], b = B[t][g], c0 = C[g][2t], c1 = C[g][2t+1]
__device__ __forceinline__ void dmma8x8x4(double& c0, double& c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// ---- generic C = alpha * op(A) op(B) + beta * C ------------------------------------------------
// CTA tile 64x64, K tile 16; 8 warps, each a 16x32 sub-tile = 2x4 DMMA tiles.
constexpr int GB_M = 64, GB_N = 64, GB_K = 16;

// Split-K: blockIdx.z owns the k range [z*kchunk, (z+1)*kchunk) and writes its partial product to
// C + z*cstride (kchunk == K, gridDim.z == 1: the plain product).
__global__ void __launch_bounds__(256)
dgemm_kernel(int transA, int transB, int M, int N, int K, double alpha, const double* __restrict__ A, int lda,
             const double* __restrict__ B, int ldb, double beta, double* C, int ldc, int kchunk,
             long long cstride, const double* Cin, int ldcin)
{
    __shared__ double sA[GB_M][GB_K + 1];      // sA[m][k]
    __shared__ double sB[GB_K][GB_N + 1];      // sB[k][n]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int m0 = blockIdx.y * GB_M, n0 = blockIdx.x * GB_N;
    const int wm = (warp >> 1) * 16, wn = (warp & 1) * 32;
    double acc[2][4][2];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    const int kbeg = blockIdx.z * kchunk;
    K = min(K, kbeg + kchunk);
    C += (size_t)blockIdx.z * cstride;
    // software pipeline: the next k tile travels global -> registers while the current one is multiplied
    double ra[4], rb[4];
    auto fetch = [&](int k0) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int e = tid + u * 256;
            int m, k;
            if (transA) { m = e % GB_M; k = e / GB_M; } else { k = e % GB_K; m = e / GB_K; }
            const int gm = m0 + m, gk = k0 + k;
            ra[u] = (gm < M && gk < K) ? (transA ? A[(size_t)gk * lda + gm] : A[(size_t)gm * lda + gk]) : 0.0;
            int kb, n;
            if (transB) { kb = e % GB_K; n = e / GB_K; } else { n = e % GB_N; kb = e / GB_N; }
            const int gkb = k0 + kb, gn = n0 + n;
            rb[u] = (gkb < K && gn < N) ? (transB ? B[(size_t)gn * ldb + gkb] : B[(size_t)gkb * ldb + gn]) : 0.0;
        }
    };
    if (kbeg < K) fetch(kbeg);
    for (int k0 = kbeg; k0 < K; k0 += GB_K) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int e = tid + u * 256;
            int m, k;
            if (transA) { m = e % GB_M; k = e / GB_M; } else { k = e % GB_K; m = e / GB_K; }
            sA[m][k] = ra[u];
            int kb, n;
            if (transB) { kb = e % GB_K; n = e / GB_K; } else { n = e % GB_N; kb = e / GB_N; }
            sB[kb][n] = rb[u];
        }
        __syncthreads();
        if (k0 + GB_K < K) fetch(k0 + GB_K);
#pragma unroll
        for (int kk = 0; kk < GB_K; kk += 4) {
            double a[2], b[4];
#pragma unroll
            for (int i = 0; i < 2; ++i) a[i] = sA[wm + 8 * i + g][kk + t];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = sB[kk + t][wn + 8 * j + g];
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) dmma8x8x4(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const int gm = m0 + wm + 8 * i + g, gn = n0 + wn + 8 * j + 2 * t + c;
                if (gm < M && gn < N) {
                    C[(size_t)gm * ldc + gn] =
                        alpha * acc[i][j][c] + (beta == 0.0 ? 0.0 : beta * Cin[(size_t)gm * ldcin + gn]);
                }
            }
}

// ---- ensemble statistics ---------------------------------------------------------------------
// rowsum[k] = scale * sum over this shard's members of X[k][:]  (one warp per row; scale = 1/Mtot turns it
// into the ensemble mean when the shard is the whole ensemble), and the rows of the gauged reaches copied
// to HX[g][0..M) in the same pass (gauge_of_pos[k] = gauge index or -1).
__global__ void __launch_bounds__(256)
enkf_stats_kernel(const double* __restrict__ X, int ld, int M, long long n, double scale,
                  const int32_t* __restrict__ gauge_of_pos, double* __restrict__ rowsum, double* __restrict__ HX)
{
    const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= n) return;
    const double* p = X + (size_t)row * ld;
    const int gi = gauge_of_pos ? gauge_of_pos[row] : -1;
    double s = 0.0;
    for (int m = 2 * lane; m < M; m += 64) {
        const double2 v = *reinterpret_cast<const double2*>(p + m);
        s += v.x;
        if (m + 1 < M) s += v.y;
        if (gi >= 0) { HX[(size_t)gi * M + m] = v.x; if (m + 1 < M) HX[(size_t)gi * M + m + 1] = v.y; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) rowsum[row] = s * scale;
}

// HA[k][m] = HX[k][m] - mean_k ; dz[k][m] = Zp[k][m] - HX[k][m]     (da.py:112)
__global__ void __launch_bounds__(256)
innovation_kernel(const double* __restrict__ HX, const double* __restrict__ Zp, const double* __restrict__ mean_obs,
                  int m, int M, double* __restrict__ HA, double* __restrict__ dz)
{
    const int gid = blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= m * M) return;
    const int k = gid / M;
    const double hx = HX[gid];
    HA[gid] = hx - mean_obs[k];
    dz[gid] = Zp[gid] - hx;
}

// S = S * scale + diag(qs) + R        (P[s][:, s] + R_cov with P = sample covariance + Q, da.py:117-119)
__global__ void __launch_bounds__(256)
innov_cov_finish_kernel(double* __restrict__ S, const double* __restrict__ qs, const double* __restrict__ R, int m,
                        double scale)
{
    const int gid = blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= m * m) return;
    const int i = gid / m, j = gid - i * m;
    S[gid] = S[gid] * scale + R[gid] + (i == j ? qs[i] : 0.0);
}

// In-place Cholesky factorisation + solve S X = B for SPD S [m][m], B [m][k].  One CTA of 1024
// threads; S stays in global memory (L2 resident).  Left-looking by column, the dot products
// of a column spread over the whole CTA (warp per row, lanes over the inner index).
__global__ void __launch_bounds__(1024)
spd_solve_kernel(double* __restrict__ S, double* __restrict__ B, int m, int k, int* __restrict__ info)
{
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = blockDim.x >> 5;
    __shared__ double diag;
    // factor: S = L L^T, L stored in the lower triangle
    for (int j = 0; j < m; ++j) {
        // rows i >= j: S[i][j] -= sum_{p<j} L[i][p] L[j][p]
        for (int i = j + warp; i < m; i += nwarp) {
            const double* Li = S + (size_t)i * m;
            const double* Lj = S + (size_t)j * m;
            double s = 0.0;
            for (int p = lane; p < j; p += 32) s += Li[p] * Lj[p];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0) S[(size_t)i * m + j] -= s;
        }
        __syncthreads();
        if (tid == 0) {
            const double d = S[(size_t)j * m + j];
            if (!(d > 0.0)) { *info = j + 1; diag = 1.0; } else diag = sqrt(d);
            S[(size_t)j * m + j] = diag;
        }
        __syncthreads();
        const double inv = 1.0 / diag;
        for (int i = j + 1 + tid; i < m; i += blockDim.x) S[(size_t)i * m + j] *= inv;
        __syncthreads();
    }
    // forward substitution L Y = B, then backward L^T X = Y.  16 threads share a right-hand-side
    // column (inner index strided over them, combined with shuffles); 64 columns per pass.
    const int q = tid & 15, cl = tid >> 4;
    for (int c0 = 0; c0 < k; c0 += 64) {
        const int c = c0 + cl;
        const bool on = c < k;
        for (int i = 0; i < m; ++i) {
            const double* Li = S + (size_t)i * m;
            double s = 0.0;
            if (on) for (int p = q; p < i; p += 16) s += Li[p] * B[(size_t)p * k + c];
#pragma unroll
            for (int o = 8; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o, 16);
            if (on && q == 0) B[(size_t)i * k + c] = (B[(size_t)i * k + c] - s) / Li[i];
            __syncwarp();
        }
        for (int i = m - 1; i >= 0; --i) {
            double s = 0.0;
            if (on) for (int p = i + 1 + q; p < m; p += 16) s += S[(size_t)p * m + i] * B[(size_t)p * k + c];
#pragma unroll
            for (int o = 8; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o, 16);
            if (on && q == 0) B[(size_t)i * k + c] = (B[(size_t)i * k + c] - s) / S[(size_t)i * m + i];
            __syncwarp();
        }
    }
}

// ---- blocked Cholesky solve for systems too large for one CTA (S [m][m] row-major, B [m][k]) -------------
constexpr int PB = 32;

// factor the diagonal block S[j0:j0+nb, j0:j0+nb] in shared memory (every CTA repeats it), then by CTA:
//   0            : write the factor back
//   1..nslab     : a 64-row slab of the panel below, L21 = A21 L11^-T (one thread per row)
//   nslab+1..    : a 64-column slab of the right-hand sides, Y1 = L11^-1 B1 (one thread per column)
__global__ void __launch_bounds__(64)
chol_panel_kernel(double* __restrict__ S, int m, double* __restrict__ B, int k, int j0, int nb, int nslab,
                  int* __restrict__ info)
{
    __shared__ double D[PB][PB + 1];
    __shared__ double invd[PB];
    const int tid = threadIdx.x;
    for (int e = tid; e < PB * PB; e += 64) {
        const int i = e / PB, c = e - i * PB;
        D[i][c] = (i < nb && c < nb) ? S[(size_t)(j0 + i) * m + j0 + c] : (i == c ? 1.0 : 0.0);
    }
    __syncthreads();
    for (int j = 0; j < nb; ++j) {
        double d = D[j][j];
        if (!(d > 0.0)) { if (tid == 0 && blockIdx.x == 0) *info = j0 + j + 1; d = 1.0; }
        const double rs = rsqrt(d);
        __syncthreads();
        if (tid == 0) { D[j][j] = d * rs; invd[j] = rs; }
        if (tid > j && tid < nb) D[tid][j] *= rs;
        __syncthreads();
        if (tid > j && tid < nb) {
            const double l = D[tid][j];
            for (int c = j + 1; c <= tid; ++c) D[tid][c] -= l * D[c][j];
        }
        __syncthreads();
    }
    const int b = blockIdx.x;
    if (b == 0) {
        for (int e = tid; e < nb * nb; e += 64) {
            const int i = e / nb, c = e - i * nb;
            if (c <= i) S[(size_t)(j0 + i) * m + j0 + c] = D[i][c];
        }
    } else if (b <= nslab) {
        const int i = j0 + nb + (b - 1) * 64 + tid;
        if (i < m) {
            double* row = S + (size_t)i * m + j0;
            double x[PB];
#pragma unroll
            for (int c = 0; c < PB; ++c) {
                if (c < nb) {
                    double v = row[c];
#pragma unroll
                    for (int q = 0; q < c; ++q) v -= x[q] * D[c][q];
                    x[c] = v * invd[c];
                } else x[c] = 0.0;
            }
#pragma unroll
            for (int c = 0; c < PB; ++c) if (c < nb) row[c] = x[c];
        }
    } else {
        const int col = (b - nslab - 1) * 64 + tid;
        if (col < k) {
            double y[PB];
#pragma unroll
            for (int r = 0; r < PB; ++r) {
                if (r < nb) {
                    double v = B[(size_t)(j0 + r) * k + col];
#pragma unroll
                    for (int q = 0; q < r; ++q) v -= D[r][q] * y[q];
                    y[r] = v * invd[r];
                } else y[r] = 0.0;
            }
#pragma unroll
            for (int r = 0; r < PB; ++r) if (r < nb) B[(size_t)(j0 + r) * k + col] = y[r];
        }
    }
}

// Z1 = L11^-T Y1 for one diagonal block (one thread per right-hand-side column)
__global__ void __launch_bounds__(64)
chol_back_kernel(const double* __restrict__ S, int m, double* __restrict__ B, int k, int j0, int nb)
{
    __shared__ double D[PB][PB + 1];
    const int tid = threadIdx.x;
    for (int e = tid; e < PB * PB; e += 64) {
        const int i = e / PB, c = e - i * PB;
        D[i][c] = (i < nb && c <= i) ? S[(size_t)(j0 + i) * m + j0 + c] : (i == c ? 1.0 : 0.0);
    }
    __syncthreads();
    const int col = blockIdx.x * 64 + tid;
    if (col >= k) return;
    double z[PB];
#pragma unroll
    for (int r = PB - 1; r >= 0; --r) {
        if (r < nb) {
            double v = B[(size_t)(j0 + r) * k + col];
#pragma unroll
            for (int q = PB - 1; q > r; --q) if (q < nb) v -= D[q][r] * z[q];
            z[r] = v / D[r][r];
        } else z[r] = 0.0;
    }
#pragma unroll
    for (int r = 0; r < PB; ++r) if (r < nb) B[(size_t)(j0 + r) * k + col] = z[r];
}

// ---- ensemble-space (Woodbury) form of the innovation solve ----------------------------------------
// With D = R + diag(Q[s,s]) constant between updates and its inverse precomputed, the m x m system
// S W = dz,  S = HA HA^T/(Mt-1) + D,  collapses to an Mt x Mt one:
//     Y  = D^-1 [HA | dz]                      C = HA^T Y = [C0 | C1]
//     (C0 + (Mt-1) I) Z = C1                   T = HA^T W/(Mt-1) = Z          W = Y_dz - Y_HA Z
// (HA^T S^-1 = (Mt-1) (C0 + (Mt-1) I)^-1 HA^T D^-1, so the ensemble transform IS the small solve.)

// Bc[k] = [HA_k | dz_k] (2*Mt doubles per gauge); Y = dinv_k * Bc when D is diagonal.
__global__ void __launch_bounds__(256)
innovation_cat_kernel(double* __restrict__ HX, const double* __restrict__ O, int ldo, const double* __restrict__ Zp,
                      const double* __restrict__ mean, const int32_t* __restrict__ obs_pos,
                      const double* __restrict__ dinv_diag, int m, int Mt, double* __restrict__ Bc, double* __restrict__ Y)
{
    const int gid = blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= m * Mt) return;
    const int k = gid / Mt, c = gid - k * Mt;
    double hx;
    if (O) { hx = O[(size_t)obs_pos[k] * ldo + c]; HX[gid] = hx; }      // the gauge rows gathered on the way
    else hx = HX[gid];
    const double ha = hx - mean[obs_pos[k]], dz = Zp[gid] - hx;
    const size_t o = (size_t)k * 2 * Mt + c;
    Bc[o] = ha; Bc[o + Mt] = dz;
    if (dinv_diag) { const double d = dinv_diag[k]; Y[o] = d * ha; Y[o + Mt] = d * dz; }
}

// (sum of the split-K partials of C) -> A = C0 + shift*I, B = C1, then (C0 + shift I) Z = C1 by Cholesky.
// (A register-resident column-by-column variant with one barrier per column measured 58 us at 64 members; the
// blocked one below 31 us.)
constexpr int CS_NSPLIT = 8;

// Factorisation A = L L^T of the MT x MT matrix in shared memory (lower triangle, leading dimension MT + 1) and the
// solve for the CTA's 8 right-hand-side columns Bs [MT][9], in place.  256 threads; the caller has synchronised.
// Panels of 8 columns, two barriers per panel:
//   panel   : warp 0; every lane factors the 8 x 8 diagonal block itself, in registers, and solves its own rows below the
//             block against it (lane l owns rows j0+8+l, j0+8+l+32, ...) -- no shuffles, no barrier inside a panel (a
//             version that exchanged the pivot column with shuffles took 283 cycles per column, this one 196).  This
//             is the critical path (64 dependent rsqrt).  Meanwhile
//             warp 1 inverts the diagonal block of the PREVIOUS panel (8 lanes, one column of L11^-1 each) and forms
//             that panel's rows of the forward substitution, Y = L11^-1 B1, with two tensor-core operations;
//   trailing: every warp takes 8x8 tiles of the lower triangle and applies the rank-8 update of the new panel, and
//             tiles of B for the update with the previous panel's Y, two FP64 tensor-core MMAs per tile.
// The forward substitution thus rides one panel behind the factorisation, off its critical path; the backward
// substitution multiplies with the inverted diagonal blocks (Z1 = L11^-T Y1, two MMAs) instead of eight dependent
// steps, one barrier per panel.  Linv: [MT/8][8][9] scratch for the inverted blocks.
template <int MT>
__device__ __forceinline__ void chol_factor_solve_smem(double* A, double* Bs, double* invd, double* Linv, int* info,
                                                       bool report)
{
    constexpr int LD = MT + 1, NT = MT / 8, RPL = MT / 32, LDB = 9, LDI = 9;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    // X = L_qq^-1 (lower triangular) -> Linv[q], then the rows of panel q of B: Y = X B_q   (one warp)
    auto invert_and_forward = [&](int q) {
        const int j0 = 8 * q;
        double* Li = Linv + q * 8 * LDI;
        if (lane < 8) {
            double x[8];
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                double v = (r == lane) ? 1.0 : 0.0;
#pragma unroll
                for (int k = 0; k < r; ++k) v -= A[(j0 + r) * LD + j0 + k] * x[k];
                x[r] = v * invd[j0 + r];
            }
#pragma unroll
            for (int r = 0; r < 8; ++r) Li[r * LDI + lane] = x[r];
        }
        __syncwarp();
        double c0 = 0.0, c1 = 0.0;
#pragma unroll
        for (int kk = 0; kk < 8; kk += 4) dmma8x8x4(c0, c1, Li[g * LDI + kk + t], Bs[(j0 + kk + t) * LDB + g]);
        __syncwarp();
        Bs[(j0 + g) * LDB + 2 * t] = c0; Bs[(j0 + g) * LDB + 2 * t + 1] = c1;
    };
    // ---- factorisation, the forward substitution one panel behind ----
    for (int p = 0; p < NT; ++p) {
        const int j0 = 8 * p;
        if (warp == 0) {
            // every lane factors the 8 x 8 diagonal block itself, in registers (36 broadcast loads, no shuffles: the
            // chain per column is rsqrt + two multiply-adds), and solves its own rows below the block against it
            double Dm[8][8], rs[8];
#pragma unroll
            for (int r = 0; r < 8; ++r)
#pragma unroll
                for (int c = 0; c <= r; ++c) Dm[r][c] = A[(j0 + r) * LD + j0 + c];
            double x[RPL][8];
#pragma unroll
            for (int q = 0; q < RPL; ++q) {
                const int i = j0 + 8 + lane + 32 * q;
#pragma unroll
                for (int cc = 0; cc < 8; ++cc) x[q][cc] = i < MT ? A[i * LD + j0 + cc] : 0.0;
            }
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
                double d = Dm[jj][jj];
                if (!(d > 0.0)) { if (lane == 0 && report) *info = j0 + jj + 1; d = 1.0; }
                rs[jj] = rsqrt(d);
                Dm[jj][jj] = d * rs[jj];
#pragma unroll
                for (int r = jj + 1; r < 8; ++r) Dm[r][jj] *= rs[jj];
#pragma unroll
                for (int r = jj + 1; r < 8; ++r)
#pragma unroll
                    for (int c = jj + 1; c <= r; ++c) Dm[r][c] -= Dm[r][jj] * Dm[c][jj];
                // column jj of the rows below: x = (x - sum_{k<jj} x_k L[jj][k]) / L[jj][jj]
#pragma unroll
                for (int q = 0; q < RPL; ++q) {
                    double v = x[q][jj];
#pragma unroll
                    for (int k = 0; k < jj; ++k) v -= x[q][k] * Dm[jj][k];
                    x[q][jj] = v * rs[jj];
                }
            }
            // every lane holds the same block: all of them store it (same value to the same address, no divergence)
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                invd[j0 + r] = rs[r];
#pragma unroll
                for (int c = 0; c <= r; ++c) A[(j0 + r) * LD + j0 + c] = Dm[r][c];
            }
#pragma unroll
            for (int q = 0; q < RPL; ++q) {
                const int i = j0 + 8 + lane + 32 * q;
                if (i < MT)
#pragma unroll
                    for (int cc = 0; cc < 8; ++cc) A[i * LD + j0 + cc] = x[q][cc];
            }
        } else if (warp == 1 && p > 0) {
            invert_and_forward(p - 1);
        }
        __syncthreads();
        // trailing update: tiles (it, ct), p < ct <= it < NT, of A with panel p; tiles it >= p of B with Y of panel p-1
        const int Tn = NT - p - 1;
        const int nA = Tn * (Tn + 1) / 2, nB = p > 0 ? NT - p : 0;
        for (int e = warp; e < nA + nB; e += 8) {
            int it, ct = 0, k0 = j0;
            const bool isB = e >= nA;
            if (!isB) {
                it = 0;
                int rem = e;
                while (rem > it) { rem -= it + 1; ++it; }                        // row it has it+1 tiles
                ct = p + 1 + rem; it = p + 1 + it;
            } else { it = p + (e - nA); k0 = j0 - 8; }
            double* cp = isB ? Bs + (8 * it + g) * LDB + 2 * t : A + (8 * it + g) * LD + 8 * ct + 2 * t;
            double c0 = cp[0], c1 = cp[1];
#pragma unroll
            for (int kk = 0; kk < 8; kk += 4) {
                const double af = -A[(8 * it + g) * LD + k0 + kk + t];
                const double bf = isB ? Bs[(k0 + kk + t) * LDB + g] : A[(8 * ct + g) * LD + k0 + kk + t];
                dmma8x8x4(c0, c1, af, bf);
            }
            cp[0] = c0; cp[1] = c1;
        }
        __syncthreads();
    }
    if (warp == 1) invert_and_forward(NT - 1);
    __syncthreads();
    // ---- backward substitution L^T Z = Y: Z_p = L_pp^-T Y_p, rows above -= L[p][it]^T Z_p ----
    auto back_block = [&](int q) {                              // one warp: rows of panel q of Bs <- Linv[q]^T times them
        const int j0 = 8 * q;
        const double* Li = Linv + q * 8 * LDI;
        double c0 = 0.0, c1 = 0.0;
#pragma unroll
        for (int kk = 0; kk < 8; kk += 4) dmma8x8x4(c0, c1, Li[(kk + t) * LDI + g], Bs[(j0 + kk + t) * LDB + g]);
        __syncwarp();
        Bs[(j0 + g) * LDB + 2 * t] = c0; Bs[(j0 + g) * LDB + 2 * t + 1] = c1;
        __syncwarp();
    };
    if (warp == 0) back_block(NT - 1);
    __syncthreads();
    for (int p = NT - 1; p > 0; --p) {
        const int j0 = 8 * p;
        // warp 0 takes the tile right above and goes straight on to the next block solve; one barrier per panel
        for (int it = p - 1 - warp; it >= 0; it -= 8) {
            double* cp = Bs + (8 * it + g) * LDB + 2 * t;
            double c0 = cp[0], c1 = cp[1];
#pragma unroll
            for (int kk = 0; kk < 8; kk += 4) {
                const double af = -A[(j0 + kk + t) * LD + 8 * it + g];
                const double bf = Bs[(j0 + kk + t) * LDB + g];
                dmma8x8x4(c0, c1, af, bf);
            }
            cp[0] = c0; cp[1] = c1;
        }
        if (warp == 0) { __syncwarp(); back_block(p - 1); }
        __syncthreads();
    }
}

// Blocked small solve (chol_factor_solve_smem) fed by the split-K partials of a GEMM launch.
// Right-hand sides are split over CTAs, 8 columns each (every CTA repeats the factorisation).
template <int MT>
__global__ void __launch_bounds__(256)
chol_solve_blocked_kernel(const double* __restrict__ Cpart, long long pstride, int Mt, double shift,
                          double* __restrict__ Z, int* __restrict__ info)
{
    constexpr int LD = MT + 1, LDB = 9;
    extern __shared__ double sm[];
    double* A = sm;                       // [MT][MT+1], lower triangle: working matrix, then L
    double* Bs = A + MT * LD;             // [MT][9]     this CTA's 8 right-hand-side columns
    double* invd = Bs + MT * LDB;         // [MT]        1 / L[j][j]
    const int tid = threadIdx.x;
    const int gc0 = blockIdx.x * 8;
    // the split-K partials are summed on the way in: 8 elements x 8 partials in flight per thread, lower triangle
    // only (the upper one is never read)
    for (int e0 = 0; e0 < MT * MT; e0 += 8 * 256) {
        double part[8][CS_NSPLIT];
        // unconditional loads (an element that is not needed reads element 0): all 64 are issued before the first add
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int e = e0 + u * 256 + tid;
            const int i = e / MT, c = e - i * MT;
            const bool need = e < MT * MT && i < Mt && c <= i;
            const double* src = Cpart + (need ? (size_t)i * 2 * Mt + c : 0);
#pragma unroll
            for (int s = 0; s < CS_NSPLIT; ++s) part[u][s] = __ldg(src + (size_t)s * pstride);
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int e = e0 + u * 256 + tid;
            const int i = e / MT, c = e - i * MT;
            const bool need = e < MT * MT && i < Mt && c <= i;
            double acc = (i == c) ? shift : 0.0;
#pragma unroll
            for (int s = 0; s < CS_NSPLIT; ++s) acc += part[u][s];
            if (e < MT * MT) A[i * LD + c] = need ? acc : ((i == c) ? 1.0 : 0.0);
        }
    }
    {
        constexpr int NB = MT * 8 / 256;                       // right-hand-side elements per thread
        double part[NB][CS_NSPLIT];
#pragma unroll
        for (int u = 0; u < NB; ++u) {
            const int e = tid + u * 256;
            const int i = e >> 3, cl = e & 7;
            const bool need = i < Mt && gc0 + cl < Mt;
            const double* src = Cpart + (need ? (size_t)i * 2 * Mt + Mt + gc0 + cl : 0);
#pragma unroll
            for (int s = 0; s < CS_NSPLIT; ++s) part[u][s] = __ldg(src + (size_t)s * pstride);
        }
#pragma unroll
        for (int u = 0; u < NB; ++u) {
            const int e = tid + u * 256;
            const int i = e >> 3, cl = e & 7;
            double v = 0.0;
#pragma unroll
            for (int s = 0; s < CS_NSPLIT; ++s) v += part[u][s];
            Bs[i * LDB + cl] = (i < Mt && gc0 + cl < Mt) ? v : 0.0;
        }
    }
    __syncthreads();
    chol_factor_solve_smem<MT>(A, Bs, invd, invd + MT, info, blockIdx.x == 0);
    for (int e = tid; e < MT * 8; e += 256) {
        const int i = e >> 3, cl = e & 7;
        if (i < Mt && gc0 + cl < Mt) Z[(size_t)i * Mt + gc0 + cl] = Bs[i * LDB + cl];
    }
}

// ---- the whole ensemble-space system in ONE launch (Mt <= 64, diagonal D) ---------------------------------------
// A cluster of NC = 16 (or 8) CTAs replaces innovation_cat + split-K GEMM + chol_solve_blocked + GEMM (4 launches, 3
// trips through global memory):
//   1. CTA r gathers its share of the gauge rows, [HA | dz] -> shared memory, and multiplies its split-K partial of
//      C = HA^T D^-1 [HA | dz] on the FP64 tensor cores (D^-1 rides on the A fragments);
//   2. reduce-scatter through distributed shared memory: CTA r sums slice r of C over the cluster (DSMEM moves
//      ~20 bytes per clock and SM, so nobody reads more than 1/NC of every partial);
//   3. the CTAs of rank < 8 collect the lower triangle of C0 (+ shift I) and their own 8 columns of C1 from the slices,
//      factor C0 + shift I (repeated, as in chol_solve_blocked_kernel) and solve their columns of Z = T; the columns
//      are scattered into every CTA's copy of Z (distributed shared memory) and written to T;
//   4. CTA r forms W = D^-1 (dz - HA Z) for its gauges from the tile it still holds.
constexpr int SS_KT = 64;                        // gauges per shared-memory tile
constexpr int SS_LDB = 136;                      // [HA | dz] row stride in doubles (128 + 8: conflict-free fragments)
constexpr int SS_LDZ = 72;
constexpr int SS_OFF_C = SS_KT * SS_LDB;                   // sC   [64][128] this CTA's partial
constexpr int SS_OFF_R = SS_OFF_C + 64 * 128;              // sR   [8192 / NC] this CTA's slice of the sum (<= 1024)
constexpr int SS_OFF_A = SS_OFF_R + 1024;                  // A    [64][65]
constexpr int SS_OFF_BS = SS_OFF_A + 64 * 65;              // Bs   [64][9]
constexpr int SS_OFF_INVD = SS_OFF_BS + 64 * 9;            // invd [64]
constexpr int SS_OFF_Z = SS_OFF_INVD + 64;                 // sZ   [64][72]
constexpr int SS_OFF_D = SS_OFF_Z + 64 * SS_LDZ;           // sd   [64]
constexpr int SS_OFF_LINV = SS_OFF_D + SS_KT;              // Linv [8][8][9] inverted diagonal blocks of the factor
constexpr int SS_SMEM = (SS_OFF_LINV + 8 * 72) * 8;        // 223,744 bytes

template <int NC>
__global__ void __launch_bounds__(256, 1)
enkf_small_system_kernel(double* __restrict__ HX, const double* __restrict__ O, int ldo, const double* __restrict__ Zp,
                         const double* __restrict__ mean, const int32_t* __restrict__ obs_pos,
                         const double* __restrict__ dinv, int m, int Mt, double shift, double* __restrict__ T,
                         double* __restrict__ W, int* __restrict__ info, unsigned long long* __restrict__ trace)
{
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    extern __shared__ double ss[];
    double* sB = ss;
    double* sC = ss + SS_OFF_C;
    double* sR = ss + SS_OFF_R;
    double* A = ss + SS_OFF_A;
    double* Bs = ss + SS_OFF_BS;
    double* invd = ss + SS_OFF_INVD;
    double* sZ = ss + SS_OFF_Z;
    double* sd = ss + SS_OFF_D;
    double* Linv = ss + SS_OFF_LINV;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int mc = (((m + NC - 1) / NC) + 3) & ~3;                 // gauges per CTA
    const int k_lo = min(m, rank * mc), k_hi = min(m, k_lo + mc);
    auto stamp = [&](int i) {                                      // development aid (TXH_SS_TRACE): phase timeline
        if (trace && tid == 0) {
            unsigned long long ns;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
            trace[rank * 8 + i] = ns;
        }
    };
    // programmatic dependent launch: this kernel may have started before the routing launch in front of it has
    // finished; what it reads is final after the wait, and the routing launch behind it (which reads T and W only
    // after a wait of its own) may start loading its tasks from here on
    // (the wait itself sits inside the first load_tile: the gauge positions, the observations and D^-1 do not come from
    // the routing launch and are requested before it)
    bool waited = false;
    stamp(0);

    // [HA | dz] of the gauges kt .. kt+63 -> sB (zero rows beyond k_hi), D^-1 -> sd; every load of a thread's
    // elements is in flight before the first use
    auto load_tile = [&](int kt) {
        const int c = tid & 63;
        int pos[16];
#pragma unroll
        for (int u = 0; u < 16; ++u) {
            const int k = kt + (tid >> 6) + 4 * u;
            pos[u] = k < k_hi ? __ldg(obs_pos + k) : -1;
        }
        double hx[16], zp[16], mu[16];
#pragma unroll
        for (int u = 0; u < 16; ++u) {
            const int k = kt + (tid >> 6) + 4 * u;
            zp[u] = (pos[u] >= 0 && c < Mt) ? __ldg(Zp + (size_t)k * Mt + c) : 0.0;
        }
        const double dk = (tid < SS_KT && kt + tid < k_hi) ? __ldg(dinv + kt + tid) : 0.0;
        if (!waited) {
            asm volatile("griddepcontrol.wait;" ::: "memory");
            asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
            waited = true;
        }
#pragma unroll
        for (int u = 0; u < 16; ++u) {
            const int k = kt + (tid >> 6) + 4 * u;
            const bool on = pos[u] >= 0 && c < Mt;
            hx[u] = on ? (O ? __ldcg(O + (size_t)pos[u] * ldo + c) : __ldcg(HX + (size_t)k * Mt + c)) : 0.0;
            mu[u] = on ? __ldcg(mean + pos[u]) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 16; ++u) {
            const int kk = (tid >> 6) + 4 * u, k = kt + kk;
            const bool on = pos[u] >= 0 && c < Mt;
            if (on && O) HX[(size_t)k * Mt + c] = hx[u];
            sB[kk * SS_LDB + c] = hx[u] - mu[u];
            sB[kk * SS_LDB + 64 + c] = zp[u] - hx[u];
        }
        if (tid < SS_KT) sd[tid] = dk;
    };

    // ---- 1. split-K partial of C = HA^T D^-1 [HA | dz]: warp tile 16 x 64 of the 64 x 128 product ----
    const int wm = (warp >> 1) * 16, wn = (warp & 1) * 64;
    double acc[2][8][2];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    for (int kt = k_lo; kt == k_lo || kt < k_hi; kt += SS_KT) {
        if (kt != k_lo) __syncthreads();
        load_tile(kt);
        __syncthreads();
        const int nk = min(SS_KT, (max(k_hi - kt, 0) + 3) & ~3);
        for (int kk = 0; kk < nk; kk += 4) {
            const double* row = sB + (kk + t) * SS_LDB;
            const double d = sd[kk + t];
            double a[2], b[8];
#pragma unroll
            for (int i = 0; i < 2; ++i) a[i] = d * row[wm + 8 * i + g];
#pragma unroll
            for (int j = 0; j < 8; ++j) b[j] = row[wn + 8 * j + g];
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) dmma8x8x4(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
    }
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j)
            *reinterpret_cast<double2*>(sC + (wm + 8 * i + g) * 128 + wn + 8 * j + 2 * t) =
                make_double2(acc[i][j][0], acc[i][j][1]);
    stamp(1);
    cluster.sync();
    stamp(2);

    // ---- 2. reduce-scatter: slice `rank` of C (8192 / NC doubles), summed over the cluster in rank order ----
    constexpr int SL = 8192 / NC;                                  // doubles per slice: 512 (NC = 16) or 1024
    {
        constexpr int PT = SL / 2 / 256;                           // double2 per thread: 1 or 2
        double2 part[PT][NC];
#pragma unroll
        for (int u = 0; u < PT; ++u) {
            const int off = rank * SL + 2 * (tid + u * 256);
#pragma unroll
            for (int r = 0; r < NC; ++r) part[u][r] = *reinterpret_cast<const double2*>(cluster.map_shared_rank(sC, r) + off);
        }
#pragma unroll
        for (int u = 0; u < PT; ++u) {
            double2 v = part[u][0];
#pragma unroll
            for (int r = 1; r < NC; ++r) { v.x += part[u][r].x; v.y += part[u][r].y; }
            *reinterpret_cast<double2*>(sR + 2 * (tid + u * 256)) = v;
        }
    }
    cluster.sync();
    stamp(3);

    // ---- 3. ranks 0..7: lower triangle of C0 + shift I -> A, 8 columns of C1 -> Bs, from the owners' slices;
    //         (C0 + shift I) Z = C1 for these columns; Z goes to T and into every CTA's sZ ----
    const int gc0 = rank * 8;
    if (rank < 8) {
        // element (i, c) of C: flat index i*128 + c, owner flat / SL
        double2 va[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int e = 2 * (tid + u * 256);                     // pair (i, c), (i, c+1) of the 64 x 64 block C0
            const int i = e >> 6, c = e & 63;
            const int flat = i * 128 + c;
            va[u] = c <= i ? *reinterpret_cast<const double2*>(cluster.map_shared_rank(sR, flat / SL) + flat % SL)
                           : make_double2(0.0, 0.0);
        }
        double vb[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int e = tid + u * 256;
            const int flat = (e >> 3) * 128 + 64 + gc0 + (e & 7);
            vb[u] = cluster.map_shared_rank(sR, flat / SL)[flat % SL];
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int e = 2 * (tid + u * 256);
            const int i = e >> 6, c = e & 63;
            A[i * 65 + c] = c <= i ? va[u].x + (i == c ? shift : 0.0) : 0.0;
            A[i * 65 + c + 1] = c + 1 <= i ? va[u].y + (i == c + 1 ? shift : 0.0) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) { const int e = tid + u * 256; Bs[(e >> 3) * 9 + (e & 7)] = vb[u]; }
        __syncthreads();
        stamp(4);
        chol_factor_solve_smem<64>(A, Bs, invd, Linv, info, rank == 0);
        stamp(5);
        for (int e = tid; e < 64 * 8; e += 256) {
            const int i = e >> 3, cl = e & 7;
            const double v = Bs[i * 9 + cl];
            if (i < Mt && gc0 + cl < Mt) T[(size_t)i * Mt + gc0 + cl] = v;
#pragma unroll
            for (int r = 0; r < NC; ++r) cluster.map_shared_rank(sZ, r)[i * SS_LDZ + gc0 + cl] = v;
        }
    }
    cluster.sync();
    stamp(6);

    // ---- 4. W = D^-1 (dz - HA Z) for this CTA's gauges: warp tile 8 gauges x 64 columns ----
    for (int kt = k_lo; kt < k_hi; kt += SS_KT) {
        if (k_hi - k_lo > SS_KT) {                             // several tiles: fetch this one again (L2)
            __syncthreads();
            load_tile(kt);
            __syncthreads();
        }
        if (kt + 8 * warp >= k_hi) continue;                   // (warp-uniform: no gauges in this warp's rows)
        double w[8][2];
#pragma unroll
        for (int j = 0; j < 8; ++j) w[j][0] = w[j][1] = 0.0;
        const double* hrow = sB + (8 * warp + g) * SS_LDB;
#pragma unroll 4
        for (int kk = 0; kk < 64; kk += 4) {
            const double a = hrow[kk + t];
            const double* zr = sZ + (kk + t) * SS_LDZ + g;
#pragma unroll
            for (int j = 0; j < 8; ++j) dmma8x8x4(w[j][0], w[j][1], a, zr[8 * j]);
        }
        const int k = kt + 8 * warp + g;
        if (k < k_hi) {
            const double d = sd[8 * warp + g];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int col = 8 * j + 2 * t;
                if (col < Mt) W[(size_t)k * Mt + col] = d * (hrow[64 + col] - w[j][0]);
                if (col + 1 < Mt) W[(size_t)k * Mt + col + 1] = d * (hrow[64 + col + 1] - w[j][1]);
            }
        }
    }
    stamp(7);
}

// sum of the split-K partials of C = [C0 | C1] -> Cf = C0 + shift*I and C1 as two dense Mt x Mt matrices
__global__ void __launch_bounds__(256)
woodbury_assemble_kernel(const double* __restrict__ Cpart, int nsplit, long long pstride, int Mt, double shift,
                         double* __restrict__ Cf, double* __restrict__ C1)
{
    const int gid = blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= Mt * 2 * Mt) return;
    const int i = gid / (2 * Mt), j = gid - i * 2 * Mt;
    double v = 0.0;
    for (int s = 0; s < nsplit; ++s) v += Cpart[(size_t)s * pstride + gid];
    if (j < Mt) Cf[(size_t)i * Mt + j] = v + (i == j ? shift : 0.0);
    else C1[(size_t)i * Mt + (j - Mt)] = v;
}

// ---- ensemble transform applied to the state ------------------------------------------------------
// gain[k][c] = sum_j (Xall[k][j] - mean_k) T[j][c]  for this shard's columns c, written to G and added to
// O in place (da.py:126, o_t_next += gain); the inflow part of _apply_gain follows in inflow_gain_kernel.
// FP64 tensor cores (DMMA m8n8k4).  A warp owns 16 rows (two 8-row MMA tiles): its anomalies of one
// 64-member k chunk live in registers as A fragments (32 doubles per lane), the matching 64 x 64 block
// of T is staged in shared memory and every B fragment read feeds two MMAs.  The k index of a fragment
// is permuted (lane t holds members 8j+2t, 8j+2t+1 for k steps 2j, 2j+1) so that a lane fetches its two
// members of a row with one 128-bit load; T is read with the same permutation.
constexpr int EU_WARPS = 8, EU_ROWS = 16 * EU_WARPS, EU_LDT = 66;

__global__ void __launch_bounds__(EU_WARPS * 32)
enkf_update_kernel(const double* __restrict__ Xall, int ldx, int Mtot, const double* __restrict__ mean,
                   const double* __restrict__ T, int ldt, int Mloc, const double* O, double* Oout, double* __restrict__ G,
                   int ld, long long n, const int32_t* __restrict__ gauge_of_pos, const double* __restrict__ qs,
                   const double* __restrict__ W, int col0, int resident, int Mb, long long blk_stride,
                   const PeerBlocks peers)
{
    // peers.count > 0: block b of the ensemble is read where it lives -- peers.p[b] is the state matrix [n][ldx] of
    // shard b, the local one or a peer GPU's mapped over NVLink (the transform overlaps the transfer tile by tile;
    // nothing is gathered first).  The posterior then goes to Oout != O: a peer may still be reading O.
    // Xall: Mtot / Mb blocks of [n][ldx], block b holding members b*Mb .. (b+1)*Mb - 1 (what an all-gather of
    // the shards' state rows produces); Mb == Mtot: one matrix
    // `resident`: every 64-member k chunk of T has its own block of shared memory and is staged once per CTA
    // (single column group); otherwise one block is restaged for every (row tile, chunk)
    extern __shared__ double sT_all[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const bool vec = (ldx & 1) == 0 && (Mb & 1) == 0;
    const int nkc = (Mtot + 63) / 64, ncg = (ld + 63) / 64;
    for (long long r0 = (long long)blockIdx.x * EU_ROWS; r0 < n; r0 += (long long)gridDim.x * EU_ROWS) {
        const long long rw = r0 + warp * 16;
        const long long row0 = rw + g, row1 = rw + 8 + g;
        const double mu0 = row0 < n ? mean[row0] : 0.0, mu1 = row1 < n ? mean[row1] : 0.0;
        for (int cg = 0; cg < ncg; ++cg) {
            const int njt = min(8, (Mloc - cg * 64 + 7) >> 3);
            double acc[2][8][2];
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
            for (int kc = 0; kc < nkc; ++kc) {
                double* sT = sT_all + (resident ? kc * 64 * EU_LDT : 0);
                if ((!resident && nkc * ncg > 1) || r0 == (long long)blockIdx.x * EU_ROWS) {
                    // stage T[kc*64 .. +64][cg*64 .. +64] (zero outside the matrix); with a single block it
                    // is staged once per CTA
                    __syncthreads();
                    for (int e = tid; e < 64 * 64; e += EU_WARPS * 32) {
                        const int k = e >> 6, c = e & 63;
                        const int gk = kc * 64 + k, gc = cg * 64 + c;
                        sT[k * EU_LDT + c] = (gk < Mtot && gc < Mloc) ? T[(size_t)gk * ldt + gc] : 0.0;
                    }
                    __syncthreads();
                }
                // A fragments: a[i][2j], a[i][2j+1] = anomalies of members kc*64 + 8j + 2t, +1
                double a[2][16];
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const long long row = i ? row1 : row0;
                    const double mu = i ? mu1 : mu0;
                    const size_t xoff = (size_t)(row < n ? row : 0) * ldx;
                    const double* xrow = Xall + xoff;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const int k = kc * 64 + 8 * j + 2 * t;
                        double x0 = mu, x1 = mu;
                        if (row < n) {
                            const int b = k / Mb, kk = k - b * Mb;
                            const double* xr = (peers.count > 0 ? peers.p[b] + xoff : xrow + (size_t)b * blk_stride) + kk;
                            if (vec && k + 1 < Mtot) {
                                const double2 v = __ldcg(reinterpret_cast<const double2*>(xr));
                                x0 = v.x; x1 = v.y;
                            } else {
                                if (k < Mtot) x0 = __ldcg(xr);
                                if (k + 1 < Mtot)
                                    x1 = (kk + 1 < Mb) ? __ldcg(xr + 1)
                                                       : __ldcg(peers.count > 0 ? peers.p[b + 1] + xoff : xrow + (size_t)(b + 1) * blk_stride);
                            }
                        }
                        a[i][2 * j] = x0 - mu; a[i][2 * j + 1] = x1 - mu;
                    }
                }
#pragma unroll
                for (int ks = 0; ks < 16; ++ks) {
                    const int k = 8 * (ks >> 1) + 2 * t + (ks & 1);
                    const double* bt = sT + k * EU_LDT + g;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        if (j < njt) {                              // column tiles beyond this shard's members: skipped
                            const double b = bt[8 * j];
                            dmma8x8x4(acc[0][j][0], acc[0][j][1], a[0][ks], b);
                            dmma8x8x4(acc[1][j][0], acc[1][j][1], a[1][ks], b);
                        }
                    }
                }
            }
            // epilogue: G = gain, O += gain (row-local, so in place is safe); gauged rows add the Q[:, s]
            // term of the gain, qs[g] * W[g][col0 + c] (da.py:117-121)
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const long long row = i ? row1 : row0;
                if (row >= n) continue;
                const int gi = gauge_of_pos[row];
                const double qg = gi >= 0 ? qs[gi] : 0.0;
                const double* wr = W + (size_t)(gi >= 0 ? gi : 0) * Mtot + col0;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int col = cg * 64 + 8 * j + 2 * t;
                    if (col >= ld) continue;
                    double2 gn = make_double2(acc[i][j][0], col + 1 < Mloc ? acc[i][j][1] : 0.0);
                    if (col >= Mloc) gn.x = 0.0;
                    if (gi >= 0) {
                        if (col < Mloc) gn.x += qg * wr[col];
                        if (col + 1 < Mloc) gn.y += qg * wr[col + 1];
                    }
                    if (O) {
                        double2 o = *reinterpret_cast<const double2*>(O + (size_t)row * ld + col);
                        o.x += gn.x; o.y += gn.y;
                        *reinterpret_cast<double2*>(Oout + (size_t)row * ld + col) = o;
                    }
                    if (G) *reinterpret_cast<double2*>(G + (size_t)row * ld + col) = gn;
                }
            }
        }
    }
}

// The common case of the above -- the whole ensemble is this shard's (Xall == O's layout, Mtot = Mloc <= 64):
// T is staged once per CTA; every warp streams its 16-row tiles through a double-buffered shared-memory
// stage (cp.async, the next tile in flight while the tensor cores work on the current one) and reads both
// the A fragments and, in the epilogue, the old outflows from it, so O is read from global memory once.
constexpr int EU64_RT = 1;                        // row tiles per warp (see enkf_update64_kernel)
constexpr int EU_RS = 576;                       // bytes per staged row: 512 + 64, conflict-free 128-bit reads
constexpr int EU64_SMEM = 64 * EU_LDT * 8 + 16 * 2 * 8 * EU_RS;   // the same for 8 warps x 16 rows and 16 warps x 8 rows

template <int RT>                                 // 8-row MMA tiles per warp: 2 (8 warps per CTA) or 1 (16 warps)
__global__ void __launch_bounds__(512 / RT * 1, 1)
enkf_update64_kernel(const double* __restrict__ X, int M, const double* __restrict__ mean, const double* __restrict__ T,
                     int ldt, double* __restrict__ O, double* __restrict__ G, int ld, long long n,
                     const int32_t* __restrict__ gauge_of_pos, const double* __restrict__ qs,
                     const double* __restrict__ W)
{
    extern __shared__ __align__(16) unsigned char eu_smem[];
    double* sT = reinterpret_cast<double*>(eu_smem);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    constexpr int NW = 16 / RT, TR = 8 * RT;          // warps per CTA, rows per warp tile
    const unsigned stage0 = (unsigned)__cvta_generic_to_shared(eu_smem + 64 * EU_LDT * 8 + warp * 2 * TR * EU_RS);
    const long long ntiles = (n + TR - 1) / TR;
    const long long tstride = (long long)gridDim.x * NW;
    long long tile = (long long)blockIdx.x * NW + warp;
    auto prefetch = [&](long long tl, int buf) {
        if (tl < ntiles && 2 * lane < ld) {
            const long long r0 = tl * TR;
#pragma unroll
            for (int r = 0; r < TR; ++r)
                if (r0 + r < n) {
                    const unsigned sa = stage0 + (buf * TR + r) * EU_RS + lane * 16;
                    const double* gp = X + (size_t)(r0 + r) * ld + 2 * lane;
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(gp) : "memory");
                }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    prefetch(tile, 0);
    {
        // all 16 loads of a thread are in flight before the first store
        double tv[8 * RT];
#pragma unroll
        for (int u = 0; u < 8 * RT; ++u) {
            const int e = tid + u * NW * 32;
            const int k = e >> 6, c = e & 63;
            tv[u] = (k < M && c < M) ? __ldg(T + (size_t)k * ldt + c) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 8 * RT; ++u) {
            const int e = tid + u * NW * 32;
            sT[(e >> 6) * EU_LDT + (e & 63)] = tv[u];
        }
    }
    __syncthreads();
    int buf = 0;
    // mean and gauge index of this lane's two rows, fetched one tile ahead (a global round trip otherwise
    // exposed at the head of every tile)
    auto row_meta = [&](long long tl, double* mu_o, int* gi_o) {
#pragma unroll
        for (int i = 0; i < RT; ++i) {
            const long long row = tl * TR + 8 * i + g;
            const bool ok = tl < ntiles && row < n;
            mu_o[i] = ok ? __ldg(mean + row) : 0.0;
            gi_o[i] = ok ? __ldg(gauge_of_pos + row) : -1;
        }
    };
    double mu_n[RT];
    int gi_n[RT];
    row_meta(tile, mu_n, gi_n);
    for (; tile < ntiles; tile += tstride, buf ^= 1) {
        prefetch(tile + tstride, buf ^ 1);
        double mu[RT];
        int gi[RT];
#pragma unroll
        for (int i = 0; i < RT; ++i) { mu[i] = mu_n[i]; gi[i] = gi_n[i]; }
        row_meta(tile + tstride, mu_n, gi_n);
        asm volatile("cp.async.wait_group 1;" ::: "memory");
        __syncwarp();
        const long long rw = tile * TR;
        long long rows[RT];
#pragma unroll
        for (int i = 0; i < RT; ++i) rows[i] = rw + 8 * i + g;
        double a[RT][16];
#pragma unroll
        for (int i = 0; i < RT; ++i) {
            const bool ok = rows[i] < n;
            const unsigned ra = stage0 + (buf * TR + 8 * i + g) * EU_RS + t * 16;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int k = 8 * j + 2 * t;
                double2 v = make_double2(0.0, 0.0);
                if (ok && k < ld) asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(ra + j * 64));
                a[i][2 * j] = (ok && k < M) ? v.x - mu[i] : 0.0;
                a[i][2 * j + 1] = (ok && k + 1 < M) ? v.y - mu[i] : 0.0;
            }
        }
        double acc[RT][8][2];
#pragma unroll
        for (int i = 0; i < RT; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
#pragma unroll
        for (int ks = 0; ks < 16; ++ks) {
            const int k = 8 * (ks >> 1) + 2 * t + (ks & 1);
            const double* bt = sT + k * EU_LDT + g;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const double b = bt[8 * j];
#pragma unroll
                for (int i = 0; i < RT; ++i) dmma8x8x4(acc[i][j][0], acc[i][j][1], a[i][ks], b);
            }
        }
        // epilogue: G = gain (+ the Q[:, s] term on gauged rows, da.py:117-121), O = old outflow + gain
#pragma unroll
        for (int i = 0; i < RT; ++i) {
            if (rows[i] >= n) continue;
            const double qg = gi[i] >= 0 ? qs[gi[i]] : 0.0;
            const double* wr = W + (size_t)(gi[i] >= 0 ? gi[i] : 0) * M;
            const unsigned ra = stage0 + (buf * TR + 8 * i + g) * EU_RS + t * 16;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int col = 8 * j + 2 * t;
                if (col >= ld) continue;
                double2 gn = make_double2(col < M ? acc[i][j][0] : 0.0, col + 1 < M ? acc[i][j][1] : 0.0);
                if (gi[i] >= 0) {
                    if (col < M) gn.x += qg * wr[col];
                    if (col + 1 < M) gn.y += qg * wr[col + 1];
                }
                if (O) {
                    double2 o;
                    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(o.x), "=d"(o.y) : "r"(ra + j * 64));
                    o.x += gn.x; o.y += gn.y;
                    *reinterpret_cast<double2*>(O + (size_t)rows[i] * ld + col) = o;
                }
                if (G) *reinterpret_cast<double2*>(G + (size_t)rows[i] * ld + col) = gn;
            }
        }
        __syncwarp();                                 // everyone is done with this buffer before it is refilled
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
}

// inflow part of _apply_gain (nutils.py:116-134, da.py:125): I[k] += sum of the gains of the reaches
// draining into k (self-loops excluded).  One thread per (row with upstream reaches, member pair): `inner` lists
// those rows, so no thread is spent on a headwater (half of a river network).
__global__ void __launch_bounds__(256)
inflow_gain_kernel(const int32_t* __restrict__ inner, long long n_inner, const int32_t* __restrict__ up_off,
                   const int32_t* __restrict__ up_pos, const double* __restrict__ G, double* __restrict__ I, int ld)
{
    const int half = ld >> 1;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= n_inner * half) return;
    const long long e = gid / half;
    const int col = (int)(gid - e * half) * 2;
    const long long k = inner[e];
    const int u0 = up_off[k], u1 = up_off[k + 1];
    double2* ip = reinterpret_cast<double2*>(I + (size_t)k * ld + col);
    double2 i = *ip;
    double2 s = make_double2(0.0, 0.0);
    for (int u = u0; u < u1; ++u) {
        const double2 v = *reinterpret_cast<const double2*>(G + (size_t)up_pos[u] * ld + col);
        s.x += v.x; s.y += v.y;
    }
    i.x += s.x; i.y += s.y;
    *ip = i;
}

// The same update when the forecast inflows ARE the sums of the upstream forecast outflows (true right after a routing
// step: nutils.py:84-85 builds i_t_next that way): i + N gain = N (o + gain), so the posterior inflows are rebuilt from
// the posterior outflows and the gains never go to memory.
// `rec` packs what a row needs into one 16-byte record {row, up to three upstream rows (-1: none)} -- one load between
// the thread and its outflow rows instead of the chain inner -> up_off -> up_pos; rec.w == -2 marks a confluence of more
// than three reaches, which takes the lists.  Two rows per thread, all loads in flight before the first add.
__global__ void __launch_bounds__(256)
inflow_rebuild_kernel(const int4* __restrict__ rec, long long n_inner, const int32_t* __restrict__ up_off,
                      const int32_t* __restrict__ up_pos, const double* __restrict__ O, double* __restrict__ I, int ld)
{
    const int half = ld >> 1;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long pairs = (n_inner + 1) >> 1;
    if (gid >= pairs * half) return;
    const long long e0 = (gid / half) * 2;
    const int col = (int)(gid % half) * 2;
    int4 r[2];
#pragma unroll
    for (int q = 0; q < 2; ++q) r[q] = e0 + q < n_inner ? __ldg(rec + e0 + q) : make_int4(-1, -1, -1, -1);
    double2 v[2][3];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        const int u[3] = {r[q].y, r[q].z, r[q].w};
#pragma unroll
        for (int j = 0; j < 3; ++j)
            v[q][j] = u[j] >= 0 ? __ldcg(reinterpret_cast<const double2*>(O + (size_t)u[j] * ld + col)) : make_double2(0.0, 0.0);
    }
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        if (r[q].x < 0) continue;
        double2 s = v[q][0];
        if (r[q].z >= 0) { s.x += v[q][1].x; s.y += v[q][1].y; }
        if (r[q].w >= 0) { s.x += v[q][2].x; s.y += v[q][2].y; }
        if (r[q].w == -2) {
            for (int u = up_off[r[q].x] + 2; u < up_off[r[q].x + 1]; ++u) {
                const double2 x = __ldcg(reinterpret_cast<const double2*>(O + (size_t)up_pos[u] * ld + col));
                s.x += x.x; s.y += x.y;
            }
        }
        __stcg(reinterpret_cast<double2*>(I + (size_t)r[q].x * ld + col), s);
    }
}

inline unsigned nblk(long long work, int threads) { return (unsigned)((work + threads - 1) / threads); }

// Hydrographs of txh_run_assimilating_rec at an update: the forecast of the recorded rows (prior_out) and what the
// update makes of them (post_out), o + (o - mean) T + qs_g W_g [row gauged] -- the rows of enkf_update_kernel, for a
// few rows and in plain FP64, read from O while it still holds the forecast.
// Used where the update is applied by the stand-alone kernels (TXH_ENKF_FUSE_LOAD=0, M > 64, the lane kernel, the update
// after the last window); where the next window applies it, that launch records the rows itself (record_posterior,
// txh_window.cu).  A CTA holds T in shared memory (M <= 64) and the anomalies of RG rows: one thread per (row, member).

__global__ void __launch_bounds__(256)
enkf_record_kernel(const double* __restrict__ O, int ld, int M, const double* __restrict__ mean,
                   const double* __restrict__ T, const int32_t* __restrict__ gauge_of_pos, const double* __restrict__ qs,
                   const double* __restrict__ W, const int32_t* __restrict__ rec_pos, int rec_count,
                   double* __restrict__ prior_out, double* __restrict__ post_out)
{
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    extern __shared__ double rs_sm[];
    const int tid = threadIdx.x;
    const int Mc = M < 256 ? M : 256;                 // threads per row
    const int RG = 256 / Mc;                          // rows per pass
    const int q = tid / Mc, cl = tid - q * Mc;
    const bool stage_a = M <= 4096, stage_t = M <= 64;
    double* sa = rs_sm;                               // [RG][M] anomalies o - mean
    double* sT = rs_sm + (stage_a ? RG * M : 0);      // [M][M]
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (stage_t)
        for (int e = tid; e < M * M; e += blockDim.x) sT[e] = __ldcg(T + e);
    for (int k0 = blockIdx.x * RG; k0 < rec_count; k0 += gridDim.x * RG) {
        const int k = k0 + q;
        const bool on = q < RG && k < rec_count;
        const int pos = on ? __ldg(rec_pos + k) : 0;
        const double* o = O + (size_t)pos * ld;
        const double mu = on ? __ldcg(mean + pos) : 0.0;
        __syncthreads();                              // the previous pass is done with sa (and T is staged)
        if (on && stage_a)
            for (int c = cl; c < M; c += Mc) sa[q * M + c] = __ldcg(o + c) - mu;
        __syncthreads();
        if (!on) continue;
        const int gi = __ldg(gauge_of_pos + pos);
        for (int c = cl; c < M; c += Mc) {
            const double oc = __ldcg(o + c);
            const size_t at = (size_t)k * M + c;
            if (prior_out) prior_out[at] = oc;
            if (!post_out) continue;
            double g = 0.0;
            for (int j = 0; j < M; ++j) {
                const double a = stage_a ? sa[q * M + j] : __ldcg(o + j) - mu;
                g = fma(a, stage_t ? sT[j * M + c] : __ldcg(T + (size_t)j * M + c), g);
            }
            if (gi >= 0) g += __ldcg(qs + gi) * __ldcg(W + (size_t)gi * M + c);
            post_out[at] = oc + g;
        }
    }
}

// ---- ensemble Kalman smoother of recorded hydrographs (txh_enks_smooth) ------------------------------------------------
// An update maps a past ensemble X to X (I + C T_u), C = I - 11^T/M the centring matrix.  Products keep that form:
//     (I + C T1)(I + C T2) = I + C compose(T1, T2),   compose(T1, T2) = T1 + T2 + (T1 C) T2
// so the updates a slot receives collapse into one cumulative transform.  Stage (a) forms one per range of updates
// [a, b] the slots need (at most two per first update a: a lag that is not a multiple of `every` splits a group), from
// in-block prefix and suffix products over blocks of Bs = ceil(sqrt(nupd)) updates: a range inside one block is a
// prefix or a suffix of it or a chain of at most Bs - 2 products, any other range is a suffix, the totals of the blocks
// in between and a prefix.  The longest chain of dependent products is about 2 sqrt(nupd) (26 at 168 updates) instead
// of nupd.  Stage (b) streams the recorded rows once: X + (X - mean) T_cum on the tensor cores.
constexpr int SM_K = 16;

// out = T1 + T2 + (T1 - rowmean(T1)) T2 for M x M row-major matrices in global memory (written by this CTA or an
// earlier launch), by a whole CTA of 256 threads: 64 x 64 output tiles, 8 warps x 16 x 32 DMMA tiles, k tiles of 16.
// out must not alias T1 or T2.  mu: M doubles of shared memory.  Ends in a barrier: out is visible to the CTA.
__device__ void enks_compose(const double* T1, const double* T2, double* out, int M, double* mu, double* sA, double* sB)
{
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int wm = (warp >> 1) * 16, wn = (warp & 1) * 32;
    for (int i = warp; i < M; i += 8) {
        double s = 0.0;
        for (int c = lane; c < M; c += 32) s += __ldcg(T1 + (size_t)i * M + c);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) mu[i] = s / M;
    }
    __syncthreads();
    for (int i0 = 0; i0 < M; i0 += 64)
        for (int j0 = 0; j0 < M; j0 += 64) {
            double acc[2][4][2];
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
            for (int k0 = 0; k0 < M; k0 += SM_K) {
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int e = tid + 256 * u;
                    const int r = e / SM_K, k = e % SM_K, gi = i0 + r, gk = k0 + k;
                    sA[r * (SM_K + 1) + k] = (gi < M && gk < M) ? __ldcg(T1 + (size_t)gi * M + gk) - mu[gi] : 0.0;
                    const int kb = e / 64, c = e % 64, gkb = k0 + kb, gc = j0 + c;
                    sB[kb * 65 + c] = (gkb < M && gc < M) ? __ldcg(T2 + (size_t)gkb * M + gc) : 0.0;
                }
                __syncthreads();
#pragma unroll
                for (int kk = 0; kk < SM_K; kk += 4) {
                    double a[2], b[4];
#pragma unroll
                    for (int i = 0; i < 2; ++i) a[i] = sA[(wm + 8 * i + g) * (SM_K + 1) + kk + t];
#pragma unroll
                    for (int j = 0; j < 4; ++j) b[j] = sB[(kk + t) * 65 + wn + 8 * j + g];
#pragma unroll
                    for (int i = 0; i < 2; ++i)
#pragma unroll
                        for (int j = 0; j < 4; ++j) dmma8x8x4(acc[i][j][0], acc[i][j][1], a[i], b[j]);
                }
                __syncthreads();
            }
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j)
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        const int gi = i0 + wm + 8 * i + g, gc = j0 + wn + 8 * j + 2 * t + c;
                        if (gi < M && gc < M) {
                            const size_t at = (size_t)gi * M + gc;
                            out[at] = __ldcg(T1 + at) + __ldcg(T2 + at) + acc[i][j][c];
                        }
                    }
        }
    __syncthreads();
}

__device__ void enks_copy(const double* src, double* dst, size_t count)
{
    for (size_t e = threadIdx.x; e < count; e += blockDim.x) dst[e] = __ldcg(src + e);
    __syncthreads();
}

// stage (a), part 1: CTA (block, 0) forms the prefix products P[u] = T_b0 o ... o T_u of its block of updates, CTA
// (block, 1) the suffix products S[u] = T_u o ... o T_b1
__global__ void __launch_bounds__(256)
enks_block_scan_kernel(const double* __restrict__ Th, int M, int nupd, int Bs, double* P, double* S)
{
    extern __shared__ double enks_mu[];
    __shared__ double sA[64 * (SM_K + 1)], sB[SM_K * 65];
    const size_t MM = (size_t)M * M;
    const int u0 = blockIdx.x * Bs, u1 = min(nupd, u0 + Bs) - 1;
    if (blockIdx.y == 0) {
        enks_copy(Th + u0 * MM, P + u0 * MM, MM);
        for (int u = u0 + 1; u <= u1; ++u) enks_compose(P + (u - 1) * MM, Th + u * MM, P + u * MM, M, enks_mu, sA, sB);
    } else {
        enks_copy(Th + u1 * MM, S + u1 * MM, MM);
        for (int u = u1 - 1; u >= u0; --u) enks_compose(Th + u * MM, S + (u + 1) * MM, S + u * MM, M, enks_mu, sA, sB);
    }
}

// the range of updates [a, b] of slots whose first update is a; which = 1: the longer of the two a lag that is not a
// multiple of `every` gives (b one further).  -1: no update reaches the slot.
__device__ __forceinline__ void enks_range(long long a, int which, int nupd, long long lag_q, int* b_out)
{
    const long long bmin = min((long long)nupd - 1, a + lag_q - 1);
    const long long b = min((long long)nupd - 1, a + lag_q - 1 + which);
    *b_out = (b < a || (which == 1 && b == bmin)) ? -1 : (int)b;
}

// stage (a), part 2: CTA r forms the cumulative transform Tc[r] of the range (a = r / 2, which = r % 2), ping-ponging
// between Tc[r] and the scratch X[r] so that the last product lands in Tc[r]
__global__ void __launch_bounds__(256)
enks_range_kernel(const double* __restrict__ Th, int M, int nupd, int Bs, long long lag_q, const double* P,
                  const double* S, double* Tc, double* X)
{
    extern __shared__ double enks_mu[];
    __shared__ double sA[64 * (SM_K + 1)], sB[SM_K * 65];
    const size_t MM = (size_t)M * M;
    const int r = blockIdx.x, a = r >> 1;
    int b;
    enks_range(a, r & 1, nupd, lag_q, &b);
    if (b < 0) return;
    const int ka = a / Bs, kb = b / Bs;
    const double* first;
    int n;                                            // products after `first`
    if (ka == kb && a == ka * Bs) { first = P + b * MM; n = 0; }
    else if (ka == kb && b == min(nupd, (ka + 1) * Bs) - 1) { first = S + a * MM; n = 0; }
    else if (ka == kb) { first = Th + a * MM; n = b - a; }
    else { first = S + a * MM; n = kb - ka; }
    double* dst = Tc + r * MM;
    if (n == 0) { enks_copy(first, dst, MM); return; }
    const double* cur = first;
    for (int i = 0; i < n; ++i) {
        const double* rhs = ka == kb ? Th + (a + 1 + i) * MM                          // chain inside the block
                                     : (i < n - 1 ? S + (size_t)(ka + 1 + i) * Bs * MM : P + b * MM);   // block totals, prefix
        double* o = ((n - 1 - i) & 1) ? X + r * MM : dst;
        enks_compose(cur, rhs, o, M, enks_mu, sA, sB);
        cur = o;
    }
}

// stage (b): out = X + (X - mean) Tc for every recorded row, a copy for slots no update reaches.  Work items are
// (slot, 128-row tile), CTA b takes a contiguous run of them and stages Tc only when the range changes.  A warp owns 16
// rows (two 8-row MMA tiles) as in enkf_update_kernel: its lanes hold the members 8j+2t, 8j+2t+1 of a row, which are
// both the permuted A fragment and the C fragment positions of output tile j, so X + gain needs no second read when
// M <= 64.  The row mean is the sum of a lane's 16 values over the 4 lanes of the row.
constexpr int ES_ROWS = 16 * 8;

template <bool ONE>                               // ONE: M <= 64, a single member block
__global__ void __launch_bounds__(256)
enks_apply_kernel(const double* __restrict__ rec, double* __restrict__ out, const double* __restrict__ Tc, int M, int nupd,
                  long long every, long long lag_c, long long rec_every, long long rec_count, long long nitems,
                  long long per_cta, int tiles_per_slot, int resident)
{
    extern __shared__ double sT_all[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int nkc = ONE ? 1 : (M + 63) / 64;
    const bool vec = (M & 1) == 0;
    const size_t MM = (size_t)M * M;
    int staged = -1;
    const long long it0 = (long long)blockIdx.x * per_cta, it1 = min(nitems, it0 + per_cta);
    for (long long it = it0; it < it1; ++it) {
        const long long j = it / tiles_per_slot;
        const long long tile = it - j * tiles_per_slot;
        const long long s = (j + 1) * rec_every, a = s / every;
        // updates a .. b reach the slot, b = the last with (b+1) every <= s + lag; r as enks_range_kernel numbers them
        int r = -1;
        const long long b = min((long long)nupd - 1, (s + lag_c) / every - 1);
        if (a < nupd && b >= a) r = (int)(2 * a + (b > min((long long)nupd - 1, a + lag_c / every - 1) ? 1 : 0));
        const long long lr0 = tile * ES_ROWS + warp * 16;                    // this warp's rows in the slot
        const double* xs = rec + (size_t)j * rec_count * M;
        double* os = out + (size_t)j * rec_count * M;
        if (r < 0) {
            for (long long q = lr0; q < lr0 + 16 && q < rec_count; ++q)
                for (int c = lane; c < M; c += 32) __stcs(os + q * M + c, __ldcs(xs + q * M + c));
            continue;
        }
        if (resident && r != staged) {
            __syncthreads();
            for (int blk = 0; blk < nkc * nkc; ++blk)
                for (int e = tid; e < 64 * 64; e += 256) {
                    const int k = e >> 6, c = e & 63, gk = (blk / nkc) * 64 + k, gc = (blk % nkc) * 64 + c;
                    sT_all[blk * 64 * EU_LDT + k * EU_LDT + c] = (gk < M && gc < M) ? __ldg(Tc + r * MM + (size_t)gk * M + gc) : 0.0;
                }
            __syncthreads();
            staged = r;
        }
        const long long rows[2] = {lr0 + g, lr0 + 8 + g};
        // this lane's members of chunk kc of its two rows (0 beyond the matrix)
        auto load_chunk = [&](int kc, double (&x)[2][16]) {
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const bool ok = rows[i] < rec_count;
                const double* xr = xs + (size_t)(ok ? rows[i] : 0) * M;
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) {
                    const int k = kc * 64 + 8 * jj + 2 * t;
                    double x0 = 0.0, x1 = 0.0;
                    if (ok && vec && k < M) {
                        const double2 v = __ldcs(reinterpret_cast<const double2*>(xr + k));
                        x0 = v.x; x1 = v.y;
                    } else if (ok) {
                        if (k < M) x0 = __ldcs(xr + k);
                        if (k + 1 < M) x1 = __ldcs(xr + k + 1);
                    }
                    x[i][2 * jj] = x0; x[i][2 * jj + 1] = x1;
                }
            }
        };
        double x[2][16], mu[2] = {0.0, 0.0};
        for (int kc = 0; kc < nkc; ++kc) {
            load_chunk(kc, x);
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int q = 0; q < 16; ++q) mu[i] += x[i][q];
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            mu[i] += __shfl_xor_sync(0xffffffffu, mu[i], 1);
            mu[i] += __shfl_xor_sync(0xffffffffu, mu[i], 2);
            mu[i] /= M;
        }
        for (int cg = 0; cg < nkc; ++cg) {
            const int njt = min(8, (M - cg * 64 + 7) >> 3);
            double acc[2][8][2];
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) acc[i][jj][0] = acc[i][jj][1] = 0.0;
            for (int kc = 0; kc < nkc; ++kc) {
                if (nkc > 1) load_chunk(kc, x);
                const double* sT = sT_all + (resident ? (kc * nkc + cg) * 64 * EU_LDT : 0);
                if (!resident) {
                    __syncthreads();
                    for (int e = tid; e < 64 * 64; e += 256) {
                        const int k = e >> 6, c = e & 63, gk = kc * 64 + k, gc = cg * 64 + c;
                        sT_all[k * EU_LDT + c] = (gk < M && gc < M) ? __ldg(Tc + r * MM + (size_t)gk * M + gc) : 0.0;
                    }
                    __syncthreads();
                }
#pragma unroll
                for (int ks = 0; ks < 16; ++ks) {
                    const int k = 8 * (ks >> 1) + 2 * t + (ks & 1);
                    const bool in = kc * 64 + k < M;          // the anomaly is formed here: x stays for the epilogue
                    const double a0 = in ? x[0][ks] - mu[0] : 0.0, a1 = in ? x[1][ks] - mu[1] : 0.0;
                    const double* bt = sT + k * EU_LDT + g;
#pragma unroll
                    for (int jj = 0; jj < 8; ++jj)
                        if (jj < njt) {
                            const double bv = bt[8 * jj];
                            dmma8x8x4(acc[0][jj][0], acc[0][jj][1], a0, bv);
                            dmma8x8x4(acc[1][jj][0], acc[1][jj][1], a1, bv);
                        }
                }
            }
            if (nkc > 1) load_chunk(cg, x);
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                if (rows[i] >= rec_count) continue;
                double* orow = os + (size_t)rows[i] * M;
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) {
                    const int col = cg * 64 + 8 * jj + 2 * t;
                    if (vec && col < M) {
                        __stcs(reinterpret_cast<double2*>(orow + col),
                               make_double2(x[i][2 * jj] + acc[i][jj][0], x[i][2 * jj + 1] + acc[i][jj][1]));
                    } else {
                        if (col < M) __stcs(orow + col, x[i][2 * jj] + acc[i][jj][0]);
                        if (col + 1 < M) __stcs(orow + col + 1, x[i][2 * jj + 1] + acc[i][jj][1]);
                    }
                }
            }
        }
    }
}

}  // namespace

cudaError_t launch_dgemm(int transA, int transB, int M, int N, int K, double alpha, const double* A, int lda,
                         const double* B, int ldb, double beta, double* C, int ldc, cudaStream_t st)
{
    if (M <= 0 || N <= 0) return cudaSuccess;
    dim3 grid((N + GB_N - 1) / GB_N, (M + GB_M - 1) / GB_M);
    dgemm_kernel<<<grid, 256, 0, st>>>(transA, transB, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, K > 0 ? K : 1, 0,
                                       C, ldc);
    count_launch();
    return cudaGetLastError();
}

// C = alpha op(A) op(B) + beta Cin   (Cin may differ from C)
cudaError_t launch_dgemm_ex(int transA, int transB, int M, int N, int K, double alpha, const double* A, int lda,
                            const double* B, int ldb, double beta, const double* Cin, int ldcin, double* C, int ldc,
                            cudaStream_t st)
{
    if (M <= 0 || N <= 0) return cudaSuccess;
    dim3 grid((N + GB_N - 1) / GB_N, (M + GB_M - 1) / GB_M);
    dgemm_kernel<<<grid, 256, 0, st>>>(transA, transB, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, K > 0 ? K : 1, 0,
                                       Cin, ldcin);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_dgemm_splitk(int transA, int transB, int M, int N, int K, const double* A, int lda, const double* B,
                                int ldb, double* Cpart, int ldc, int nsplit, long long pstride, cudaStream_t st)
{
    if (M <= 0 || N <= 0 || nsplit < 1) return cudaSuccess;
    int kchunk = (K + nsplit - 1) / nsplit;
    kchunk = (kchunk + GB_K - 1) / GB_K * GB_K;
    dim3 grid((N + GB_N - 1) / GB_N, (M + GB_M - 1) / GB_M, nsplit);
    dgemm_kernel<<<grid, 256, 0, st>>>(transA, transB, M, N, K, 1.0, A, lda, B, ldb, 0.0, Cpart, ldc, kchunk, pstride,
                                       Cpart, ldc);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_innovation_cat(double* HX, const double* O, int ldo, const double* Zp, const double* mean,
                                  const int32_t* obs_pos, const double* dinv_diag, int m, int Mt, double* Bc, double* Y,
                                  cudaStream_t st)
{
    innovation_cat_kernel<<<nblk((long long)m * Mt, 256), 256, 0, st>>>(HX, O, ldo, Zp, mean, obs_pos, dinv_diag, m, Mt, Bc, Y);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_chol_solve_small(const double* Cpart, int nsplit, long long pstride, int Mt, double shift, double* Z,
                                    int* info, cudaStream_t st)
{
    if (nsplit != CS_NSPLIT || Mt > 128) return cudaErrorInvalidValue;
    const int MT = Mt <= 64 ? 64 : (Mt <= 96 ? 96 : 128);
    const int ncta = (Mt + 7) / 8;                      // 8 right-hand-side columns per CTA
    const size_t smem_b = ((size_t)MT * (MT + 1) + (size_t)MT * 9 + MT + (size_t)(MT / 8) * 72) * sizeof(double);
    void (*kern)(const double*, long long, int, double, double*, int*) =
        MT == 64 ? chol_solve_blocked_kernel<64> : (MT == 96 ? chol_solve_blocked_kernel<96> : chol_solve_blocked_kernel<128>);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b);
    if (e != cudaSuccess) return e;
    kern<<<ncta, 256, smem_b, st>>>(Cpart, pstride, Mt, shift, Z, info);
    count_launch();
    return cudaGetLastError();
}

// The ensemble-space system in one cluster launch (Mt <= 64, D diagonal): HX (gathered from O when O != nullptr), T, W.
// 16 CTAs per cluster where the device takes it (non-portable size), else 8.
cudaError_t launch_enkf_small_system(double* HX, const double* O, int ldo, const double* Zp, const double* mean,
                                     const int32_t* obs_pos, const double* dinv_diag, int m, int Mt, double shift,
                                     double* T, double* W, int* info, cudaStream_t st)
{
    if (Mt > 64 || Mt < 1 || m < 1) return cudaErrorInvalidValue;
    auto k16 = enkf_small_system_kernel<16>;
    auto k8 = enkf_small_system_kernel<8>;
    static int nc = 0;
    cudaError_t e;
    if (nc == 0) {
        if ((e = cudaFuncSetAttribute(k8, cudaFuncAttributeMaxDynamicSharedMemorySize, SS_SMEM)) != cudaSuccess) return e;
        nc = 8;
        int want = 16;
        if (const char* k = getenv("TXH_SS_CLUSTER")) want = atoi(k);
        if (want >= 16 && cudaFuncSetAttribute(k16, cudaFuncAttributeMaxDynamicSharedMemorySize, SS_SMEM) == cudaSuccess &&
            cudaFuncSetAttribute(k16, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess) {
            cudaLaunchConfig_t q{};
            q.gridDim = dim3(16); q.blockDim = dim3(256); q.dynamicSmemBytes = SS_SMEM;
            cudaLaunchAttribute at{};
            at.id = cudaLaunchAttributeClusterDimension; at.val.clusterDim.x = 16; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
            q.attrs = &at; q.numAttrs = 1;
            int ncl = 0;
            if (cudaOccupancyMaxActiveClusters(&ncl, k16, &q) == cudaSuccess && ncl >= 1) nc = 16;
        }
        cudaGetLastError();
    }
    static const char* trace_file = getenv("TXH_SS_TRACE");
    unsigned long long* d_trace = nullptr;
    if (trace_file && *trace_file) {
        if ((e = cudaMalloc((void**)&d_trace, 16 * 8 * sizeof(unsigned long long))) != cudaSuccess) return e;
        cudaMemsetAsync(d_trace, 0, 16 * 8 * sizeof(unsigned long long), st);
    }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(nc); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = SS_SMEM; cfg.stream = st;
    static const bool pdl = [] { const char* k = getenv("TXH_PDL"); return !(k && atoi(k) == 0); }();
    cudaLaunchAttribute attr[2]{};
    attr[0].id = cudaLaunchAttributeClusterDimension; attr[0].val.clusterDim.x = nc; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization; attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = pdl ? 2 : 1;
    e = cudaLaunchKernelEx(&cfg, nc == 16 ? k16 : k8, HX, O, ldo, Zp, mean, obs_pos, dinv_diag, m, Mt, shift, T, W, info, d_trace);
    count_launch();
    if (e == cudaSuccess) e = cudaGetLastError();
    if (d_trace) {
        // development aid: per-CTA phase stamps (ns relative to the first) appended to the file, synchronous
        unsigned long long h[16 * 8];
        cudaMemcpyAsync(h, d_trace, sizeof(h), cudaMemcpyDeviceToHost, st);
        cudaStreamSynchronize(st);
        cudaFree(d_trace);
        if (FILE* fp = fopen(trace_file, "a")) {
            unsigned long long t0 = ~0ull;
            for (int r = 0; r < nc; ++r) if (h[r * 8] && h[r * 8] < t0) t0 = h[r * 8];
            for (int r = 0; r < nc; ++r) {
                for (int i = 0; i < 8; ++i) fprintf(fp, "%lld ", h[r * 8 + i] ? (long long)(h[r * 8 + i] - t0) : -1ll);
                fprintf(fp, "\n");
            }
            fprintf(fp, "\n");
            fclose(fp);
        }
    }
    return e;
}

cudaError_t launch_woodbury_assemble(const double* Cpart, int nsplit, long long pstride, int Mt, double shift, double* Cf,
                                     double* C1, cudaStream_t st)
{
    woodbury_assemble_kernel<<<nblk((long long)Mt * 2 * Mt, 256), 256, 0, st>>>(Cpart, nsplit, pstride, Mt, shift, Cf, C1);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_enkf_stats(const double* X, int ld, int M, int64_t n, double scale, const int32_t* gauge_of_pos,
                              double* rowsum, double* HX, cudaStream_t st)
{
    enkf_stats_kernel<<<nblk(n, 8), 256, 0, st>>>(X, ld, M, n, scale, gauge_of_pos, rowsum, HX);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_innovation(const double* HX, const double* Zp, const double* mean_obs, int m, int M, double* HA,
                              double* dz, cudaStream_t st)
{
    innovation_kernel<<<nblk((long long)m * M, 256), 256, 0, st>>>(HX, Zp, mean_obs, m, M, HA, dz);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_innov_cov_finish(double* S, const double* qs, const double* R, int m, double scale, cudaStream_t st)
{
    innov_cov_finish_kernel<<<nblk((long long)m * m, 256), 256, 0, st>>>(S, qs, R, m, scale);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_spd_solve(double* S, double* B, int m, int k, int* info, cudaStream_t st)
{
    if (m <= 48) {
        spd_solve_kernel<<<1, 1024, 0, st>>>(S, B, m, k, info);
        count_launch();
        return cudaGetLastError();
    }
    // blocked right-looking Cholesky, panels of PB columns: factor the diagonal block, solve the panel below
    // and the matching rows of B, update the trailing matrix and the rest of B on the tensor cores
    cudaError_t e;
    for (int j0 = 0; j0 < m; j0 += PB) {
        const int nb = m - j0 < PB ? m - j0 : PB;
        const int below = m - j0 - nb;
        const int nslab = (below + 63) / 64, ncol = (k + 63) / 64;
        chol_panel_kernel<<<1 + nslab + ncol, 64, 0, st>>>(S, m, B, k, j0, nb, nslab, info);
        count_launch();
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        if (below > 0) {
            const double* L21 = S + (size_t)(j0 + nb) * m + j0;
            double* S22 = S + (size_t)(j0 + nb) * m + (j0 + nb);
            if ((e = launch_dgemm(0, 1, below, below, nb, -1.0, L21, m, L21, m, 1.0, S22, m, st)) != cudaSuccess) return e;
            if ((e = launch_dgemm(0, 0, below, k, nb, -1.0, L21, m, B + (size_t)j0 * k, k, 1.0, B + (size_t)(j0 + nb) * k, k, st)) != cudaSuccess) return e;
        }
    }
    // backward substitution L^T X = Y, panels from the bottom: solve the block, then update the rows above
    const int last0 = ((m - 1) / PB) * PB;
    for (int j0 = last0; j0 >= 0; j0 -= PB) {
        const int nb = m - j0 < PB ? m - j0 : PB;
        chol_back_kernel<<<(k + 63) / 64, 64, 0, st>>>(S, m, B, k, j0, nb);
        count_launch();
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        if (j0 > 0) {
            // Y[0:j0] -= L[j0:j0+nb, 0:j0]^T Z1
            if ((e = launch_dgemm(1, 0, j0, k, nb, -1.0, S + (size_t)j0 * m, m, B + (size_t)j0 * k, k, 1.0, B, k, st)) != cudaSuccess) return e;
        }
    }
    return cudaSuccess;
}

cudaError_t launch_enkf_update(const double* Xall, int ldx, int Mtot, const double* mean, const double* T, int ldt,
                               int Mloc, double* O, double* G, int ld, int64_t n, const int32_t* gauge_of_pos,
                               const double* qs, const double* W, int col0, int num_sms, int Mb, long long blk_stride,
                               cudaStream_t st, const PeerBlocks* peers, double* Oout)
{
    long long tiles = (n + EU_ROWS - 1) / EU_ROWS;
    PeerBlocks pb{};
    if (peers) pb = *peers;
    if (!Oout) Oout = O;
    if (!peers && Mtot == Mloc && Mtot <= 64 && ld <= 64 && ldx == ld && col0 == 0) {
        constexpr int RT = EU64_RT;
        tiles = (n + 8 * RT - 1) / (8 * RT);
        tiles = (tiles + 16 / RT - 1) / (16 / RT);             // CTAs' worth of warp tiles
        cudaError_t e = cudaFuncSetAttribute(enkf_update64_kernel<RT>, cudaFuncAttributeMaxDynamicSharedMemorySize, EU64_SMEM);
        if (e != cudaSuccess) return e;
        const long long grid2 = tiles < (long long)num_sms ? tiles : (long long)num_sms;
        enkf_update64_kernel<RT><<<(unsigned)grid2, 512 / RT, EU64_SMEM, st>>>(Xall, Mtot, mean, T, ldt, O, G, ld, n,
                                                                               gauge_of_pos, qs, W);
        count_launch();
        return cudaGetLastError();
    }
    long long grid = tiles < (long long)num_sms ? tiles : (long long)num_sms;
    const int nkc = (Mtot + 63) / 64;
    const int resident = (ld <= 64 && nkc <= 6) ? 1 : 0;
    const size_t smem = (size_t)(resident ? nkc : 1) * 64 * EU_LDT * sizeof(double);
    cudaError_t e = cudaFuncSetAttribute(enkf_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    enkf_update_kernel<<<(unsigned)grid, EU_WARPS * 32, smem, st>>>(Xall, ldx, Mtot, mean, T, ldt, Mloc, O, Oout, G, ld, n,
                                                                    gauge_of_pos, qs, W, col0, resident, Mb, blk_stride, pb);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_inflow_rebuild(const int4* rec, int64_t n_inner, const int32_t* up_off, const int32_t* up_pos,
                                  const double* O, double* I, int ld, cudaStream_t st)
{
    if (n_inner == 0) return cudaSuccess;
    inflow_rebuild_kernel<<<nblk(((n_inner + 1) >> 1) * (ld >> 1), 256), 256, 0, st>>>(rec, n_inner, up_off, up_pos, O, I, ld);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_enkf_record(const double* O, int ld, int M, const double* mean, const double* T,
                               const int32_t* gauge_of_pos, const double* qs, const double* W, const int32_t* rec_pos,
                               int rec_count, double* prior_out, double* post_out, cudaStream_t st)
{
    const long long work = (long long)rec_count * M;
    if (work == 0 || (!prior_out && !post_out)) return cudaSuccess;
    static const bool pdl = [] { const char* k = getenv("TXH_PDL"); return !(k && atoi(k) == 0); }();
    const int Mc = M < 256 ? M : 256, RG = 256 / Mc;
    const size_t smem = sizeof(double) * ((M <= 4096 ? (size_t)RG * M : 0) + (M <= 64 ? (size_t)M * M : 0));
    const int grid = (int)((rec_count + RG - 1) / RG);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr{};
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr.val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = &attr; cfg.numAttrs = pdl ? 1 : 0;
    cudaError_t e = cudaLaunchKernelEx(&cfg, enkf_record_kernel, O, ld, M, mean, T, gauge_of_pos, qs, W, rec_pos, rec_count,
                                       prior_out, post_out);
    count_launch();
    return e != cudaSuccess ? e : cudaGetLastError();
}

cudaError_t launch_inflow_gain(const int32_t* inner, int64_t n_inner, const int32_t* up_off, const int32_t* up_pos,
                               const double* G, double* I, int ld, cudaStream_t st)
{
    if (n_inner == 0) return cudaSuccess;
    inflow_gain_kernel<<<nblk(n_inner * (ld >> 1), 256), 256, 0, st>>>(inner, n_inner, up_off, up_pos, G, I, ld);
    count_launch();
    return cudaGetLastError();
}

// work: P [nupd], S [nupd], Tc [2 nupd], X [2 nupd] matrices of M x M (txh_enks_work_size)
cudaError_t launch_enks_smooth(int M, int nupd, long long every, const double* T_hist, long long nslots, long long rec_count,
                               long long rec_every, long long lag, const double* rec, double* out, double* work,
                               cudaStream_t st)
{
    if (nslots == 0 || rec_count == 0) return cudaSuccess;
    const size_t MM = (size_t)M * M;
    double *P = work, *S = P + nupd * MM, *Tc = S + nupd * MM, *X = Tc + 2 * nupd * MM;
    if (lag == 0) nupd = 0;                               // nothing reaches any slot: stage (b) copies
    const long long lag_c = lag < (nupd + 1LL) * every ? lag : (nupd + 1LL) * every;   // beyond: the same ranges
    cudaError_t e;
    if (nupd > 0) {
        int Bs = 1;
        while ((long long)Bs * Bs < nupd) ++Bs;
        const size_t smem = sizeof(double) * M;
        enks_block_scan_kernel<<<dim3((nupd + Bs - 1) / Bs, 2), 256, smem, st>>>(T_hist, M, nupd, Bs, P, S);
        count_launch();
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        enks_range_kernel<<<2 * nupd, 256, smem, st>>>(T_hist, M, nupd, Bs, lag_c / every, P, S, Tc, X);
        count_launch();
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    const int nkc = (M + 63) / 64;
    const int resident = nkc <= 2 ? 1 : 0;               // every 64 x 64 block of Tc in shared memory (<= 135 KB)
    const size_t smem = (size_t)(resident ? nkc * nkc : 1) * 64 * EU_LDT * sizeof(double);
    auto kern = nkc == 1 ? enks_apply_kernel<true> : enks_apply_kernel<false>;
    if ((e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
    int dev = 0, num_sms = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
    if ((e = cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
    const int tiles_per_slot = (int)((rec_count + ES_ROWS - 1) / ES_ROWS);
    const long long nitems = nslots * tiles_per_slot;
    const long long want = (long long)num_sms * 2;      // 168-198 registers: one CTA of 8 warps per SM
    const long long grid = nitems < want ? nitems : want;
    const long long per_cta = (nitems + grid - 1) / grid;
    kern<<<(unsigned)((nitems + per_cta - 1) / per_cta), 256, smem, st>>>(
        rec, out, Tc, M, nupd, every, lag_c, rec_every, rec_count, nitems, per_cta, tiles_per_slot, resident);
    count_launch();
    return cudaGetLastError();
}

}  // namespace txh
