// txh_kf.cu -- glue kernels of the dense per-sub-basin Kalman filter (KalmanFilter.filter,
// tx_fast_hydrology/da.py:91-136) so that one update is a chain of launches with no host round trip:
//
//   X  = pack(P)                      columns of P ride as members          (launch_pack)
//   X  = A X                          nutils.py:148-154 per column          (init_inflows + routing launch)
//   X2 = pack(X^T)                    kf_repack_transposed_kernel
//   X2 = A X2                         second pass of _aqat_par, nutils.py:194-214
//   P- = unpack(X2) + Q, and the gauge slices P-[:, s], P-[s], P-[s][:, s] + R   kf_prior_finish_kernel
//   S^-1                              inverse_smem_kernel (np.linalg.inv, da.py:119)
//   K = P-[:, s] S^-1                 DMMA dgemm
//   dz = z - o[s], gain = K dz        kf_innovation_kernel, kf_gain_kernel  (da.py:112, 121)
//   P+ = P- - K P-[s]                 DMMA dgemm                            (da.py:122)
//   o += gain, i += sum of upstream gains                                   (apply_gain, nutils.py:116-134)
#include <cuda_runtime.h>

#include <cstdint>

#include "txh_kernels.cuh"

namespace txh {

namespace {

// X2[k][c] = X[pos_of_reach[c]][reach_of_pos[k]]  (= pack of the transposed unpacked matrix), pad columns zeroed
__global__ void __launch_bounds__(256)
kf_repack_transposed_kernel(const int32_t* __restrict__ reach_of_pos, const int32_t* __restrict__ pos_of_reach,
                            const double* __restrict__ X, double* __restrict__ X2, int n, int ld)
{
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)n * ld) return;
    const int k = (int)(gid / ld), c = (int)(gid - (long long)k * ld);
    X2[gid] = c < n ? X[(size_t)pos_of_reach[c] * ld + reach_of_pos[k]] : 0.0;
}

// P-[r][c] = X2[pos(r)][c] + Q[r][c], scattered on the way into the slices the update needs
__global__ void __launch_bounds__(256)
kf_prior_finish_kernel(const int32_t* __restrict__ reach_of_pos, const int32_t* __restrict__ pos_of_reach,
                       const int32_t* __restrict__ gauge_of_pos, const double* __restrict__ X2, int ld,
                       const double* __restrict__ Q, const double* __restrict__ R, int n, int m,
                       double* __restrict__ Pm, double* __restrict__ Ps, double* __restrict__ Prow, double* __restrict__ S)
{
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)n * n) return;
    const int k = (int)(gid / n), c = (int)(gid - (long long)k * n);
    const int r = reach_of_pos[k];
    const size_t e = (size_t)r * n + c;
    const double v = X2[(size_t)k * ld + c] + Q[e];
    Pm[e] = v;
    const int gr = gauge_of_pos[k], gc = gauge_of_pos[pos_of_reach[c]];
    if (gc >= 0) Ps[(size_t)r * m + gc] = v;
    if (gr >= 0) {
        Prow[(size_t)gr * n + c] = v;
        if (gc >= 0) S[(size_t)gr * m + gc] = v + R[(size_t)gr * m + gc];
    }
}

// dz[g] = z[g] - o[s][g]   (da.py:112; the model is single-member: column 0 of its state rows)
__global__ void kf_innovation_kernel(const int32_t* __restrict__ obs_pos, const double* __restrict__ z,
                                     const double* __restrict__ O, int ldo, int m, double* __restrict__ dz)
{
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g < m) dz[g] = z[g] - O[(size_t)obs_pos[g] * ldo];
}

// gain = K dz (da.py:121), in reach order and as a state row block for apply_gain
__global__ void __launch_bounds__(256)
kf_gain_kernel(const int32_t* __restrict__ reach_of_pos, const double* __restrict__ K, const double* __restrict__ dz,
               int n, int m, int ldg, double* __restrict__ gain, double* __restrict__ Gp)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int r = reach_of_pos[k];
    const double* row = K + (size_t)r * m;
    double s = 0.0;
    for (int g = 0; g < m; ++g) s += row[g] * dz[g];
    gain[r] = s;
    Gp[(size_t)k * ldg] = s;
    for (int c = 1; c < ldg; ++c) Gp[(size_t)k * ldg + c] = 0.0;
}

// In-place Gauss-Jordan inverse with partial pivoting (np.linalg.inv of da.py:119), one CTA: A <- inv(A).
// The matrix lives in shared memory when it fits (in_smem), else it is worked on where it is.  Two barriers
// per column: the elimination of column j also publishes column j + 1 as it will look afterwards, so every
// warp can find the next pivot on its own; rows are swapped as the pivots are chosen and the columns swapped
// back in reverse order at the end.
__device__ __forceinline__ void inverse_in_cta(double* __restrict__ A, int m, int in_smem, int* __restrict__ info, double* sm)
{
    double* colv = sm;                       // column j (of the rows as they are before the swap), double buffered
    double* prow = sm + 2 * m;               // scaled pivot row
    int* perm = reinterpret_cast<int*>(sm + 3 * m);
    double* a = in_smem ? sm + 4 * m : A;
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31;
    const int mm = m * m;
    if (in_smem) for (int e = tid; e < mm; e += nt) a[e] = A[e];
    __syncthreads();
    for (int i = tid; i < m; i += nt) colv[i] = a[(size_t)i * m];
    __syncthreads();
    // (row, column) of the elements this thread owns, advanced without divisions
    const int i0 = tid / m, c0 = tid - i0 * m, di = nt / m, dc = nt - di * m;
    for (int j = 0; j < m; ++j) {
        double* cv = colv + (j & 1) * m;
        double* cn = colv + ((j + 1) & 1) * m;
        // first row of maximal |a[i][j]|, i >= j (every warp finds it for itself)
        double bv = -1.0; int bi = j;
        for (int i = j + lane; i < m; i += 32) { const double v = fabs(cv[i]); if (v > bv) { bv = v; bi = i; } }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
        }
        const int pr = bi;
        double inv = 1.0;
        if (bv > 0.0) inv = 1.0 / cv[pr]; else if (tid == 0) *info = -(j + 1);   // negative: Gauss-Jordan pivot (txh_check)
        // swap rows j <-> pr, a[j][j] := 1, scale the pivot row
        for (int c = tid; c < m; c += nt) {
            const double vp = a[(size_t)pr * m + c];
            if (pr != j) a[(size_t)pr * m + c] = a[(size_t)j * m + c];
            const double s = (c == j ? 1.0 : vp) * inv;
            a[(size_t)j * m + c] = s;
            prow[c] = s;
        }
        if (tid == 0) perm[j] = pr;
        __syncthreads();
        // eliminate column j from every other row; f of row pr is what row j held before the swap
        {
            int i = i0, c = c0;
            for (int e = tid; e < mm; e += nt) {
                if (i != j) {
                    const double f = (i == pr) ? cv[j] : cv[i];
                    const double v = (c == j ? 0.0 : a[e]) - f * prow[c];
                    a[e] = v;
                    if (c == j + 1) cn[i] = v;
                } else if (c == j + 1) {
                    cn[i] = prow[c];
                }
                i += di; c += dc;
                if (c >= m) { c -= m; ++i; }
            }
        }
        __syncthreads();
    }
    // undo the row swaps on the columns, last first
    for (int j = m - 1; j >= 0; --j) {
        const int pr = perm[j];
        if (pr != j)
            for (int i = tid; i < m; i += nt) {
                const double x = a[(size_t)i * m + j];
                a[(size_t)i * m + j] = a[(size_t)i * m + pr];
                a[(size_t)i * m + pr] = x;
            }
        __syncthreads();
    }
    if (in_smem) for (int e = tid; e < mm; e += nt) A[e] = a[e];
}

__global__ void __launch_bounds__(1024)
inverse_smem_kernel(double* __restrict__ A, int m, int in_smem, int* __restrict__ info)
{
    extern __shared__ __align__(16) double sm[];
    inverse_in_cta(A, m, in_smem, info, sm);
}

// ---- batched form: the filters of a whole generation of sub-models in ONE chain of launches ------------------
// (app/app.py:130-141 binds one KalmanFilter per sub-model; da.py:91-136 fires for each of them after every step.)
// The sub-models are disjoint forests, so their union is one network: the columns of every covariance block ride as
// members of the SAME two routing launches (block k occupies the rows of its reaches and the first n_k columns), and
// the per-block dense algebra runs with one CTA / one thread group per block.

// X[pos(r)][c] = P_k[i][c]  (r = reach i of block k; zero beyond the block's columns and for inactive blocks)
__global__ void __launch_bounds__(256)
kfb_pack_kernel(const KfbBlock* __restrict__ blocks, const int32_t* __restrict__ blk_of_reach,
                const int32_t* __restrict__ pos_of_reach, const double* __restrict__ P, double* __restrict__ X, int n_u, int ld)
{
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)n_u * ld) return;
    const int r = (int)(gid / ld), c = (int)(gid - (long long)r * ld);
    const KfbBlock b = blocks[blk_of_reach[r]];
    double v = 0.0;
    if (b.active && c < b.n) v = P[b.p_off + (long long)(r - b.row0) * b.n + c];
    X[(size_t)pos_of_reach[r] * ld + c] = v;
}

// X2[pos(row0 + j)][c] = X[pos(row0 + c)][j]: the transposed block, packed again (second pass of _aqat_par)
__global__ void __launch_bounds__(256)
kfb_transpose_kernel(const KfbBlock* __restrict__ blocks, const int32_t* __restrict__ blk_of_reach,
                     const int32_t* __restrict__ pos_of_reach, const double* __restrict__ X, double* __restrict__ X2, int n_u,
                     int ld)
{
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)n_u * ld) return;
    const int r = (int)(gid / ld), c = (int)(gid - (long long)r * ld);
    const KfbBlock b = blocks[blk_of_reach[r]];
    double v = 0.0;
    if (b.active && c < b.n) v = X[(size_t)pos_of_reach[b.row0 + c] * ld + (r - b.row0)];
    X2[(size_t)pos_of_reach[r] * ld + c] = v;
}

// P-_k[j][c] = X2[pos(row0 + j)][c] + Q_k[j][c], scattered into the gauge slices (kf_prior_finish_kernel per block)
__global__ void __launch_bounds__(256)
kfb_finish_kernel(const KfbBlock* __restrict__ blocks, const int32_t* __restrict__ blk_of_reach,
                  const int32_t* __restrict__ pos_of_reach, const int32_t* __restrict__ gl_of_reach,
                  const double* __restrict__ X2, int n_u, int ld, const double* __restrict__ Q, const double* __restrict__ R,
                  double* __restrict__ Pm, double* __restrict__ Ps, double* __restrict__ Prow, double* __restrict__ S)
{
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)n_u * ld) return;
    const int r = (int)(gid / ld), c = (int)(gid - (long long)r * ld);
    const KfbBlock b = blocks[blk_of_reach[r]];
    if (!b.active || c >= b.n) return;
    const int j = r - b.row0;
    const long long e = b.p_off + (long long)j * b.n + c;
    const double v = X2[(size_t)pos_of_reach[r] * ld + c] + Q[e];
    Pm[e] = v;
    const int gr = gl_of_reach[r], gc = gl_of_reach[b.row0 + c];
    if (gc >= 0) Ps[b.nm_off + (long long)j * b.m + gc] = v;
    if (gr >= 0) {
        Prow[b.nm_off + (long long)gr * b.n + c] = v;
        if (gc >= 0) S[b.mm_off + (long long)gr * b.m + gc] = v + R[b.mm_off + (long long)gr * b.m + gc];
    }
}

// S_k <- inv(S_k), one CTA per block (np.linalg.inv, da.py:119)
__global__ void __launch_bounds__(256)
kfb_inverse_kernel(const KfbBlock* __restrict__ blocks, double* __restrict__ S, int* __restrict__ info)
{
    extern __shared__ __align__(16) double sm[];
    const KfbBlock b = blocks[blockIdx.x];
    if (!b.active || b.m <= 0) return;
    inverse_in_cta(S + b.mm_off, b.m, 1, info, sm);
}

// per reach: K_k[j][:] = P-_k[j, s] S_k^-1 (da.py:119), gain = K dz with dz = z - o[s] (da.py:112, 121).
// An inactive block adds a zero gain to the state and keeps K, dz and gain of its last update.
__global__ void __launch_bounds__(128)
kfb_gain_kernel(const KfbBlock* __restrict__ blocks, const int32_t* __restrict__ blk_of_reach,
                const int32_t* __restrict__ pos_of_reach, const int32_t* __restrict__ obs_reach, const double* __restrict__ z,
                const double* __restrict__ O, int ldo, const double* __restrict__ Ps, const double* __restrict__ Sinv,
                double* __restrict__ K, double* __restrict__ dz, double* __restrict__ gain, double* __restrict__ Gp, int n_u)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_u) return;
    const KfbBlock b = blocks[blk_of_reach[r]];
    const size_t gp = (size_t)pos_of_reach[r] * ldo;
    double g = 0.0;
    if (b.active) {
        const int j = r - b.row0;
        const double* ps = Ps + b.nm_off + (long long)j * b.m;
        const double* si = Sinv + b.mm_off;
        for (int q = 0; q < b.m; ++q) {
            double kq = 0.0;
            for (int t = 0; t < b.m; ++t) kq += ps[t] * si[(long long)t * b.m + q];
            K[b.nm_off + (long long)j * b.m + q] = kq;
            const double d = z[b.g_off + q] - O[(size_t)pos_of_reach[obs_reach[b.g_off + q]] * ldo];
            if (j == 0) dz[b.g_off + q] = d;
            g += kq * d;
        }
        gain[r] = g;
    }
    Gp[gp] = g;
    for (int c = 1; c < ldo; ++c) Gp[gp + c] = 0.0;
}

// P+_k = P-_k - K_k P-_k[s]  (da.py:122)
__global__ void __launch_bounds__(256)
kfb_post_kernel(const KfbBlock* __restrict__ blocks, const int32_t* __restrict__ blk_of_reach, const double* __restrict__ Pm,
                const double* __restrict__ K, const double* __restrict__ Prow, double* __restrict__ P, int n_u, int ld)
{
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)n_u * ld) return;
    const int r = (int)(gid / ld), c = (int)(gid - (long long)r * ld);
    const KfbBlock b = blocks[blk_of_reach[r]];
    if (!b.active || c >= b.n) return;
    const int j = r - b.row0;
    const long long e = b.p_off + (long long)j * b.n + c;
    double v = Pm[e];
    const double* kr = K + b.nm_off + (long long)j * b.m;
    const double* pr = Prow + b.nm_off + c;
    for (int q = 0; q < b.m; ++q) v -= kr[q] * pr[(long long)q * b.n];
    P[e] = v;
}

}  // namespace

cudaError_t launch_kf_repack_transposed(const int32_t* reach_of_pos, const int32_t* pos_of_reach, const double* X,
                                        double* X2, int n, int ld, cudaStream_t st)
{
    kf_repack_transposed_kernel<<<nblk((long long)n * ld, 256), 256, 0, st>>>(reach_of_pos, pos_of_reach, X, X2, n, ld);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_kf_prior_finish(const int32_t* reach_of_pos, const int32_t* pos_of_reach, const int32_t* gauge_of_pos,
                                   const double* X2, int ld, const double* Q, const double* R, int n, int m, double* Pm,
                                   double* Ps, double* Prow, double* S, cudaStream_t st)
{
    kf_prior_finish_kernel<<<nblk((long long)n * n, 256), 256, 0, st>>>(reach_of_pos, pos_of_reach, gauge_of_pos, X2, ld, Q,
                                                                        R, n, m, Pm, Ps, Prow, S);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_kf_gain(const int32_t* reach_of_pos, const int32_t* obs_pos, const double* z, const double* O, int ldo,
                           const double* K, int n, int m, double* dz, double* gain, double* Gp, cudaStream_t st)
{
    kf_innovation_kernel<<<nblk(m, 128), 128, 0, st>>>(obs_pos, z, O, ldo, m, dz);
    count_launch();
    kf_gain_kernel<<<nblk(n, 256), 256, 0, st>>>(reach_of_pos, K, dz, n, m, ldo, gain, Gp);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_kfb_pack(const KfbBlock* blocks, const int32_t* blk_of_reach, const int32_t* pos_of_reach, const double* P,
                            double* X, int n_u, int ld, cudaStream_t st)
{
    kfb_pack_kernel<<<nblk((long long)n_u * ld, 256), 256, 0, st>>>(blocks, blk_of_reach, pos_of_reach, P, X, n_u, ld);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_kfb_transpose(const KfbBlock* blocks, const int32_t* blk_of_reach, const int32_t* pos_of_reach,
                                 const double* X, double* X2, int n_u, int ld, cudaStream_t st)
{
    kfb_transpose_kernel<<<nblk((long long)n_u * ld, 256), 256, 0, st>>>(blocks, blk_of_reach, pos_of_reach, X, X2, n_u, ld);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_kfb_update(const KfbBlock* blocks, int nblocks, int max_m, const int32_t* blk_of_reach,
                              const int32_t* pos_of_reach, const int32_t* gl_of_reach, const int32_t* obs_reach,
                              const double* X2, int n_u, int ld, const double* Q, const double* R, const double* z,
                              const double* O, int ldo, double* Pm, double* Ps, double* Prow, double* S, double* K, double* dz,
                              double* gain, double* Gp, double* P, int* info, cudaStream_t st)
{
    kfb_finish_kernel<<<nblk((long long)n_u * ld, 256), 256, 0, st>>>(blocks, blk_of_reach, pos_of_reach, gl_of_reach, X2, n_u,
                                                                      ld, Q, R, Pm, Ps, Prow, S);
    count_launch();
    const size_t smem = ((size_t)4 * max_m + (size_t)max_m * max_m) * sizeof(double);
    cudaError_t e = cudaFuncSetAttribute(kfb_inverse_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kfb_inverse_kernel<<<nblocks, 256, smem, st>>>(blocks, S, info);
    count_launch();
    kfb_gain_kernel<<<nblk(n_u, 128), 128, 0, st>>>(blocks, blk_of_reach, pos_of_reach, obs_reach, z, O, ldo, Ps, S, K, dz, gain,
                                                    Gp, n_u);
    count_launch();
    kfb_post_kernel<<<nblk((long long)n_u * ld, 256), 256, 0, st>>>(blocks, blk_of_reach, Pm, K, Prow, P, n_u, ld);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_inverse(double* A, double* W, int m, int* info, cudaStream_t st)
{
    (void)W;
    const size_t vec = (size_t)4 * m * sizeof(double);
    const size_t full = vec + (size_t)m * m * sizeof(double);
    const int in_smem = full <= 200 * 1024;
    const size_t smem = in_smem ? full : vec;
    cudaError_t e = cudaFuncSetAttribute(inverse_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return e;
    inverse_smem_kernel<<<1, 1024, smem, st>>>(A, m, in_smem, info);
    count_launch();
    return cudaGetLastError();
}

}  // namespace txh
