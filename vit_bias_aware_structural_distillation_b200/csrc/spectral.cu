// Spectral kernels of the BASD loss path (fp32, shared-memory one-sided Jacobi):
//   pooled_eig_kernel   Marchenko-Pastur rank + centred-Gram eigenbases   (layer_selector.py:8-20, 23-37, 90-92)
//   angles_kernel       principal angles, Grassmann distance and its pre-computed backward
//                       (layer_selector.py:95-105; SURVEY.md B.4/B.5)
//   mix_weights_kernel  softmax mixing weights                              (layer_selector.py:107-108)
//   (the per-sample Procrustes core lives in polar.cu)
//   selector_bwd_kernel softmax/temperature backward + Gamma assembly       (SURVEY.md B.3, B.5)
#include "spectral.h"

#include <math_constants.h>
#include <cstring>
#include <mutex>
#include <vector>

#include "cta_linalg.cuh"
#include "jacobi.cuh"

namespace basd {

constexpr float kJacobiTol = 3.0e-7f;
constexpr int kJacobiMaxSweeps = 40;
constexpr float kFp32Eps = 1.1920929e-7f;

// round-robin Jacobi on one CTA, dispatched on the column length (jacobi.cuh)
__device__ __forceinline__ int run_jacobi(float* A, int ld, int n) {
    const int chunks = (ld + JAC_CHUNK_ROWS - 1) / JAC_CHUNK_ROWS;
    switch (chunks) {
        case 1: return jacobi_orthogonalize<1>(A, ld, n, kJacobiTol, kJacobiMaxSweeps);
        case 2: return jacobi_orthogonalize<2>(A, ld, n, kJacobiTol, kJacobiMaxSweeps);
        case 3: return jacobi_orthogonalize<3>(A, ld, n, kJacobiTol, kJacobiMaxSweeps);
        case 4: return jacobi_orthogonalize<4>(A, ld, n, kJacobiTol, kJacobiMaxSweeps);
        case 5: return jacobi_orthogonalize<5>(A, ld, n, kJacobiTol, kJacobiMaxSweeps);
        case 6: return jacobi_orthogonalize<6>(A, ld, n, kJacobiTol, kJacobiMaxSweeps);
        case 7: return jacobi_orthogonalize<7>(A, ld, n, kJacobiTol, kJacobiMaxSweeps);
        default: return jacobi_orthogonalize<8>(A, ld, n, kJacobiTol, kJacobiMaxSweeps);
    }
}

// odd-even ordering with register-resident columns over the CTAs of the cluster (jacobi.cuh); all CTAs call;
// false = shape not supported, nothing done
__device__ __forceinline__ bool run_jacobi_oddeven_cluster(float* A, int ld, int n, float* inbox, uint64_t* bars, int* flags, int* nsweeps) {
    const int chunks = (ld + JAC_CHUNK_ROWS - 1) / JAC_CHUNK_ROWS;
    switch (chunks) {
        case 1: *nsweeps = jacobi_orthogonalize_oddeven_cluster<1>(A, ld, n, kJacobiTol, kJacobiMaxSweeps, inbox, bars, flags); return true;
        case 2: *nsweeps = jacobi_orthogonalize_oddeven_cluster<2>(A, ld, n, kJacobiTol, kJacobiMaxSweeps, inbox, bars, flags); return true;
        case 3: *nsweeps = jacobi_orthogonalize_oddeven_cluster<3>(A, ld, n, kJacobiTol, kJacobiMaxSweeps, inbox, bars, flags); return true;
        case 4: *nsweeps = jacobi_orthogonalize_oddeven_cluster<4>(A, ld, n, kJacobiTol, kJacobiMaxSweeps, inbox, bars, flags); return true;
        case 5: *nsweeps = jacobi_orthogonalize_oddeven_cluster<5>(A, ld, n, kJacobiTol, kJacobiMaxSweeps, inbox, bars, flags); return true;
        case 6: *nsweeps = jacobi_orthogonalize_oddeven_cluster<6>(A, ld, n, kJacobiTol, kJacobiMaxSweeps, inbox, bars, flags); return true;
        case 7: *nsweeps = jacobi_orthogonalize_oddeven_cluster<7>(A, ld, n, kJacobiTol, kJacobiMaxSweeps, inbox, bars, flags); return true;
        case 8: *nsweeps = jacobi_orthogonalize_oddeven_cluster<8>(A, ld, n, kJacobiTol, kJacobiMaxSweeps, inbox, bars, flags); return true;
        default: return false;
    }
}

// ------------------------------------------------------------------------------------------------
// pooled_eig_kernel: one CLUSTER of CTAs per symmetric problem of size n = Ds.  Rank 0 of the cluster holds the matrix
// and runs every phase; the other ranks only take their share of the Jacobi pairs (jacobi.cuh).
//   mode kEigPooled (the loss):  problem p in [0, Lt)      : centred eigen-decomposition of teacher layer p AND its MP rank
//                                problem p in [Lt, Lt + P) : centred eigen-decomposition of student extraction point p - Lt
//   mode kEigMpOnly (the free function marchenko_pastur_rank): problem p in [0, Lt): MP rank from the uncentred G / M itself
// The MP rank (layer_selector.py:8-20) needs the eigenvalues of the UNCENTRED second moment G / M.  With c the column sums,
// G / M = G_c / M + (c / M)(c / M)^T is a rank-one update of the centred Gram whose eigensystem (lambda_i, v_i) this kernel
// computes anyway: its eigenvalues x_i are the roots of the secular equation f(x) = 1 + sum_i u_i^2 / (d_i - x) = 0 with
// d_i = lambda_i / M, u_i = v_i . c / M, and they interlace the d_i.  Only the median and a count above a threshold are
// needed, both of which come from the inertia count  #{x > t} = #{d_i > t} + [f(t) < 0]  (mp_count_above below), so the Lt
// separate uncentred eigenproblems of the first version of this kernel (12 of 28 at cfg2) are gone.
// stats layout: [(Lt + P)][n*n + n]  (Gram row-major, then column sums)
// ------------------------------------------------------------------------------------------------
// History of the Jacobi phase on B200 (cfg2, ms for the 28 pooled problems), one 768-thread CTA per problem, round-robin
// ordering: 16-lane groups / two passes 5.6, 8-lane groups 4.6, two pairs in flight per group 5.4, block-2 ordering 5.0;
// then the odd-even / cluster versions of jacobi.cuh.
// A (column-major, ld) = symmetrised Gram / M, centred unless mp_mode.  One warp per column, eight rows per lane in
// flight: the element-per-iteration loop this replaces (a divide, a modulo and two dependent-latency L2 loads per
// iteration) was half of the 0.1 ms the kernel spends before the Jacobi phase.
__device__ __forceinline__ void pooled_load_gram(const float* __restrict__ G, const float* __restrict__ csum, int n, int ld, float invM,
                                                 bool mp_mode, float* __restrict__ A) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int c = warp; c < n; c += nw) {
        const float cc = csum[c];
        for (int r0 = lane; r0 < ld; r0 += 32 * 8) {
            float g0[8], g1[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int r = r0 + 32 * u;
                g0[u] = r < n ? G[r * n + c] : 0.f;
                g1[u] = r < n ? G[c * n + r] : 0.f;
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int r = r0 + 32 * u;
                if (r < ld) {
                    // symmetrise the split-K atomics result (bitwise symmetric input keeps Jacobi well behaved)
                    const float g = 0.5f * (g0[u] + g1[u]);
                    A[c * ld + r] = r < n ? (mp_mode ? g * invM : (g - csum[r] * cc * invM)) : 0.f;      // (r, c)-symmetric rounding
                }
            }
        }
    }
}

// Number of eigenvalues of diag(d) + u u^T above t (one warp; u2 = u^2).  Interlacing puts x_i in [d_i, d_(i+1)]
// (ascending), so for t between two poles only one eigenvalue is undecided, and it lies above t iff f(t) < 0 (f rises from
// -inf to +inf between two poles).  t == d_i counts as t = d_i + 0.  All 32 lanes call; the result is warp-uniform.
__device__ __forceinline__ int mp_count_above(const float* __restrict__ d, const float* __restrict__ u2, int n, float t) {
    const int lane = threadIdx.x & 31;
    int cnt = 0;
    float f = 0.f;
    for (int i = lane; i < n; i += 32) {
        const float di = d[i], den = di - t;
        cnt += di > t;
        f += u2[i] / (den == 0.f ? -1e-37f : den);
    }
    f = warp_sum(f);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    return cnt + ((1.f + f) < 0.f ? 1 : 0);
}
// MP rank of diag(d) + u u^T (warp 0 of the CTA; d_lo / d_hi bracket the median eigenvalue by interlacing)
__device__ __forceinline__ int mp_rank_secular(const float* __restrict__ d, const float* __restrict__ u2, int n, float d_lo, float d_hi,
                                               float q_ratio /* D / M */, int want) {
    // median of the top m eigenvalues = the smallest t with #{x > t} <= want = m - 1 - (m-1)/2 (torch.median: lower middle)
    float lo = d_lo, hi = d_hi;
    for (int it = 0; it < 40; ++it) {
        const float mid = 0.5f * (lo + hi);
        if (!(mid > lo && mid < hi)) break;             // the bracket is one ulp wide
        if (mp_count_above(d, u2, n, mid) <= want) hi = mid; else lo = mid;
    }
    const float med = mp_count_above(d, u2, n, lo) <= want ? lo : hi;
    const float sq = 1.f + sqrtf(q_ratio);
    return mp_count_above(d, u2, n, med * sq * sq);
}

constexpr int kPooledThreads = 256;        // 32 eight-lane groups per CTA: n <= 64 x cluster size; 255 registers per thread, no spills
constexpr int kPooledCluster = 4;           // smallest cluster (n = 192: 24 pairs per CTA); pooled_pick_cluster takes a larger one when the SMs are there
constexpr int kPooledLargeThreads = 768;
// global-memory Jacobi on one CTA: 4-lane groups when that puts every pair of a step in flight at once
__device__ __forceinline__ int run_jacobi_global(float* A, int ld, int n) {
    const int half = (n + 1) / 2;
    if (half > static_cast<int>(blockDim.x) / 8 && half <= static_cast<int>(blockDim.x) / 4)
        return jacobi_orthogonalize_global<4>(A, ld, n, kJacobiTol, kJacobiMaxSweeps);
    return jacobi_orthogonalize_global<8>(A, ld, n, kJacobiTol, kJacobiMaxSweeps);
}
// LARGE = true (n > 224: the matrix no longer fits one SM's shared memory): one plain CTA of 768 threads per problem,
// the matrix in `scratch` (global memory, L2-resident), Jacobi by jacobi_orthogonalize_global; every other phase is
// the same code on a global pointer.  The Cholesky preconditioner needs one thread per row (n <= 768); larger
// problems (marchenko_pastur_rank on unprojected teacher features) run Jacobi on the Gram itself.
template <bool LARGE>
__global__ void __launch_bounds__(LARGE ? kPooledLargeThreads : kPooledThreads, 1)
pooled_eig_kernel(const float* __restrict__ stats, int n, int Lt, int P, float M_teacher, float M_student,
                  int* __restrict__ ranks, float* __restrict__ evals, float* __restrict__ evecs_km,
                  float* __restrict__ evecs_cm, int* __restrict__ sweeps_out, float* __restrict__ scratch, int phase,
                  int* __restrict__ chol_flags, int mode) {
    // phase (LARGE only): 1 = everything in this launch; 0 = up to the Cholesky factor (the Jacobi sweeps then run in
    // jacobi_cluster_global_kernel over a cluster per problem); 2 = from the rotated columns on
    extern __shared__ float sm[];
    const int ld = jacobi_ld(n);
    float* A = LARGE ? scratch + static_cast<size_t>(blockIdx.x) * ld * n : sm;
    float* vals = LARGE ? sm : A + static_cast<size_t>(ld) * n;
    float* csum = vals + n;
    int* order = reinterpret_cast<int*>(csum + n);
    float* inbox = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(order + n + 64) + 15) & ~uintptr_t(15));   // one column (Jacobi across CTAs)
    __shared__ int s_count;
    __shared__ int s_flags[16];
    __shared__ __align__(8) uint64_t s_bars[2];
    __shared__ int s_bad;

    const int crank = LARGE ? 0 : static_cast<int>(cooperative_groups::this_cluster().block_rank());
    const int p = LARGE ? blockIdx.x : blockIdx.x / static_cast<int>(cooperative_groups::this_cluster().num_blocks());
    const bool mp_mode = mode == kEigMpOnly;
    const int gram_idx = p;                                       // index into stats (teacher 0..Lt-1, student Lt..)
    const float Mrows = gram_idx < Lt ? M_teacher : M_student;
    const float* G = stats + static_cast<size_t>(gram_idx) * (n * n + n);
    const float* cs = G + n * n;
    const float invM = 1.f / Mrows;
    bool use_chol = false;
    if (LARGE && phase == 2) {
        use_chol = chol_flags[blockIdx.x] != 0;
        for (int i = threadIdx.x; i < n; i += blockDim.x) csum[i] = cs[i];
        if (threadIdx.x == 0) s_count = 0;
        __syncthreads();
    } else
    if (crank == 0) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) csum[i] = cs[i];
    if (threadIdx.x == 0) s_count = 0;
    __syncthreads();
    pooled_load_gram(G, csum, n, ld, invM, mp_mode, A);
    __syncthreads();
    // Veselic-Hari preconditioning: G = L L^T, then one-sided Jacobi on the Cholesky factor instead of on G.  The
    // singular values of L are the square roots of the eigenvalues (half the condition number in digits), the rotated
    // columns L V = U Sigma are still sigma_i times the eigenvectors of G, and the sweep count roughly halves.
    // A non-positive pivot (numerically singular Gram) falls back to Jacobi on G itself.
    if (threadIdx.x == 0) s_bad = 0;
    __syncthreads();
    float dmax = 0.f;
    for (int i = threadIdx.x; i < n; i += blockDim.x) dmax = fmaxf(dmax, A[i * ld + i]);
    for (int o = 16; o > 0; o >>= 1) dmax = fmaxf(dmax, __shfl_xor_sync(0xffffffffu, dmax, o));
    if ((threadIdx.x & 31) == 0) vals[threadIdx.x >> 5] = dmax;
    __syncthreads();
    dmax = 0.f;
    for (int wv = 0; wv < (blockDim.x >> 5); ++wv) dmax = fmaxf(dmax, vals[wv]);
    __syncthreads();
    const bool chol_fits = n <= static_cast<int>(blockDim.x);        // one matrix row per thread
    if (chol_fits) cta_cholesky_lower(A, ld, n, &s_bad, 1e-6f * dmax);       // pivots below 1e-6 of the largest diagonal: not trusted in fp32
    use_chol = chol_fits && s_bad == 0;
    if (chol_fits && !use_chol) {          // rebuild G from the statistics
        pooled_load_gram(G, csum, n, ld, invM, mp_mode, A);
    }
    __syncthreads();
    }   // crank == 0
    int nsweeps = 0;
    if constexpr (LARGE) {
        if (phase == 0) {
            if (threadIdx.x == 0) chol_flags[blockIdx.x] = use_chol ? 1 : 0;
            return;
        }
        if (phase == 1) nsweeps = run_jacobi_global(A, ld, n);
    } else {
        jac_cluster_sync();                     // the matrix is ready in rank 0's shared memory
        const int n_cluster = static_cast<int>(cooperative_groups::this_cluster().num_blocks());
        const int groups_per_cta = ((n + 1) / 2 + n_cluster - 1) / n_cluster;
        const bool cluster_ok = groups_per_cta * JAC_GROUP <= static_cast<int>(blockDim.x) &&
                                run_jacobi_oddeven_cluster(A, ld, n, inbox, s_bars, s_flags, &nsweeps);      // uniform over the cluster
        if (crank != 0) return;                 // (the Jacobi routine ends with a cluster barrier: nobody touches this CTA again)
        if (!cluster_ok) nsweeps = run_jacobi(A, ld, n);
    }
    column_norms(A, ld, n, n, vals);        // sigma_i (Cholesky route) or lambda_i (fallback)
    __syncthreads();
    if (use_chol)
        for (int i = threadIdx.x; i < n; i += blockDim.x) vals[i] = vals[i] * vals[i];
    __syncthreads();
    rank_descending(vals, n, order);
    __syncthreads();
    if (threadIdx.x == 0 && sweeps_out && !(LARGE && phase == 2)) sweeps_out[p] = nsweeps;

    if (mp_mode) {
        // M < D (layer_selector.py:14-15): the reference takes the M eigenvalues of F F^T / M - the top M of the D x D
        // Gram used here (its other D - M are zero up to rounding and are left out of the median and the count).
        const int m_eff = Mrows < static_cast<float>(n) ? max(1, static_cast<int>(Mrows + 0.5f)) : n;
        // ascending index (m-1)/2 == descending index m-1-(m-1)/2  (torch.median = lower middle)
        const float med = vals[order[m_eff - 1 - (m_eff - 1) / 2]];
        const float sq = 1.f + sqrtf(static_cast<float>(n) * invM);
        const float lam_plus = med * sq * sq;
        int local = 0;
        for (int i = threadIdx.x; i < m_eff; i += blockDim.x) local += vals[order[i]] > lam_plus;
        atomicAdd(&s_count, local);
        __syncthreads();
        if (threadIdx.x == 0) ranks[p] = min(s_count, n - 1);
        return;
    }
    if (p < Lt && ranks) {
        // MP rank of this teacher layer from the centred eigensystem (see the header), in units of M: the eigenvalues of
        // G_c + c c^T / M = diag(lambda) + u u^T with u_i = v_i . c / sqrt(M), v_i = column_i / |column_i|
        float* u2 = inbox;                                        // (the Jacobi mailbox column is free now; ld + 8 >= n floats)
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
        for (int c = warp; c < n; c += nwarps) {
            const float* col = A + static_cast<size_t>(c) * ld;
            float dot = 0.f;
            for (int r = lane; r < n; r += 32) dot = fmaf(col[r], csum[r], dot);
            dot = warp_sum(dot);
            if (lane == 0) {
                const float nv2 = use_chol ? vals[c] : vals[c] * vals[c];       // |column|^2
                u2[c] = nv2 > 0.f ? dot * dot / nv2 * invM : 0.f;
            }
        }
        __syncthreads();
        if (warp == 0) {
            // M < D (layer_selector.py:14-15): the reference takes the M eigenvalues of F F^T / M = the top M of the D x D problem
            // (the other D - M are zero): median and count run over those.
            const int m_eff = Mrows < static_cast<float>(n) ? max(1, static_cast<int>(Mrows + 0.5f)) : n;
            const int want = m_eff - 1 - (m_eff - 1) / 2;         // eigenvalues above the median (descending index of the median)
            // bracket of the median by interlacing (descending order: lambda_i <= x_i <= lambda_(i-1)), the top one extended by |u|^2
            const float d_lo = vals[order[want]];
            float d_hi;
            if (want >= 1) d_hi = vals[order[want - 1]];
            else { float su = 0.f; for (int i = lane; i < n; i += 32) su += u2[i]; d_hi = d_lo + warp_sum(su); }
            const int rk = mp_rank_secular(vals, u2, n, d_lo, d_hi, static_cast<float>(n) * invM, want);
            if (lane == 0) ranks[p] = min(rk, n - 1);
        }
        __syncthreads();
    }
    const int q = p;                                              // output slot: teacher 0..Lt-1, student Lt..Lt+P-1
    float* ev = evals + static_cast<size_t>(q) * n;
    float* vk = evecs_km + static_cast<size_t>(q) * n * n;        // [eig][component]
    float* vc = evecs_cm + static_cast<size_t>(q) * n * n;        // [component][eig]
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int col = order[i];
        ev[i] = vals[col];
        const float nv = use_chol ? sqrtf(vals[col]) : vals[col];   // norm of the rotated column
        csum[i] = nv > 0.f ? 1.f / nv : 0.f;                        // (csum is free now) 1 / norm of eigenvector i's column
    }
    __syncthreads();
    // eigenvector e = column order[e] of A, normalised; one warp per eigenvector, lanes over components (conflict-free
    // shared reads; the [eig][comp] store is coalesced, the [comp][eig] one is a 4-byte scatter that L2 merges)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    for (int e = warp; e < n; e += nwarps) {
        const float* col = A + static_cast<size_t>(order[e]) * ld;
        const float s = csum[e];
        for (int c = lane; c < n; c += 32) {
            const float v = col[c] * s;
            vk[e * n + c] = v;
            vc[c * n + e] = v;
        }
    }
}

// Jacobi sweeps of the LARGE path for n <= 384: a cluster of CTAs per problem, columns resident in registers (up to 12
// chunks of 32 rows), the matrix in global memory, mailboxes in shared memory (jacobi.cuh, COMPACT).  One CTA streaming a
// 384 x 384 matrix through its L2 port three times per Jacobi step took 70 ms for the 28 problems of cfg5.
template <int CHUNKS>
__global__ void __launch_bounds__(kPooledThreads, 1)
jacobi_cluster_global_kernel(float* __restrict__ scratch, int n, int* __restrict__ sweeps_out) {
    extern __shared__ __align__(16) float jsm[];
    float* sm = jsm;
    __shared__ int s_flags[16];
    __shared__ __align__(8) uint64_t s_bars[2];
    const int ld = jacobi_ld(n);
    const int C = static_cast<int>(cooperative_groups::this_cluster().num_blocks());
    const int p = blockIdx.x / C;
    const int gpc = ((n + 1) / 2 + C - 1) / C;
    float* mail = sm;                                   // [gpc][ld]
    float* inbox = sm + static_cast<size_t>(gpc) * ld;  // [ld]
    float* A = scratch + static_cast<size_t>(p) * ld * n;
    const int nsw = jacobi_orthogonalize_oddeven_cluster<CHUNKS, true>(A, ld, n, kJacobiTol, kJacobiMaxSweeps, inbox, s_bars, s_flags, mail);
    if (cooperative_groups::this_cluster().block_rank() == 0 && threadIdx.x == 0 && sweeps_out) sweeps_out[p] = nsw;
}

// ------------------------------------------------------------------------------------------------
// angles_kernel: grid (Lt, P).  Per (student point i, teacher layer j):
//   A = V_s[:, :k]^T (P_s^T U_t)   (k x k);  cos = svdvals(A) via Jacobi on A^T A;
//   d2 = sum sw theta^2 / sum sw;  Gamma_sym = d(d2)/dG_s + transpose   (n x n, saved for backward)
// ------------------------------------------------------------------------------------------------
// LARGE = true (n > 224): the n-sized operands stay in global memory (L2); see j_in_smem for the k x k Jacobi matrix.
constexpr int kAnglesLargeSmemK = 128;
constexpr int kAnglesLargeStageFloats = 30 * 1024;     // extra staging room behind the k x k matrix (LARGE): 64 KB + 120 KB = k <= 61 at n = 384
template <bool LARGE>
__global__ void __launch_bounds__(kSpectralThreads, 1)
angles_kernel(int n, int Lt, int P, const int* __restrict__ ranks, const float* __restrict__ evals,
              const float* __restrict__ evecs_km, const float* __restrict__ evecs_cm, const float* __restrict__ proj_s,
              float* __restrict__ scratch_all, float* __restrict__ d2_out, float* __restrict__ gamma_out,
              float* __restrict__ cos_out) {
    extern __shared__ float sm[];
    const int j = blockIdx.x, i = blockIdx.y;
    const int k = ranks[j];
    const int ld = jacobi_ld(max(k, 1));
    float* vals = LARGE ? sm : sm + static_cast<size_t>(jacobi_ld(n - 1)) * (n - 1);
    float* coef = vals + n;
    float* red = coef + n;                                       // 33 floats
    int* order = reinterpret_cast<int*>(red + 40);
    float* inbox = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(order + n + 8) + 15) & ~uintptr_t(15));   // odd-even Jacobi: one column
    // k x k Jacobi matrix (ld x k).  n <= 224: any k fits shared memory.  LARGE: the MP rank k is far below n in practice
    // (16 .. 60 of 384 on the BASELINE shapes): up to kAnglesLargeSmemK it runs in shared memory like the small problems, only
    // a larger one falls back to the spare n x n slot of the scratch area (global memory, L2 latency on every rotation).
    const bool j_in_smem = !LARGE || k <= kAnglesLargeSmemK;
    float* J = !LARGE ? sm
               : j_in_smem ? inbox + jacobi_ld(n) + 8
                           : scratch_all + (static_cast<size_t>(blockIdx.y) * Lt + blockIdx.x) * (8 * static_cast<size_t>(n) * n) + 7 * static_cast<size_t>(n) * n;
    __shared__ int s_flags[16];
    __shared__ __align__(8) uint64_t s_bars[2];

    const float* lam_t = evals + static_cast<size_t>(j) * n;
    const float* Ut = evecs_km + static_cast<size_t>(j) * n * n;             // [eig][comp]
    const float* lam_s = evals + static_cast<size_t>(Lt + i) * n;
    const float* Vs_km = evecs_km + static_cast<size_t>(Lt + i) * n * n;     // [eig][comp]
    const float* Vs_cm = evecs_cm + static_cast<size_t>(Lt + i) * n * n;     // [comp][eig]
    float* gam = gamma_out + (static_cast<size_t>(i) * Lt + j) * n * n;
    float* scratch = scratch_all + (static_cast<size_t>(i) * Lt + j) * (8 * static_cast<size_t>(n) * n);
    float* Ur = scratch;                      // [b][c]   k x n
    float* Wg = Ur + n * n;                   // [b][e]   column b contiguous in e
    float* Qg = Wg + 2 * n * n;               // [b'][b]
    float* WQg = Qg + n * n;                  // [b'][e]
    float* Fg = WQg + n * n;                  // [a][e]
    float* T1g = Fg + n * n;                  // H [a][c]

    if (k == 0) {                              // reference: 0/0 -> NaN (layer_selector.py:105)
        if (threadIdx.x == 0) d2_out[i * Lt + j] = CUDART_NAN_F;
        for (int t = threadIdx.x; t < n * n; t += blockDim.x) gam[t] = 0.f;
        return;
    }
    // (a) Ur[b][c] = sum_r Ut[b][r] P_s[r][c]
    const bool vec_ok = (n & 3) == 0;                  // 128-bit operand loads (cta_gemm_mk); every D_s the library accepts is a multiple of 8
    if (vec_ok) {
        cta_gemm_mk(n, k, n, proj_s, n, Ut, n, [&](int c, int b, float v) { Ur[b * n + c] = v; });
    } else {
        cta_gemm(n, k, n,
                 [&](int c, int r) { return proj_s[r * n + c]; },
                 [&](int r, int b) { return Ut[b * n + r]; },
                 [&](int c, int b, float v) { Ur[b * n + c] = v; });
    }
    __syncthreads();
    for (int t = threadIdx.x; t < ld * k; t += blockDim.x) J[t] = 0.f;
    __syncthreads();
    // (b) W[e][b] = sum_c Vs[e][c] Ur[b][c];   its top k x k block is A = V_s[:, :k]^T (P_s^T U_t)
    //     J = A^T goes straight to shared memory: column a of J = row a of A
    if (vec_ok) {
        cta_gemm_mk(n, k, n, Vs_cm, n, Ur, n, [&](int e, int b, float v) { Wg[b * n + e] = v; if (e < k) J[e * ld + b] = v; });
    } else {
        cta_gemm(n, k, n,
                 [&](int e, int c) { return Vs_cm[c * n + e]; },
                 [&](int c, int b) { return Ur[b * n + c]; },
                 [&](int e, int b, float v) { Wg[b * n + e] = v; if (e < k) J[e * ld + b] = v; });
    }
    __syncthreads();
    // (c) one-sided Jacobi on A^T:  A^T R = Y Sigma  =>  A^T A = Y Sigma^2 Y^T.  The rotated columns are sigma_m y_m: their
    //     norms are the cosines themselves (no squaring through A^T A) and their directions the right singular vectors.
    // odd-even ordering with register-resident columns (a "cluster" of this one CTA): half the shared-memory round trips
    // and barriers of the round-robin version per rotation; k x k with k ~ 15-40 is a pure latency chain
    if (!j_in_smem) {
        __threadfence_block();
        run_jacobi_global(J, ld, k);
    } else {
        int nsw;
        if (!run_jacobi_oddeven_cluster(J, ld, k, inbox, s_bars, s_flags, &nsw)) run_jacobi(J, ld, k);
    }
    column_norms(J, ld, k, k, vals);          // vals = sigma
    __syncthreads();
    rank_descending(vals, k, order);
    __syncthreads();
    // (d) distances and d(d2)/dsigma
    float swsum = 0.f, acc = 0.f;
    for (int r = threadIdx.x; r < k; r += blockDim.x) swsum += sqrtf(fmaxf(lam_t[r], 0.f));
    swsum = cta_sum(swsum, red);
    for (int r = threadIdx.x; r < k; r += blockDim.x) {
        const int col = order[r];
        const float sig = vals[col];
        const float sw = sqrtf(fmaxf(lam_t[r], 0.f));
        const float clampv = 1.f - kFp32Eps;
        const float sc = fminf(sig, clampv);
        const float th = acosf(sc);
        acc += sw * th * th;
        float ds = 0.f;
        if (sig <= clampv) ds = sw * 2.f * th * (-rsqrtf(fmaxf(1.f - sc * sc, 1e-30f))) / swsum;
        // Q = Y diag(dsigma / sigma) Y^T with Y = normalised columns (column norm = sigma)
        coef[col] = (sig > 1e-20f) ? ds / (sig * vals[col] * vals[col]) : 0.f;
        if (cos_out) cos_out[(static_cast<size_t>(i) * Lt + j) * n + r] = sig;
    }
    acc = cta_sum(acc, red);
    if (threadIdx.x == 0) d2_out[i * Lt + j] = acc / swsum;
    __syncthreads();
    // Q[b][b'] = sum_m J[b][m] coef_m J[b'][m]     (rows kq = k rounded up to 4 apart: 16-byte aligned for the 128-bit loads below)
    const int kq = (k + 3) & ~3;
    cta_gemm(k, k, k,
             [&](int b, int m) { return J[m * ld + b] * coef[m]; },
             [&](int m, int b2) { return J[m * ld + b2]; },
             [&](int b, int b2, float v) { Qg[b2 * kq + b] = v; });
    __syncthreads();
    // (e) WQ[e][b'] = sum_b W[e][b] Q[b][b']
    if (vec_ok) {
        cta_gemm_mk(n, k, k, Wg, n, Qg, kq, [&](int e, int b2, float v) { WQg[b2 * n + e] = v; });
    } else {
        cta_gemm(n, k, k,
                 [&](int e, int b) { return Wg[b * n + e]; },
                 [&](int b, int b2) { return Qg[b2 * kq + b]; },
                 [&](int e, int b2, float v) { WQg[b2 * n + e] = v; });
    }
    __syncthreads();
    //     F[e][a] = (sum_b' WQ[e][b'] A[a][b']) / (lam_a - lam_e)   for e >= k, a < k
    const int nc = n - k;
    cta_gemm(nc, k, k,
             [&](int e, int b2) { return WQg[b2 * n + k + e]; },
             [&](int b2, int a) { return Wg[b2 * n + a]; },
             [&](int e, int a, float v) { Fg[a * n + e] = v / (lam_s[a] - lam_s[k + e]); });      // (row a of F from column 0: aligned)
    __syncthreads();
    // (f) Gamma = V_hi^T F V_lo  (V_hi = eigenvectors e >= k, V_lo = a < k), associated as (V_hi^T F) V_lo: n k (n + nc)
    //     multiply-adds instead of the n n nc of V_hi^T (F V_lo), k << nc.
    //     H[c][a] = sum_{e>=k} Vs[e][c] F[e][a]
    if (vec_ok) {
        cta_gemm_mk(n, k, nc, Vs_km + static_cast<size_t>(k) * n, n, Fg, n, [&](int c, int a, float v) { T1g[a * n + c] = v; });
    } else {
        cta_gemm(n, k, nc,
                 [&](int c, int e) { return Vs_km[(k + e) * n + c]; },
                 [&](int e, int a) { return Fg[a * n + e]; },
                 [&](int c, int a, float v) { T1g[a * n + c] = v; });
    }
    __syncthreads();
    //     Gamma_sym[c][c'] = sum_a H[c][a] Vs[a][c'] + Vs[a][c] H[c'][a]   (one product of inner size 2k; symmetric, so the
    //     store may run along c)
    if ((n & 3) == 0) {
        // H and the first k eigenvectors (k x n each) are staged in the shared memory the Jacobi matrix no longer needs: read
        // straight from the L2-resident scratch, this product's four 128-bit loads per 32 FMAs were pure latency (134 k of the
        // 430 k cycles of a k = 15 CTA at n = 192)
        const size_t stage_floats = LARGE ? static_cast<size_t>(jacobi_ld(kAnglesLargeSmemK)) * kAnglesLargeSmemK + kAnglesLargeStageFloats
                                          : static_cast<size_t>(jacobi_ld(n - 1)) * (n - 1);
        float* stage = LARGE ? inbox + jacobi_ld(n) + 8 : sm;
        if (2 * static_cast<size_t>(k) * n <= stage_floats) {
            float* sH = stage;
            float* sV = stage + static_cast<size_t>(k) * n;
            __syncthreads();                                  // (the Jacobi matrix and Q products are done with this memory)
            for (int t = threadIdx.x * 4; t < k * n; t += blockDim.x * 4) {
                *reinterpret_cast<float4*>(sH + t) = *reinterpret_cast<const float4*>(T1g + t);
                *reinterpret_cast<float4*>(sV + t) = *reinterpret_cast<const float4*>(Vs_km + t);
            }
            __syncthreads();
            cta_gemm_sym2(n, k, sH, sV, n, [&](int c, int c2, float v) { gam[c2 * n + c] = v; });
        } else {
            cta_gemm_sym2(n, k, T1g, Vs_km, n, [&](int c, int c2, float v) { gam[c2 * n + c] = v; });
        }
    } else {
        cta_gemm(n, n, 2 * k,
                 [&](int c, int a) { return a < k ? T1g[a * n + c] : Vs_km[(a - k) * n + c]; },
                 [&](int a, int c2) { return a < k ? Vs_km[a * n + c2] : T1g[(a - k) * n + c2]; },
                 [&](int c, int c2, float v) { gam[c2 * n + c] = v; });
    }
}

// w = softmax(-d2 / softplus(log_temperature))   one warp per extraction point
__global__ void mix_weights_kernel(const float* __restrict__ d2, const float* __restrict__ log_temp, int Lt, int P,
                                   float* __restrict__ w) {
    const int i = blockIdx.x;
    if (i >= P) return;
    const float lt = log_temp[i];
    const float tau = lt > 20.f ? lt : log1pf(expf(lt));
    float mx = -CUDART_INF_F;
    for (int j = threadIdx.x; j < Lt; j += 32) mx = fmaxf(mx, -d2[i * Lt + j] / tau);
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float s = 0.f;
    for (int j = threadIdx.x; j < Lt; j += 32) s += expf(-d2[i * Lt + j] / tau - mx);
    s = warp_sum(s);
    for (int j = threadIdx.x; j < Lt; j += 32) {
        const float d = d2[i * Lt + j];
        w[i * Lt + j] = (d == d) ? expf(-d / tau - mx) / s : CUDART_NAN_F;
    }
}

// ------------------------------------------------------------------------------------------------
// selector_bwd_kernel: grid (tiles, P).  gd_j = d L / d d2_ij from d L / d w (SURVEY.md B.3), then
//   Gamma'_i = sum_j gd_j Gamma_sym_ij  -> bf16 hi/lo;  corr_i = mu_i^T Gamma'_i;  grad log_temperature.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
selector_bwd_kernel(int n, int Lt, int P, const float* __restrict__ gw_raw, const float* __restrict__ scale_ptr,
                    float scale_host, const float* __restrict__ w, const float* __restrict__ d2,
                    const float* __restrict__ log_temp, const float* __restrict__ gamma,
                    const float* __restrict__ stats, float M_student,
                    __nv_bfloat16* __restrict__ gam_hi, __nv_bfloat16* __restrict__ gam_lo, float* __restrict__ corr,
                    float* __restrict__ grad_log_temp) {
    __shared__ float gd[64];
    const int i = blockIdx.y;
    const float scale = scale_host * (scale_ptr ? *scale_ptr : 1.f);
    const float lt = log_temp[i];
    const float tau = lt > 20.f ? lt : log1pf(expf(lt));
    if (threadIdx.x < 32) {
        float dotw = 0.f;
        for (int j = threadIdx.x; j < Lt; j += 32) dotw += w[i * Lt + j] * gw_raw[i * Lt + j] * scale;
        dotw = warp_sum(dotw);
        float gtau = 0.f;
        for (int j = threadIdx.x; j < Lt; j += 32) {
            const float gx = w[i * Lt + j] * (gw_raw[i * Lt + j] * scale - dotw);
            gd[j] = -gx / tau;
            gtau += gx * d2[i * Lt + j] / (tau * tau);
        }
        gtau = warp_sum(gtau);
        if (threadIdx.x == 0 && blockIdx.x == 0) grad_log_temp[i] = gtau / (1.f + expf(-lt));
    }
    __syncthreads();
    // each CTA handles a strip of rows c; every thread a few (c, c') entries
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < n * n; t += gridDim.x * blockDim.x) {
        float acc = 0.f;
        for (int j = 0; j < Lt; ++j) acc = fmaf(gd[j], gamma[(static_cast<size_t>(i) * Lt + j) * n * n + t], acc);
        const __nv_bfloat16 hi = __float2bfloat16(acc);
        gam_hi[static_cast<size_t>(i) * n * n + t] = hi;
        gam_lo[static_cast<size_t>(i) * n * n + t] = __float2bfloat16(acc - __bfloat162float(hi));
    }
}
// corr[i][c'] = sum_c mu_i[c] Gamma'_i[c][c']  (the centring correction of the student gradient) in a fixed order: a warp
// per 32 columns c', lanes along c' (coalesced rows of Gamma'), eight warps of the CTA each taking every eighth row c
// ascending, combined in warp order (the atomicAdd version of this sum was one of the sources of launch-to-launch
// differences; one thread per column walking all rows was 58 us of dependent L2 latency at cfg2).
__global__ void __launch_bounds__(256)
selector_corr_kernel(int n, int Lt, const float* __restrict__ stats, float M_student, const __nv_bfloat16* __restrict__ gam_hi,
                     const __nv_bfloat16* __restrict__ gam_lo, float* __restrict__ corr) {
    __shared__ float part[8][32];
    const int i = blockIdx.y;
    const float* csum = stats + static_cast<size_t>(Lt + i) * (n * n + n) + n * n;
    const float invM = 1.f / M_student;
    const __nv_bfloat16* gh = gam_hi + static_cast<size_t>(i) * n * n;
    const __nv_bfloat16* gl = gam_lo + static_cast<size_t>(i) * n * n;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int c2 = blockIdx.x * 32 + lane;
    float acc = 0.f;
    if (c2 < n)
        for (int c = warp; c < n; c += 8) acc = fmaf(csum[c] * invM, __bfloat162float(gh[c * n + c2]) + __bfloat162float(gl[c * n + c2]), acc);
    part[warp][lane] = acc;
    __syncthreads();
    if (warp == 0 && c2 < n) {
        float tot = 0.f;
#pragma unroll
        for (int wv = 0; wv < 8; ++wv) tot += part[wv][lane];
        corr[i * n + c2] = tot;
    }
}

// ------------------------------------------------------------------------------------------------ launchers
static size_t pooled_smem(int n, bool large) { return ((large ? 0 : static_cast<size_t>(jacobi_ld(n)) * n) + 3 * n + 64 + jacobi_ld(n) + 8) * sizeof(float); }
static size_t angles_smem(int n, bool large) {
    const size_t jmat = large ? static_cast<size_t>(jacobi_ld(kAnglesLargeSmemK)) * kAnglesLargeSmemK + kAnglesLargeStageFloats + 16
                              : static_cast<size_t>(jacobi_ld(n - 1)) * (n - 1);
    return (jmat + 3 * n + 128 + n + 16 + jacobi_ld(n)) * sizeof(float);
}
bool spectral_large(int n) { return n > kSpectralSmemMax; }
size_t pooled_eig_scratch_floats(int n, int problems) { return spectral_large(n) ? static_cast<size_t>(problems) * jacobi_ld(n) * n + problems + 64 : 0; }

// Cluster size of the shared-memory solver: the Jacobi pair-step is a dependent chain whose latency grows with the warps an
// SM has to issue for (jacobi.cuh), so every problem gets as many CTAs as the GPU can co-schedule for ALL problems at once
// (a cluster lives inside one GPC: cudaOccupancyMaxActiveClusters knows how many fit).  Cached per device and shape.
// When the problems do not fit at once whatever the size (cfg4: 28 problems of size 384, 24 six-CTA clusters fit) the smallest
// cluster stays: picking the size from a waves x pair-step-time model chose a larger one there and measured 10.0 ms against
// 9.4 ms (r2w); 320- / 384-thread CTAs (clusters of 5 / 4, all 28 problems in ONE wave; the 12-chunk columns then live in 168
// registers with 44 bytes of spills) measured 9.26 against 9.39 ms (r3b) - at n = 384 the pair-step is bound by the instructions
// an SM issues, not by the chain, so fewer SMs per problem give back what the second wave cost; not kept.  Splitting the launch
// (24 problems on 6-CTA clusters, then the last 4 on 8-CTA clusters) measured 10.2 ms (r3c): in ONE launch the remaining clusters
// start as soon as any problem converges, the split makes them wait for the slowest of the first 24.
static int pooled_pick_cluster(const void* kern, int n, int problems, size_t smem_fixed, size_t smem_per_group_floats) {
    const int groups = (n + 1) / 2, per_cta = kPooledThreads / JAC_GROUP;
    const int c_min = (groups + per_cta - 1) / per_cta;
    struct Key { int dev, n, problems, cluster; const void* kern; };
    static std::mutex mu;
    static std::vector<Key> cache;
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lock(mu);
    for (const Key& k : cache)
        if (k.dev == dev && k.n == n && k.problems == problems && k.kern == kern) return k.cluster;
    int pick = c_min > kPooledCluster ? c_min : kPooledCluster;
    for (int c = 8; c > pick; --c) {
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof cfg);
        cfg.gridDim = dim3(problems * c);
        cfg.blockDim = dim3(kPooledThreads);
        cfg.dynamicSmemBytes = smem_fixed + static_cast<size_t>((groups + c - 1) / c) * smem_per_group_floats * sizeof(float);
        cudaLaunchAttribute attr;
        attr.id = cudaLaunchAttributeClusterDimension;
        attr.val.clusterDim.x = c; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
        cfg.attrs = &attr;
        cfg.numAttrs = 1;
        int fit = 0;
        if (cudaOccupancyMaxActiveClusters(&fit, kern, &cfg) == cudaSuccess && fit >= problems) { pick = c; break; }
        cudaGetLastError();
    }
    cache.push_back({dev, n, problems, pick, kern});
    return pick;
}

cudaError_t launch_pooled_eig(const float* stats, int n, int Lt, int P, float Mt, float Ms, int* ranks, float* evals,
                              float* evecs_km, float* evecs_cm, int* sweeps, float* scratch, cudaStream_t st, int mode) {
    const bool large = spectral_large(n);
    const size_t smem = pooled_smem(n, large);
    const int problems = mode == kEigMpOnly ? Lt : Lt + P;
    if (problems < 1) return cudaErrorInvalidValue;
    if (large) {
        if (!scratch) return cudaErrorInvalidValue;
        cudaError_t e = cudaFuncSetAttribute(pooled_eig_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
        if (e != cudaSuccess) return e;
        const int ld = jacobi_ld(n);
        const int chunks = (ld + JAC_CHUNK_ROWS - 1) / JAC_CHUNK_ROWS;
        int* chol_flags = reinterpret_cast<int*>(scratch + static_cast<size_t>(problems) * ld * n);     // (pooled_eig_scratch_floats leaves room)
        if (chunks > 12) {          // beyond the register-resident cluster solver (marchenko_pastur_rank on wide features): one CTA per problem
            pooled_eig_kernel<true><<<problems, kPooledLargeThreads, smem, st>>>(stats, n, Lt, P, Mt, Ms, ranks, evals, evecs_km, evecs_cm, sweeps, scratch, 1, chol_flags, mode);
            return cudaGetLastError();
        }
        pooled_eig_kernel<true><<<problems, kPooledLargeThreads, smem, st>>>(stats, n, Lt, P, Mt, Ms, ranks, evals, evecs_km, evecs_cm, sweeps, scratch, 0, chol_flags, mode);
        e = cudaGetLastError();
        if (e != cudaSuccess) return e;
        {
            const int groups = (n + 1) / 2, per_cta = kPooledThreads / JAC_GROUP;
            if ((groups + per_cta - 1) / per_cta > 8) return cudaErrorInvalidValue;                     // at least 6 CTAs for n = 384
            using JK = void (*)(float*, int, int*);
            static const JK kerns[5] = {jacobi_cluster_global_kernel<8>, jacobi_cluster_global_kernel<9>, jacobi_cluster_global_kernel<10>,
                                        jacobi_cluster_global_kernel<11>, jacobi_cluster_global_kernel<12>};
            const JK kern = kerns[chunks < 8 ? 0 : chunks - 8];
            e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>((static_cast<size_t>(per_cta) * ld + ld + 8) * sizeof(float)));
            if (e != cudaSuccess) return e;
            const int cluster = pooled_pick_cluster(reinterpret_cast<const void*>(kern), n, problems, (ld + 8) * sizeof(float), ld);
            const int gpc = (groups + cluster - 1) / cluster;
            const size_t jsmem = (static_cast<size_t>(gpc) * ld + ld + 8) * sizeof(float);
            cudaLaunchConfig_t cfg;
            memset(&cfg, 0, sizeof cfg);
            cfg.gridDim = dim3(problems * cluster);
            cfg.blockDim = dim3(kPooledThreads);
            cfg.dynamicSmemBytes = jsmem;
            cfg.stream = st;
            cudaLaunchAttribute attr;
            attr.id = cudaLaunchAttributeClusterDimension;
            attr.val.clusterDim.x = cluster; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
            cfg.attrs = &attr;
            cfg.numAttrs = 1;
            e = cudaLaunchKernelEx(&cfg, kern, scratch, n, sweeps);
            if (e != cudaSuccess) return e;
        }
        pooled_eig_kernel<true><<<problems, kPooledLargeThreads, smem, st>>>(stats, n, Lt, P, Mt, Ms, ranks, evals, evecs_km, evecs_cm, sweeps, scratch, 2, chol_flags, mode);
        return cudaGetLastError();
    }
    cudaError_t e = cudaFuncSetAttribute(pooled_eig_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    const int cluster = pooled_pick_cluster(reinterpret_cast<const void*>(pooled_eig_kernel<false>), n, problems, smem, 0);
    cfg.gridDim = dim3(problems * cluster);
    cfg.blockDim = dim3(kPooledThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = cluster; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
    cfg.attrs = &attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, pooled_eig_kernel<false>, stats, n, Lt, P, Mt, Ms, ranks, evals, evecs_km, evecs_cm, sweeps, scratch, 1,
                              static_cast<int*>(nullptr), mode);
}

cudaError_t launch_angles(int n, int Lt, int P, const int* ranks, const float* evals, const float* evecs_km,
                          const float* evecs_cm, const float* proj_s, float* scratch, float* d2, float* gamma,
                          float* cos_out, const float* log_temp, float* w, cudaStream_t st) {
    const bool large = spectral_large(n);
    const size_t smem = angles_smem(n, large);
    cudaError_t e = large ? cudaFuncSetAttribute(angles_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem))
                          : cudaFuncSetAttribute(angles_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    if (large) angles_kernel<true><<<dim3(Lt, P), kSpectralThreads, smem, st>>>(n, Lt, P, ranks, evals, evecs_km, evecs_cm, proj_s, scratch, d2, gamma, cos_out);
    else angles_kernel<false><<<dim3(Lt, P), kSpectralThreads, smem, st>>>(n, Lt, P, ranks, evals, evecs_km, evecs_cm, proj_s, scratch, d2, gamma, cos_out);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    mix_weights_kernel<<<P, 32, 0, st>>>(d2, log_temp, Lt, P, w);
    return cudaGetLastError();
}

cudaError_t launch_selector_bwd(int n, int Lt, int P, const float* gw_raw, const float* scale_ptr, float scale_host,
                                const float* w, const float* d2, const float* log_temp, const float* gamma,
                                const float* stats, float Ms, __nv_bfloat16* gam_hi, __nv_bfloat16* gam_lo, float* corr,
                                float* grad_log_temp, cudaStream_t st) {
    const int tiles = (n * n + 255) / 256;
    selector_bwd_kernel<<<dim3(tiles < 64 ? tiles : 64, P), 256, 0, st>>>(n, Lt, P, gw_raw, scale_ptr, scale_host, w, d2, log_temp,
                                                                          gamma, stats, Ms, gam_hi, gam_lo, corr, grad_log_temp);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    selector_corr_kernel<<<dim3((n + 31) / 32, P), 256, 0, st>>>(n, Lt, stats, Ms, gam_hi, gam_lo, corr);
    return cudaGetLastError();
}

}  // namespace basd
