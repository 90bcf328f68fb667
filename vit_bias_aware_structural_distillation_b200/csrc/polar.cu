// Procrustes core of the BASD loss (relational.py:36-50 and its backward, SURVEY.md B.1) as a Newton-Schulz polar
// iteration on the tensor cores.
//
// Per (extraction point, sample):  C = s_w^T t_w  (D_s x D_t),  loss_b = tr_s + tr_t - 2 ||C||_*.
// The polar factor R of C (C = R H) gives ||C||_* = <R, C>, d||C||_*/ds_w = t_w R^T, d||C||_*/dt_w = s_w R.
// R is never formed: the iterate is kept factored as X_k = W_k t_w with W_k (D_s x N), so that with the weighted,
// centred teacher token Gram K_t = t_w t_w^T (N x N)
//     A_k = X_k X_k^T = W_k K_t W_k^T,      W_{k+1} = (a_k I + b_k A_k + c_k A_k^2) W_k,      W_0 = s_w^T / ||C||_F
// and at convergence   ||C||_* = <K_t W^T, s_w>,   d/ds_w = K_t W^T,   d/dt_w = (s_w W) t_w.
// (a_k, b_k, c_k) are the minimax odd quintics for the shrinking interval [l_k, 1.03] starting at l_0 = 3e-5
// (relative to ||C||_F): every singular value above l_0 ends within 4e-6 of 1 after 10 steps (smaller ones are left
// partially converged - they carry no weight in the nuclear norm); the 3 % head room above 1 keeps rounding from
// pushing the top singular value into the divergent region.
// All products are one-CTA-per-problem tcgen05 GEMMs on split-bf16 operands (polar_gemm.cuh).
// Requires rank(C) = D_s, i.e. D_s <= N - 1 and a teacher token Gram of rank >= D_s.
#include "cta_linalg.cuh"
#include "polar_gemm.cuh"
#include "spectral.h"

namespace basd {

namespace {

constexpr int kPolarSteps = kPolarStepsDefault;      // rows of the schedule below
// minimax odd quintics on [l_k, 1.03] (l_0 = 3e-5), each rescaled to a maximum of 1: tools/ns_schedule.py 3e-5 10 1.03
// l_k: 3.0e-5 1.0e-4 4.2e-4 1.7e-3 7.1e-3 2.9e-2 0.118 0.42 0.906 0.99967 -> 0.999996
const float kPolarCoef[kPolarSteps][3] = {
    {4.133071044f, -11.567471663f, 8.093880162f},
    {4.132779328f, -11.565168373f, 8.091968276f},
    {4.131589050f, -11.555734998f, 8.084133962f},
    {4.126671962f, -11.516778686f, 8.051782671f},
    {4.106352567f, -11.356677293f, 7.918925272f},
    {4.022478221f, -10.711657944f, 7.385453943f},
    {3.688471560f, -8.386451534f, 5.490484485f},
    {2.745572830f, -3.677073572f, 1.889197392f},
    {1.941173422f, -1.383242341f, 0.441739912f},
    {1.847826056f, -1.196240433f, 0.348410606f},
};

// Coefficients of step k out of `steps` (>= kPolarSteps): extra steps run FIRST with the l -> 0 limit polynomial (row 0 is
// within 1e-4 of it), each one lowering the floor l_0 by the polynomial's slope at zero (~4.13): 12 steps reach
// singular values of 2e-6 ||C||_F, 16 steps 6e-9 (below split-bf16 resolution).
__host__ inline const float* polar_coef(int k, int steps) {
    const int idx = k - (steps - kPolarSteps);
    return kPolarCoef[idx < 0 ? 0 : idx];
}

// eight consecutive values -> one 16-byte store per half (idx a multiple of 8)
__device__ __forceinline__ void store_split8(__nv_bfloat16* hi, __nv_bfloat16* lo, size_t idx, const float* v) {
    uint32_t hw[4], lw[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __nv_bfloat162 hv = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
        const float2 hf = __bfloat1622float2(hv);
        const __nv_bfloat162 lv = __floats2bfloat162_rn(v[2 * i] - hf.x, v[2 * i + 1] - hf.y);
        hw[i] = *reinterpret_cast<const uint32_t*>(&hv);
        lw[i] = *reinterpret_cast<const uint32_t*>(&lv);
    }
    *reinterpret_cast<uint4*>(hi + idx) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
    *reinterpret_cast<uint4*>(lo + idx) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
}

constexpr int kPrepThreads = 512;

// ------------------------------------------------------------------------------------------------
// prep_student: s_w = sqrt(a) (s - mu_s)  ->  SW [N][Ds] (split), W_0 = s_w^T [Ds][Np] (split), ksd, tr_s; one CTA per problem.
// D_s is a multiple of 8 (check_shape): the raw bf16 tile stays in shared memory as it was read (16-byte loads, 78 KB
// instead of 151 KB of fp32 -> two CTAs per SM overlap each other's load / compute / store phases) and
// s_w = sqrt(a) (s - mu) is recomputed where it is consumed; every global access is 16 bytes wide.
// ------------------------------------------------------------------------------------------------
// STAGE = false (tiles that do not fit shared memory, e.g. 576 x 384): the same passes read the tokens straight from
// global memory (L2-resident: 442 KB per problem).
// SPLIT: split-bf16 students (g.student_lo, dense): every token is read as hi + lo, before the centring; with STAGE the lo tile
// is staged behind the hi tile.
// (8 consecutive values of a raw row as fp32: hi + lo for split students)
template <bool SPLIT>
__device__ __forceinline__ void prep_ld8(const __nv_bfloat16* raw, const __nv_bfloat16* raw_lo, size_t idx, float* f) {
    const uint4 v = *reinterpret_cast<const uint4*>(raw + idx);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const float2 t = __bfloat1622float2(h[e]);
        f[2 * e] = t.x;
        f[2 * e + 1] = t.y;
    }
    if (SPLIT) {
        const uint4 u = *reinterpret_cast<const uint4*>(raw_lo + idx);
        const __nv_bfloat162* l = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float2 t = __bfloat1622float2(l[e]);
            f[2 * e] += t.x;
            f[2 * e + 1] += t.y;
        }
    }
}
template <bool STAGE, bool SPLIT = false>
__global__ void __launch_bounds__(kPrepThreads, STAGE && !SPLIT ? 2 : 1)
polar_prep_student_vec_kernel(PolarArgs g) {
    extern __shared__ __align__(16) uint8_t sm_raw[];
    const int N = g.Ns, D = g.Ds, pitch = STAGE ? D + 8 : D, oct = D / 8;      // pitch in bf16: rows stay 16-byte aligned
    const size_t tile_bytes = STAGE ? ((static_cast<size_t>(N) * pitch * 2 + 15) & ~size_t(15)) : 0;
    float* a_s = reinterpret_cast<float*>(sm_raw + (SPLIT ? 2 : 1) * tile_bytes);
    float* q_s = a_s + N;
    float* mu = q_s + N;                                            // [D]
    float* red = mu + D;                                            // 40
    float* partial = red + 40;                                      // [slices][D]
    const int prob = blockIdx.x;
    const int i = prob / g.B, b = prob % g.B;
    const __nv_bfloat16* S = g.student[i] + static_cast<size_t>(b) * g.student_bs;
    const __nv_bfloat16* S_lo = SPLIT ? g.student_lo[i] + static_cast<size_t>(b) * g.student_bs : nullptr;
    const __nv_bfloat16* raw = STAGE ? reinterpret_cast<const __nv_bfloat16*>(sm_raw) : S;      // [N][pitch]
    const __nv_bfloat16* raw_lo = STAGE ? reinterpret_cast<const __nv_bfloat16*>(sm_raw + tile_bytes) : S_lo;
    for (int n = threadIdx.x; n < N; n += blockDim.x) {
        const float a = g.a[static_cast<size_t>(prob) * N + n];
        a_s[n] = a;
        q_s[n] = sqrtf(a);
    }
    if (STAGE) {
        __nv_bfloat16* stage = reinterpret_cast<__nv_bfloat16*>(sm_raw);
        for (int t = threadIdx.x; t < N * oct; t += blockDim.x) {
            const int n = t / oct, o = t - n * oct;
            *reinterpret_cast<uint4*>(stage + n * pitch + o * 8) = *reinterpret_cast<const uint4*>(S + static_cast<size_t>(n) * D + o * 8);
            if (SPLIT)
                *reinterpret_cast<uint4*>(stage + tile_bytes / 2 + n * pitch + o * 8) = *reinterpret_cast<const uint4*>(S_lo + static_cast<size_t>(n) * D + o * 8);
        }
    }
    __syncthreads();
    // mu[d] = sum_n a[n] s[n][d]: thread = (octet of d, slice of n)
    const int slices = blockDim.x / oct;
    {
        const int o = threadIdx.x % oct, sl = threadIdx.x / oct;
        if (sl < slices) {
            float m[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            for (int n = sl; n < N; n += slices) {
                float f[8];
                prep_ld8<SPLIT>(raw, raw_lo, static_cast<size_t>(n) * pitch + o * 8, f);
                const float an = a_s[n];
#pragma unroll
                for (int e = 0; e < 8; ++e) m[e] = fmaf(an, f[e], m[e]);
            }
#pragma unroll
            for (int e = 0; e < 8; ++e) partial[sl * D + o * 8 + e] = m[e];
        }
    }
    __syncthreads();
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
        float m = 0.f;
        for (int sl = 0; sl < slices; ++sl) m += partial[sl * D + d];
        mu[d] = m;
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    // row norms of s_w
    float* ksd = g.vec + static_cast<size_t>(prob) * 4 * N;
    float part = 0.f;
    for (int n = warp; n < N; n += nw) {
        float s = 0.f;
        const float qn = q_s[n];
        for (int o = lane; o < oct; o += 32) {
            float f[8];
            prep_ld8<SPLIT>(raw, raw_lo, static_cast<size_t>(n) * pitch + o * 8, f);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float x = qn * (f[2 * e] - mu[o * 8 + 2 * e]), y = qn * (f[2 * e + 1] - mu[o * 8 + 2 * e + 1]);
                s = fmaf(x, x, fmaf(y, y, s));
            }
        }
        s = warp_sum(s);
        if (lane == 0) { ksd[n] = s; part += s; }
    }
    const float tr_s = cta_sum(part, red);
    if (threadIdx.x == 0) g.scal[prob * 4 + 1] = tr_s;
    // SW = s_w [N][Ds], tiled [d block][n][64]: a thread takes 8 consecutive d of one row
    __nv_bfloat16* swh = g.SW.hi + prob * g.SW.batch_stride;
    __nv_bfloat16* swl = g.SW.lo + prob * g.SW.batch_stride;
    const int n_cb = (D + 63) / 64;
    for (int t = threadIdx.x; t < n_cb * N * 8; t += blockDim.x) {
        const int j0 = (t & 7) * 8, n = (t >> 3) % N, cb = (t >> 3) / N;
        const int d0 = cb * 64 + j0;
        float v[8];
        if (d0 < D) {
            float f[8];
            prep_ld8<SPLIT>(raw, raw_lo, static_cast<size_t>(n) * pitch + d0, f);
            const float qn = q_s[n];
#pragma unroll
            for (int e = 0; e < 8; ++e) v[e] = qn * (f[e] - mu[d0 + e]);
        } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) v[e] = 0.f;
        }
        store_split8(swh, swl, (static_cast<size_t>(cb) * N + n) * 64 + j0, v);
    }
    if (g.vt) return;
    // W_0 = s_w^T [Ds][N], tiled [n block][d][64], padding columns zero: a thread takes 8 consecutive n of one d; lanes run
    // along d (conflict-free 2-byte shared reads; the 16-byte stores of a warp land 128 B apart and are merged in L2).
    // (Walking (row, block) incrementally instead of dividing the flat index - a warp per octet of n here, running indices in the
    // loop above and in prep_teacher - was measured: 0.31 -> 0.30 ms at cfg2, 1.25 -> 1.67 ms at cfg5, where the tile is read
    // from global memory and the flat order keeps neighbouring warps on the same lines; taken out.)
    __nv_bfloat16* wh = g.W.hi + prob * g.W.batch_stride;
    __nv_bfloat16* wl = g.W.lo + prob * g.W.batch_stride;
    const int n_nb = (N + 63) / 64;
    for (int t = threadIdx.x; t < n_nb * 8 * D; t += blockDim.x) {
        const int d = t % D, j0 = ((t / D) & 7) * 8, nb = t / (8 * D);
        const float md = mu[d];
        float v[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int n = nb * 64 + j0 + e;
            float x = 0.f;
            if (n < N) {
                x = __bfloat162float(raw[n * pitch + d]);
                if (SPLIT) x += __bfloat162float(raw_lo[n * pitch + d]);
            }
            v[e] = n < N ? q_s[n] * (x - md) : 0.f;
        }
        store_split8(wh, wl, (static_cast<size_t>(nb) * D + d) * 64 + j0, v);
    }
}

// ------------------------------------------------------------------------------------------------
// prep_teacher: K_t = q (Ktt - m 1^T - 1 m^T + mm) q  (weighted + centred token Gram, split), diag, tr_t
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
polar_prep_teacher_kernel(PolarArgs g) {
    extern __shared__ float sm[];
    const int N = g.Ns;
    float* a_s = sm;                 // [N]
    float* q_s = a_s + N;
    float* m_s = q_s + N;
    float* red = m_s + N;            // 40
    const int prob = blockIdx.x;
    const float* Ktt = g.Ktt + static_cast<size_t>(prob) * N * N;
    for (int n = threadIdx.x; n < N; n += blockDim.x) {
        const float a = g.a[static_cast<size_t>(prob) * N + n];
        a_s[n] = a;
        q_s[n] = sqrtf(a);
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int n = warp; n < N; n += nw) {
        float s = 0.f;
        for (int m = lane; m < N; m += 32) s = fmaf(Ktt[static_cast<size_t>(n) * N + m], a_s[m], s);
        s = warp_sum(s);
        if (lane == 0) m_s[n] = s;
    }
    __syncthreads();
    float part = 0.f;
    for (int n = threadIdx.x; n < N; n += blockDim.x) part += a_s[n] * m_s[n];
    const float mm = cta_sum(part, red);
    float* ktd = g.vec + static_cast<size_t>(prob) * 4 * N + N;
    part = 0.f;
    for (int n = threadIdx.x; n < N; n += blockDim.x) {
        const float v = a_s[n] * (Ktt[static_cast<size_t>(n) * N + n] - 2.f * m_s[n] + mm);
        ktd[n] = v;
        part += v;
    }
    const float tr_t = cta_sum(part, red);
    if (threadIdx.x == 0) g.scal[prob * 4 + 2] = tr_t;
    __nv_bfloat16* kh = g.Kt.hi + prob * g.Kt.batch_stride;
    __nv_bfloat16* kl = g.Kt.lo + prob * g.Kt.batch_stride;
    // storage order [col block][row n][64]: a thread takes 8 consecutive columns of one row (two 16-byte loads of Ktt when
    // N is a multiple of 4, one 16-byte store per half); the second read of Ktt comes from L2
    const int n_cb = (N + 63) / 64;
    const bool vec_ok = (N & 3) == 0;
    for (int t = threadIdx.x; t < n_cb * N * 8; t += blockDim.x) {
        const int j0 = (t & 7) * 8, n = (t >> 3) % N, cb = (t >> 3) / N;
        const int m0 = cb * 64 + j0;
        float v[8];
        const float* row = Ktt + static_cast<size_t>(n) * N;
        if (vec_ok && m0 + 8 <= N) {
            const float4 k0 = *reinterpret_cast<const float4*>(row + m0), k1 = *reinterpret_cast<const float4*>(row + m0 + 4);
            v[0] = k0.x; v[1] = k0.y; v[2] = k0.z; v[3] = k0.w; v[4] = k1.x; v[5] = k1.y; v[6] = k1.z; v[7] = k1.w;
        } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) v[e] = m0 + e < N ? row[m0 + e] : 0.f;
        }
        const float qn = q_s[n], mn = m_s[n] - mm;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int m = m0 + e;
            v[e] = m < N ? qn * q_s[m] * (v[e] - mn - m_s[m]) : 0.f;
        }
        store_split8(kh, kl, (static_cast<size_t>(cb) * N + n) * 64 + j0, v);
    }
}

// ------------------------------------------------------------------------------------------------
// finish: nuclear norm, direct student gradient, importance gradient, per-sample loss
//   Gsw = K_t W^T = d nuc / d s_w  [N][Ds]
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
polar_finish_kernel(PolarArgs g) {
    extern __shared__ float sm[];
    const int N = g.Ns, D = g.Ds;
    float* dots = sm;                // [N]
    float* ga = dots + N;            // [N]
    float* red = ga + N;             // 40
    const int prob = blockIdx.x;
    const float* G = g.Gsw + static_cast<size_t>(prob) * N * D;
    const __nv_bfloat16* swh = g.SW.hi + prob * g.SW.batch_stride;
    const __nv_bfloat16* swl = g.SW.lo + prob * g.SW.batch_stride;
    const float* a = g.a + static_cast<size_t>(prob) * N;
    float* gdir = g.gdir + static_cast<size_t>(prob) * N * D;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    if ((D & 7) == 0) {
        // a lane takes 8 consecutive d of one row: 16-byte loads of both halves of s_w, 2 x 16-byte loads of Gsw, 2 x 16-byte
        // stores of gdir; a warp covers 256 columns per pass
        // (the grid is a single wave, so the kernel lasts as long as one warp's chain of rows: four rows are in flight)
        constexpr int RU = 4;
        for (int n0 = warp * RU; n0 < N; n0 += nw * RU) {
            float s[RU];
#pragma unroll
            for (int u = 0; u < RU; ++u) s[u] = 0.f;
            for (int d0 = lane * 8; d0 < D; d0 += 256) {
                uint4 h[RU], l[RU];
                float4 g0[RU], g1[RU];
#pragma unroll
                for (int u = 0; u < RU; ++u) {
                    const int n = n0 + u < N ? n0 + u : N - 1;
                    const size_t idx = g.SW.at(n, d0);
                    h[u] = *reinterpret_cast<const uint4*>(swh + idx);
                    l[u] = *reinterpret_cast<const uint4*>(swl + idx);
                    g0[u] = *reinterpret_cast<const float4*>(G + static_cast<size_t>(n) * D + d0);
                    g1[u] = *reinterpret_cast<const float4*>(G + static_cast<size_t>(n) * D + d0 + 4);
                }
#pragma unroll
                for (int u = 0; u < RU; ++u) {
                    if (n0 + u < N) {
                        const int n = n0 + u;
                        const float qn = sqrtf(a[n]);
                        const __nv_bfloat162* hp = reinterpret_cast<const __nv_bfloat162*>(&h[u]);
                        const __nv_bfloat162* lp = reinterpret_cast<const __nv_bfloat162*>(&l[u]);
                        float sw[8];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const float2 x = __bfloat1622float2(hp[e]), y = __bfloat1622float2(lp[e]);
                            sw[2 * e] = x.x + y.x; sw[2 * e + 1] = x.y + y.y;
                        }
                        const float gv[8] = {g0[u].x, g0[u].y, g0[u].z, g0[u].w, g1[u].x, g1[u].y, g1[u].z, g1[u].w};
                        float o[8];
#pragma unroll
                        for (int e = 0; e < 8; ++e) { s[u] = fmaf(sw[e], gv[e], s[u]); o[e] = qn * (2.f * sw[e] - 2.f * gv[e]); }
                        float* od = gdir + static_cast<size_t>(n) * D + d0;
                        *reinterpret_cast<float4*>(od) = make_float4(o[0], o[1], o[2], o[3]);
                        *reinterpret_cast<float4*>(od + 4) = make_float4(o[4], o[5], o[6], o[7]);
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < RU; ++u) {
                const float t = warp_sum(s[u]);
                if (lane == 0 && n0 + u < N) dots[n0 + u] = t;
            }
        }
    } else {
        for (int n = warp; n < N; n += nw) {
            const float qn = sqrtf(a[n]);
            float s = 0.f;
            for (int d = lane; d < D; d += 32) {
                const size_t idx = g.SW.at(n, d);
                const float sw = __bfloat162float(swh[idx]) + __bfloat162float(swl[idx]);
                const float gv = G[static_cast<size_t>(n) * D + d];
                s = fmaf(sw, gv, s);
                gdir[static_cast<size_t>(n) * D + d] = qn * (2.f * sw - 2.f * gv);
            }
            s = warp_sum(s);
            if (lane == 0) dots[n] = s;
        }
    }
    __syncthreads();
    const float* ksd = g.vec + static_cast<size_t>(prob) * 4 * N;
    const float* ktd = ksd + N;
    float p_nuc = 0.f, p_gdot = 0.f;
    for (int n = threadIdx.x; n < N; n += blockDim.x) {
        p_nuc += dots[n];
        const float v = (ksd[n] + ktd[n] - 2.f * dots[n]) / a[n];
        ga[n] = v;
        p_gdot += v * a[n];
    }
    const float nuc = cta_sum(p_nuc, red);
    const float gdot = cta_sum(p_gdot, red);
    const float inv_ssum = 1.f / g.ssum[prob];
    for (int n = threadIdx.x; n < N; n += blockDim.x) g.gwt[static_cast<size_t>(prob) * N + n] = (ga[n] - gdot) * inv_ssum;
    if (threadIdx.x == 0) {
        const float tr_s = g.scal[prob * 4 + 1], tr_t = g.scal[prob * 4 + 2];
        g.loss_b[prob] = tr_s + tr_t - 2.f * nuc;
        if (g.dbg) {
            g.dbg[prob * 5 + 0] = nuc; g.dbg[prob * 5 + 1] = tr_s; g.dbg[prob * 5 + 2] = tr_t;
            float fro = 0.f, rs = 0.f;
            for (int sl = 0; sl < g.fro_slots; ++sl) {
                fro += g.fro2[static_cast<size_t>(prob) * g.fro_slots + sl];
                rs += g.resid[static_cast<size_t>(prob) * g.fro_slots + sl];
            }
            // convergence evidence: ||X X^T - I||_F going INTO the last step (every |sigma^2 - 1| is below it; <= 0.1 means the
            // last polynomial leaves every singular value within 1e-3 of 1); NaN-safe: a NaN residual stays NaN
            g.dbg[prob * 5 + 3] = sqrtf(rs); g.dbg[prob * 5 + 4] = fro;
        }
    }
}

// ================================================================================================
// Teacher-token-space form  (D_s > min(N_s, N_t) - 1 with N_t <= N_s: the cross-covariance C = s_w^T t_w has rank
// N_t - 1 < D_s, e.g. a 7 x 7 CNN grid against a ViT-S student, or ViT-S <- ViT-L at 196 tokens).
//
// t_w = F Tbar with F = diag(q)(I - 1 a^T) E  [N_s x N_t]  (E = the 2-tap token resampling, I when N_t == N_s),
// Tbar the mixed teacher on its OWN token grid.  F 1 = 0, so C = s_w^T F Tbar_c with Tbar_c = (I - 1 1^T / N_t) Tbar.
// With K_R = Tbar_c Tbar_c^T + c_r 1^ 1^^T = G G^T (Cholesky, N_t x N_t; 1^ = 1 / sqrt(N_t) decouples the common null
// direction) the rows of Q^T = G^-1 [Tbar_c, sqrt(c_r) 1^] are orthonormal, so
//     C^+ = X_0^T Q^T,   X_0 = G^T F^T s_w  (N_t x D_s)  plus one decoupled column beta z^ (z^ = G^T 1^ / sqrt(c_r)),
//     polar(C) = X_inf^T G^-1 Tbar_c,     ||C||_* = <X_inf, X_0>,
//     d||C||_* / d s_w = F G X_inf,       d L_b / d Tbar = [2 F^T F - 2 G^-T (X_0 X_inf^T) G^-1 (I - 1 1^T / N_t)] Tbar.
// X_inf = polar factor of X_0^+ by the plain Newton-Schulz iteration on X itself (A = X X^T is symmetric positive
// semi-definite by construction; the factored form W K W^T of the student-feature form loses definiteness to the
// rounding of K when K is ill conditioned).  tools/scratch/vt_model.py states this pipeline in fp64 against autograd.
// ================================================================================================
constexpr int kVtThreads = 512;
__global__ void __launch_bounds__(kVtThreads, 1)
vt_prep_teacher_kernel(PolarArgs g) {
    extern __shared__ __align__(16) float sm[];
    const int N = g.Ns, M = g.Nt, ld = (M + 3) & ~3;
    float* K = sm;                                        // [M][ld] column-major: element (r, c) at K[c * ld + r]
    float* a_s = K + static_cast<size_t>(ld) * M;         // [N]
    float* q_s = a_s + N;                                 // [N]
    float* ebar = q_s + N;                                // [M]   E^T a
    float* eg = ebar + M;                                 // [M]   ebar^T G
    float* rowm = eg + M;                                 // [M]
    float* red = rowm + M;                                // 40
    __shared__ int s_bad;
    const int prob = blockIdx.x;
    const float* Ktt = g.Ktt + static_cast<size_t>(prob) * M * M;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int n = threadIdx.x; n < N; n += blockDim.x) {
        const float a = g.a[static_cast<size_t>(prob) * N + n];
        a_s[n] = a;
        q_s[n] = sqrtf(a);
    }
    for (int t = threadIdx.x; t < M * ld; t += blockDim.x) {
        const int c = t / ld, r = t - c * ld;
        K[t] = r < M ? 0.5f * (Ktt[static_cast<size_t>(r) * M + c] + Ktt[static_cast<size_t>(c) * M + r]) : 0.f;
    }
    if (threadIdx.x < M) ebar[threadIdx.x] = 0.f;
    if (threadIdx.x == 0) s_bad = 0;
    __syncthreads();
    // double centring + the decoupling term: K_R = H K H + (tr(H K H) / M) 1^ 1^^T
    for (int i = warp; i < M; i += nw) {
        float sacc = 0.f;
        for (int j = lane; j < M; j += 32) sacc += K[j * ld + i];
        sacc = warp_sum(sacc);
        if (lane == 0) rowm[i] = sacc / static_cast<float>(M);
    }
    __syncthreads();
    float part = 0.f;
    for (int i = threadIdx.x; i < M; i += blockDim.x) part += rowm[i];
    const float tot = cta_sum(part, red) / static_cast<float>(M);
    part = 0.f;
    for (int i = threadIdx.x; i < M; i += blockDim.x) part += K[i * ld + i] - 2.f * rowm[i] + tot;
    const float cr = cta_sum(part, red) / static_cast<float>(M);
    const float shift = tot + cr / static_cast<float>(M);
    for (int t = threadIdx.x; t < M * ld; t += blockDim.x) {
        const int c = t / ld, r = t - c * ld;
        if (r < M) K[t] += shift - rowm[r] - rowm[c];
    }
    __syncthreads();
    float dmax = 0.f;
    for (int i = threadIdx.x; i < M; i += blockDim.x) dmax = fmaxf(dmax, K[i * ld + i]);
    for (int o = 16; o > 0; o >>= 1) dmax = fmaxf(dmax, __shfl_xor_sync(0xffffffffu, dmax, o));
    if (lane == 0) red[warp] = dmax;
    __syncthreads();
    dmax = 0.f;
    for (int wv = 0; wv < nw; ++wv) dmax = fmaxf(dmax, red[wv]);
    __syncthreads();
    cta_cholesky_lower(K, ld, M, &s_bad, 1e-6f * dmax);   // K = G (lower), strict upper triangle zeroed
    // ebar = E^T a   (one thread per teacher token walks the student tokens in order: no atomics, bitwise repeatable)
    for (int m = threadIdx.x; m < M; m += blockDim.x) {
        float sacc = 0.f;
        for (int n = 0; n < N; ++n) {
            int i0, i1; float lam;
            interp_index(n, M, N, i0, i1, lam);
            if (i0 == m) sacc = fmaf(a_s[n], 1.f - lam, sacc);
            if (i1 == m && lam != 0.f) sacc = fmaf(a_s[n], lam, sacc);
        }
        ebar[m] = sacc;
    }
    __syncthreads();
    // eg[m] = sum_m' ebar[m'] G[m'][m];  z^[m] = sum_m' G[m'][m] / sqrt(M c_r)   (column m of G = K[m * ld + .])
    float* zhat = g.vec + static_cast<size_t>(prob) * 4 * N + 2 * N;
    for (int m = warp; m < M; m += nw) {
        float se = 0.f, sz = 0.f;
        for (int i = lane; i < M; i += 32) { const float gv = K[m * ld + i]; se = fmaf(ebar[i], gv, se); sz += gv; }
        se = warp_sum(se); sz = warp_sum(sz);
        if (lane == 0) { eg[m] = se; zhat[m] = sz * rsqrtf(static_cast<float>(M) * cr); }
    }
    __syncthreads();
    // F G [N][M] -> FG (rows N, inner M) and FGt (rows M, inner N), padding columns zero; ktd[n] = |(F G)[n]|^2
    float* ktd = g.vec + static_cast<size_t>(prob) * 4 * N + N;
    part = 0.f;
    for (int n = warp; n < N; n += nw) {
        int i0, i1; float lam;
        interp_index(n, M, N, i0, i1, lam);
        float sacc = 0.f;
        for (int m = lane; m < M; m += 32) {
            const float v = q_s[n] * ((1.f - lam) * K[m * ld + i0] + lam * K[m * ld + i1] - eg[m]);
            sacc = fmaf(v, v, sacc);
        }
        sacc = warp_sum(sacc);
        if (lane == 0) { ktd[n] = sacc; part += sacc; }
    }
    const float tr_t = cta_sum(part, red);
    if (threadIdx.x == 0) g.scal[prob * 4 + 2] = tr_t;
    {
        __nv_bfloat16* fh = g.FG.hi + prob * g.FG.batch_stride;
        __nv_bfloat16* fl = g.FG.lo + prob * g.FG.batch_stride;
        const int n_cb = (M + 63) / 64;
        for (int t = threadIdx.x; t < n_cb * N * 8; t += blockDim.x) {
            const int j0 = (t & 7) * 8, n = (t >> 3) % N, cb = (t >> 3) / N;
            int i0, i1; float lam;
            interp_index(n, M, N, i0, i1, lam);
            float v[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const int m = cb * 64 + j0 + e;
                v[e] = m < M ? q_s[n] * ((1.f - lam) * K[m * ld + i0] + lam * K[m * ld + i1] - eg[m]) : 0.f;
            }
            store_split8(fh, fl, (static_cast<size_t>(cb) * N + n) * 64 + j0, v);
        }
        __nv_bfloat16* th = g.FGt.hi + prob * g.FGt.batch_stride;
        __nv_bfloat16* tl = g.FGt.lo + prob * g.FGt.batch_stride;
        const int n_nb = (N + 63) / 64;
        for (int t = threadIdx.x; t < n_nb * 8 * M; t += blockDim.x) {
            const int m = t % M, j0 = ((t / M) & 7) * 8, nb = t / (8 * M);
            float v[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const int n = nb * 64 + j0 + e;
                float x = 0.f;
                if (n < N) {
                    int i0, i1; float lam;
                    interp_index(n, M, N, i0, i1, lam);
                    x = q_s[n] * ((1.f - lam) * K[m * ld + i0] + lam * K[m * ld + i1] - eg[m]);
                }
                v[e] = x;
            }
            store_split8(th, tl, (static_cast<size_t>(nb) * M + m) * 64 + j0, v);
        }
    }
    // F^T F = E^T diag(a) E - ebar ebar^T   (banded + rank one; fp32, read by vt_theta_kernel)
    float* ftf = g.ftf + static_cast<size_t>(prob) * M * M;
    for (int t = threadIdx.x; t < M * M; t += blockDim.x) ftf[t] = -ebar[t / M] * ebar[t % M];
    __syncthreads();
    // E^T diag(a) E is tridiagonal (two taps per student token): thread u owns (u, u) and (u, u + 1) = (u + 1, u)
    for (int u = threadIdx.x; u < M; u += blockDim.x) {
        float d0 = 0.f, d1 = 0.f;
        for (int n = 0; n < N; ++n) {
            int i0, i1; float lam;
            interp_index(n, M, N, i0, i1, lam);
            const float w0 = 1.f - lam, a = a_s[n];
            if (i0 == u) d0 = fmaf(a, w0 * w0, d0);
            if (lam != 0.f) {
                if (i1 == u) d0 = fmaf(a, lam * lam, d0);
                if (i0 == u && i1 == u + 1) d1 = fmaf(a, w0 * lam, d1);
                if (i0 == u && i1 == u) d0 = fmaf(a, 2.f * w0 * lam, d0);
            }
        }
        ftf[u * M + u] += d0;
        if (u + 1 < M) { ftf[u * M + u + 1] += d1; ftf[(u + 1) * M + u] += d1; }
    }
    // G^-1 in place of G (G is dead from here on; row-by-row substitution in shared memory), then its two operand forms
    __syncthreads();
    cta_lower_inverse_inplace(K, ld, M);
    const float* ginv = K;                                // column-major: G^-1(r, c) = ginv[c * ld + r], zero above the diagonal
    for (int r = threadIdx.x; r < M; r += blockDim.x) {
        float sacc = 0.f;
        for (int c = 0; c <= r; ++c) sacc += ginv[c * ld + r];
        rowm[r] = sacc / static_cast<float>(M);
    }
    __syncthreads();
    {
        __nv_bfloat16* ch = g.GinvC.hi + prob * g.GinvC.batch_stride;
        __nv_bfloat16* cl = g.GinvC.lo + prob * g.GinvC.batch_stride;
        __nv_bfloat16* th = g.GinvT.hi + prob * g.GinvT.batch_stride;
        __nv_bfloat16* tl = g.GinvT.lo + prob * g.GinvT.batch_stride;
        const int n_cb = (M + 63) / 64;
        for (int t = threadIdx.x; t < n_cb * M * 8; t += blockDim.x) {
            const int r = t % M, j0 = ((t / M) & 7) * 8, cb = t / (8 * M);
            float vc[8], vt[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const int c = cb * 64 + j0 + e;
                // GinvC[r][c] = Ginv(r, c) - rowmean(r);   GinvT[r][c] = Ginv(c, r)
                vc[e] = c < M ? (c <= r ? ginv[c * ld + r] : 0.f) - rowm[r] : 0.f;
                vt[e] = c < M ? (r <= c ? ginv[r * ld + c] : 0.f) : 0.f;
            }
            store_split8(ch, cl, (static_cast<size_t>(cb) * M + r) * 64 + j0, vc);
            store_split8(th, tl, (static_cast<size_t>(cb) * M + r) * 64 + j0, vt);
        }
    }
}

// ||X_0||_F^2 -> the decoupled augmentation column beta z^ at column Ds16 of X_0 (beta = rms of the other singular values)
__global__ void __launch_bounds__(256)
vt_augment_kernel(PolarArgs g) {
    __shared__ float red[40];
    const int M = g.Nt, D = g.Ds, N = g.Ns;
    const int prob = blockIdx.x;
    __nv_bfloat16* xh = g.X0.hi + prob * g.X0.batch_stride;
    __nv_bfloat16* xl = g.X0.lo + prob * g.X0.batch_stride;
    float part = 0.f;
    const int data_elems = ((D + 63) / 64) * M * 64;              // column blocks the product wrote (padding columns are zero)
    for (int t = threadIdx.x; t < data_elems / 2; t += blockDim.x) {
        const float2 h = __bfloat1622float2(reinterpret_cast<const __nv_bfloat162*>(xh)[t]);
        const float2 l = __bfloat1622float2(reinterpret_cast<const __nv_bfloat162*>(xl)[t]);
        const float x = h.x + l.x, y = h.y + l.y;
        part = fmaf(x, x, fmaf(y, y, part));
    }
    const float fro2 = cta_sum(part, red);
    const float beta = sqrtf(fro2 / static_cast<float>(M > 1 ? M - 1 : 1));
    const float* zhat = g.vec + static_cast<size_t>(prob) * 4 * N + 2 * N;
    const int d16 = (D + 15) & ~15, dend = (g.Dsp + 63) & ~63;
    for (int t = threadIdx.x; t < M * (dend - D); t += blockDim.x) {
        const int m = t % M, c = D + t / M;
        const float v = c == d16 ? beta * zhat[m] : 0.f;
        const size_t idx = g.X0.at(m, c);
        const __nv_bfloat16 h = __float2bfloat16(v);
        xh[idx] = h;
        xl[idx] = __float2bfloat16(v - __bfloat162float(h));
    }
}

// Theta'' = 2 F^T F - 2 G^-T (X_0 X_inf^T) G^-1 (I - 1 1^T / N_t)  -> row-major split pair [Nt][NtPad]
__global__ void __launch_bounds__(256)
vt_theta_kernel(PolarArgs g) {
    const int M = g.Nt;
    const size_t prob = blockIdx.y;
    const float* ftf = g.ftf + prob * M * M;
    const float* raw = g.thraw + prob * M * M;
    __nv_bfloat16* oh = g.theta + prob * M * g.NtPad;
    __nv_bfloat16* ol = g.theta_lo + prob * M * g.NtPad;
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < M * M; t += gridDim.x * blockDim.x) {
        const int i = t / M, j = t - i * M;
        const float v = 2.f * ftf[t] - 2.f * raw[t];
        const __nv_bfloat16 h = __float2bfloat16(v);
        oh[static_cast<size_t>(i) * g.NtPad + j] = h;
        ol[static_cast<size_t>(i) * g.NtPad + j] = __float2bfloat16(v - __bfloat162float(h));
    }
}

}  // namespace

int polar_steps() { return kPolarSteps; }
// slots for the per-warp partial traces of the first A product: 4 epilogue warps x row tiles x column tiles (column
// tiles are at least 128 wide); rounded up to a multiple of 8
int polar_fro_slots(int core) {
    const int t = (core + 127) / 128;
    return (4 * t * t + 7) & ~7;
}
int polar_launches_per_step(int Ds, int Ns) { return polar_fused_supported(Ds, Ns) ? 3 : 4; }

#define PCK(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) return _e; } while (0)

// prep_student (both polar forms): the raw token tile is staged in shared memory when it fits (split-bf16
// students stage their lo tile too), otherwise read from global memory
template <bool SPLIT>
static cudaError_t launch_prep_student_vec(const PolarArgs& g, cudaStream_t st) {
    const int N = g.Ns, D = g.Ds, nprob = g.n_problems;
    const int slices = kPrepThreads / (D / 8);
    const size_t small = (2 * N + D + 40 + static_cast<size_t>(slices) * D) * sizeof(float);
    const size_t smem = (SPLIT ? 2 : 1) * ((static_cast<size_t>(N) * (D + 8) * 2 + 15) & ~size_t(15)) + small;
    if (smem <= 227 * 1024) {
        PCK(cudaFuncSetAttribute(polar_prep_student_vec_kernel<true, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
        polar_prep_student_vec_kernel<true, SPLIT><<<nprob, kPrepThreads, smem, st>>>(g);
    } else {
        PCK(cudaFuncSetAttribute(polar_prep_student_vec_kernel<false, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(small)));
        polar_prep_student_vec_kernel<false, SPLIT><<<nprob, kPrepThreads, small, st>>>(g);
    }
    return cudaGetLastError();
}
static cudaError_t launch_prep_student_vec(const PolarArgs& g, cudaStream_t st) {
    return g.student_lo[0] ? launch_prep_student_vec<true>(g, st) : launch_prep_student_vec<false>(g, st);
}

cudaError_t launch_polar_procrustes(const PolarArgs& g, cudaStream_t st) {
    const int N = g.Ns, D = g.Ds, nprob = g.n_problems;
    {
        TimingScope ts(kSlotPolarPrep, st, 2);
        PCK(launch_prep_student_vec(g, st));
        polar_prep_teacher_kernel<<<nprob, 256, (3 * N + 64) * sizeof(float), st>>>(g);
        PCK(cudaGetLastError());
    }
    // partial traces of the first A = T W^T per problem (their sum = ||C||_F^2)
    PCK(cudaMemsetAsync(g.fro2, 0, sizeof(float) * nprob * g.fro_slots, st));

    // The chain of products is sequentially dependent per problem; every launch batches all problems.
    const bool fused = polar_fused_supported(D, N);
    const int steps = g.steps >= kPolarStepsMin && g.steps <= kPolarStepsMax ? g.steps : kPolarSteps;
    PCK(cudaMemsetAsync(g.resid, 0, sizeof(float) * nprob * g.fro_slots, st));
    {
        TimingScope ts(kSlotPolarGemm, st, (fused ? 3 : 4) * steps + 2);
        // Step 0 runs on the unnormalised W_0 = s_w^T; r = 1 / ||C||_F^2 (trace of W_0 K_t W_0^T, accumulated by the first
        // A product) enters the later epilogues of that step as a per-problem scalar.
        SplitMat Wc = g.W, Wn = g.W2;
        const SplitMat &T = g.T, &A = g.A, &Bm = g.Bm, &Kt = g.Kt;
        int dir = 0;                           // alternate the problem order launch by launch (L2 reuse of the previous output)
        for (int k = 0; k < steps; ++k) {
            const float* coef = polar_coef(k, steps);
            const float ca = coef[0], cb = coef[1], cc = coef[2];
            const bool first = k == 0, last = k == steps - 1;
            const float* norm = first ? g.fro2 : nullptr;
            PolarGemmArgs a;
            // G1: T = W K_t
            memset(&a, 0, sizeof a);
            a.epi = PG_EPI_SPLIT; a.out_hi = T.hi; a.out_lo = T.lo; a.out_stride = T.batch_stride; a.scale_c = 1.f;
            a.reverse = (dir++) & 1;
            PCK(polar_gemm(false, Wc, Kt, nprob, a, st));
            if (fused) {
                // G2 + G3 in one kernel: A = T W^T stays in TMEM / shared memory, Bm = a I + b (rA) + c (rA)^2 leaves
                // (step 0: trace(A) = ||C||_F^2 is reduced inside and written to fro2 for G4's epilogue)
                PolarFusedArgs f;
                memset(&f, 0, sizeof f);
                f.ca = ca; f.cb = cb; f.cc = cc; f.first = first ? 1 : 0; f.fro2 = g.fro2; f.fro_slots = g.fro_slots;
                f.resid = last ? g.resid : nullptr;
                f.reverse = (dir++) & 1;
                PCK(polar_fused_abm(T, Wc, Bm, nprob, f, st));
            } else {
                // G2: A = T W^T                (step 0: trace(A) = ||C||_F^2, read by the epilogues of G3 / G4 of that step)
                memset(&a, 0, sizeof a);
                a.epi = PG_EPI_SPLIT; a.out_hi = A.hi; a.out_lo = A.lo; a.out_stride = A.batch_stride; a.scale_c = 1.f;
                if (first) { a.trace = g.fro2; a.fro_slots = g.fro_slots; }
                a.reverse = (dir++) & 1;
                PCK(polar_gemm(false, T, Wc, nprob, a, st));
                // G3: Bm = a I + b (rA) + c (rA)^2   (A is both operands: the A tile aliases the B tile; the b A term is added from
                //     a TMA-loaded copy of the output-shaped tile of A in the epilogue)
                memset(&a, 0, sizeof a);
                a.epi = PG_EPI_SPLIT; a.out_hi = Bm.hi; a.out_lo = Bm.lo; a.out_stride = Bm.batch_stride;
                a.a_alias_b = 1; a.aux_mode = 1; a.aux_hi = A.hi; a.aux_lo = A.lo;
                a.aux_c = cb; a.aux_p = first ? 1.f : 0.f; a.scale_c = cc; a.scale_p = first ? 2.f : 0.f; a.diag_add = ca; a.norm2 = norm; a.fro_slots = g.fro_slots;
                a.resid = last ? g.resid : nullptr;
                a.reverse = (dir++) & 1;
                PCK(polar_gemm(false, A, A, nprob, a, st));
            }
            // G4: W_next = sqrt(r) Bm W      (W enters as the MN-major B operand; ping-pong buffers)
            memset(&a, 0, sizeof a);
            a.epi = PG_EPI_SPLIT; a.out_hi = Wn.hi; a.out_lo = Wn.lo; a.out_stride = Wn.batch_stride;
            a.scale_c = 1.f; a.scale_p = first ? 0.5f : 0.f; a.norm2 = norm; a.fro_slots = g.fro_slots;
            a.reverse = (dir++) & 1;
            PCK(polar_gemm(true, Bm, Wc, nprob, a, st));
            const SplitMat tmp = Wc; Wc = Wn; Wn = tmp;
        }
        PolarGemmArgs a;
        // Gsw = K_t W^T  [N][Ds]
        memset(&a, 0, sizeof a);
        a.epi = PG_EPI_F32; a.out_f32 = g.Gsw; a.out_f32_stride = static_cast<long long>(N) * D; a.ld_f32 = D;
        a.reverse = (dir++) & 1;
        PCK(polar_gemm(false, Kt, Wc, nprob, a, st));
        // Psi = s_w W  [N][N]  -> Theta' = 2 (diag(a) - q Psi q - a a^T), stored as a split pair
        memset(&a, 0, sizeof a);
        a.epi = PG_EPI_THETA; a.out_hi = g.theta; a.out_lo = g.theta_lo;
        a.out_stride = static_cast<long long>(N) * g.NsPad; a.ld_out = g.NsPad;
        a.vec_a = g.a;
        a.reverse = (dir++) & 1;
        PCK(polar_gemm(true, g.SW, Wc, nprob, a, st));
    }
    {
        TimingScope ts(kSlotPolarFinish, st, 1);
        polar_finish_kernel<<<nprob, 256, (2 * N + 64) * sizeof(float), st>>>(g);
        PCK(cudaGetLastError());
    }
    return cudaSuccess;
}

cudaError_t launch_polar_procrustes_vt(const PolarArgs& g, cudaStream_t st) {
    const int N = g.Ns, M = g.Nt, D = g.Ds, nprob = g.n_problems;
    if (M > kVtMaxTokens || M > kVtThreads) return cudaErrorInvalidValue;
    {
        TimingScope ts(kSlotPolarPrep, st, 3);
        PCK(launch_prep_student_vec(g, st));
        const int ld = (M + 3) & ~3;
        const size_t smem_t = (static_cast<size_t>(ld) * M + 2 * N + 3 * M + 64) * sizeof(float);
        PCK(cudaFuncSetAttribute(vt_prep_teacher_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem_t)));
        vt_prep_teacher_kernel<<<nprob, kVtThreads, smem_t, st>>>(g);
        PCK(cudaGetLastError());
    }
    const int steps = g.steps >= kPolarStepsMin && g.steps <= kPolarStepsMax ? g.steps : kPolarSteps;
    PCK(cudaMemsetAsync(g.fro2, 0, sizeof(float) * nprob * g.fro_slots, st));
    PCK(cudaMemsetAsync(g.resid, 0, sizeof(float) * nprob * g.fro_slots, st));
    {
        TimingScope ts(kSlotPolarGemm, st, 3 * steps + 7);
        PolarGemmArgs a;
        // X_0 = (F G)^T s_w   [Nt][Ds]  (s_w enters as the MN-major operand), then the augmentation column
        memset(&a, 0, sizeof a);
        a.epi = PG_EPI_SPLIT; a.out_hi = g.X0.hi; a.out_lo = g.X0.lo; a.out_stride = g.X0.batch_stride; a.scale_c = 1.f;
        PCK(polar_gemm(true, g.FGt, g.SW, nprob, a, st));
        vt_augment_kernel<<<nprob, 256, 0, st>>>(g);
        PCK(cudaGetLastError());
        SplitMat Xc = g.X0, Xn = g.X1;
        int dir = 0;
        for (int k = 0; k < steps; ++k) {
            const float* coef = polar_coef(k, steps);
            const float ca = coef[0], cb = coef[1], cc = coef[2];
            const bool first = k == 0, last = k == steps - 1;
            const float* norm = first ? g.fro2 : nullptr;
            // A = X X^T   (step 0: trace(A) = ||X_0^+||_F^2)
            memset(&a, 0, sizeof a);
            a.epi = PG_EPI_SPLIT; a.out_hi = g.A.hi; a.out_lo = g.A.lo; a.out_stride = g.A.batch_stride; a.scale_c = 1.f;
            a.a_alias_b = 1;
            if (first) { a.trace = g.fro2; a.fro_slots = g.fro_slots; }
            a.reverse = (dir++) & 1;
            PCK(polar_gemm(false, Xc, Xc, nprob, a, st));
            // Bm = a I + b (rA) + c (rA)^2
            memset(&a, 0, sizeof a);
            a.epi = PG_EPI_SPLIT; a.out_hi = g.Bm.hi; a.out_lo = g.Bm.lo; a.out_stride = g.Bm.batch_stride;
            a.a_alias_b = 1; a.aux_mode = 1; a.aux_hi = g.A.hi; a.aux_lo = g.A.lo;
            a.aux_c = cb; a.aux_p = first ? 1.f : 0.f; a.scale_c = cc; a.scale_p = first ? 2.f : 0.f; a.diag_add = ca; a.norm2 = norm; a.fro_slots = g.fro_slots;
            a.resid = last ? g.resid : nullptr;
            a.reverse = (dir++) & 1;
            PCK(polar_gemm(false, g.A, g.A, nprob, a, st));
            // X_next = sqrt(r) Bm X
            memset(&a, 0, sizeof a);
            a.epi = PG_EPI_SPLIT; a.out_hi = Xn.hi; a.out_lo = Xn.lo; a.out_stride = Xn.batch_stride;
            a.scale_c = 1.f; a.scale_p = first ? 0.5f : 0.f; a.norm2 = norm; a.fro_slots = g.fro_slots;
            a.reverse = (dir++) & 1;
            PCK(polar_gemm(true, g.Bm, Xc, nprob, a, st));
            Xc = Xn;
            Xn = (Xc.hi == g.X1.hi) ? g.X2 : g.X1;
        }
        const int d16 = (D + 15) & ~15;
        // Gsw = F G X_inf[:, :Ds] = d nuc / d s_w   [Ns][Ds]
        memset(&a, 0, sizeof a);
        a.epi = PG_EPI_F32; a.out_f32 = g.Gsw; a.out_f32_stride = static_cast<long long>(N) * D; a.ld_f32 = D; a.n_override = D;
        PCK(polar_gemm(true, g.FG, Xc, nprob, a, st));
        // H = X_0 X_inf^T over the student features (the augmentation column left out)
        memset(&a, 0, sizeof a);
        a.epi = PG_EPI_SPLIT; a.out_hi = g.Hm.hi; a.out_lo = g.Hm.lo; a.out_stride = g.Hm.batch_stride; a.scale_c = 1.f; a.k_override = d16;
        PCK(polar_gemm(false, g.X0, Xc, nprob, a, st));
        // M2 = H G^-1 (I - 1 1^T / Nt),  Theta_raw = G^-T M2
        memset(&a, 0, sizeof a);
        a.epi = PG_EPI_SPLIT; a.out_hi = g.M2.hi; a.out_lo = g.M2.lo; a.out_stride = g.M2.batch_stride; a.scale_c = 1.f;
        PCK(polar_gemm(true, g.Hm, g.GinvC, nprob, a, st));
        memset(&a, 0, sizeof a);
        a.epi = PG_EPI_F32; a.out_f32 = g.thraw; a.out_f32_stride = static_cast<long long>(M) * M; a.ld_f32 = M;
        PCK(polar_gemm(true, g.GinvT, g.M2, nprob, a, st));
        vt_theta_kernel<<<dim3((M * M + 255) / 256 < 8 ? (M * M + 255) / 256 : 8, nprob), 256, 0, st>>>(g);
        PCK(cudaGetLastError());
    }
    {
        TimingScope ts(kSlotPolarFinish, st, 1);
        polar_finish_kernel<<<nprob, 256, (2 * N + 64) * sizeof(float), st>>>(g);
        PCK(cudaGetLastError());
    }
    return cudaSuccess;
}

}  // namespace basd
