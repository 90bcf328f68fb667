// Bandwidth-bound kernels of the BASD loss path: coalesced, 128-bit vectorised, fp32 accumulation.
//   importance_rows   teacher attention -> per-layer token importance       (relational.py:22-27, before mixing)
//   importance_mix    mix + resample + normalise importance                 (layer_selector.py:112, relational.py:29-34)
//   mix_teacher       mix + token-grid resample of teacher tokens (hi/lo)   (layer_selector.py:111, combined.py:9-14)
//   wgrad_dots        d loss / d mixing weights                             (SURVEY.md B.2)
//   colsum, split_bf16, pack_bf16, loss_reduce  small helpers
#include "cta_linalg.cuh"
#include "spectral.h"

namespace basd {

__device__ __forceinline__ uint4 ld_nc_16(const void* p) {
    uint4 r;
    asm("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ void bf16x8_to_float(const uint4& v, float* f) {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 t = __bfloat1622float2(h[i]);
        f[2 * i] = t.x;
        f[2 * i + 1] = t.y;
    }
}
// f[i] += the eight bf16 of v (the lo half of a split-bf16 pair onto its hi half)
__device__ __forceinline__ void add_bf16x8(const uint4& v, float* f) {
    float l[8];
    bf16x8_to_float(v, l);
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] += l[i];
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
}

// ---------------------------------------------------------------------------------------------- importance rows
template <typename T>
__device__ __forceinline__ float ld_as_float(const T* p);
template <>
__device__ __forceinline__ float ld_as_float<float>(const float* p) { return __ldg(p); }
template <>
__device__ __forceinline__ float ld_as_float<__nv_bfloat16>(const __nv_bfloat16* p) { return __bfloat162float(*p); }

template <typename T>
__global__ void importance_rows_kernel(PtrTable attn, int B, int H, int Nt, int has_cls, long long sb, long long sh,
                                       long long sq, long long sk, float* __restrict__ rows) {
    const int b = blockIdx.x, j = blockIdx.y;
    const T* A = reinterpret_cast<const T*>(attn.p[j]) + static_cast<long long>(b) * sb;
    float* out = rows + (static_cast<size_t>(j) * B + b) * Nt;
    if (has_cls == 2) {                                 // BASD_ATTN_QUERY_MEAN: [B,H,1,Nt] rows already averaged over the queries
        for (int n = threadIdx.x; n < Nt; n += blockDim.x) {
            float s = 0.f;
            for (int h = 0; h < H; ++h) s += ld_as_float(A + h * sh + n * sk);
            out[n] = s / static_cast<float>(H);
        }
    } else if (has_cls) {
        for (int n = threadIdx.x; n < Nt; n += blockDim.x) {
            float s = 0.f;
            for (int h = 0; h < H; ++h) s += ld_as_float(A + h * sh + (1 + n) * sk);     // query 0 (CLS), keys 1..Nt
            out[n] = s / static_cast<float>(H);
        }
    } else {
        for (int n = threadIdx.x; n < Nt; n += blockDim.x) {
            float s = 0.f;
            for (int h = 0; h < H; ++h)
                for (int q = 0; q < Nt; ++q) s += ld_as_float(A + h * sh + q * sq + n * sk);
            out[n] = s / static_cast<float>(H * Nt);
        }
    }
}

cudaError_t launch_importance_rows(const PtrTable& attn, int attn_is_bf16, int Lt, int B, int H, int Nt, int has_cls,
                                   const long long* s, float* rows, cudaStream_t st) {
    if (attn_is_bf16)
        importance_rows_kernel<__nv_bfloat16><<<dim3(B, Lt), 256, 0, st>>>(attn, B, H, Nt, has_cls, s[0], s[1], s[2], s[3], rows);
    else
        importance_rows_kernel<float><<<dim3(B, Lt), 256, 0, st>>>(attn, B, H, Nt, has_cls, s[0], s[1], s[2], s[3], rows);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------- CLS attention rows
// SURVEY.md section 8(f) rank 1: the reference's teacher hook (src/models/teacher.py:27-39) recomputes the full
// softmax(Q K^T / sqrt(d)) [B,H,N+1,N+1] per block only for the loss to read its CLS query row (relational.py:24).
// This kernel emits that row directly from Q and K: out[b,h,0,:] = softmax_s(q[b,h,0,:] . k[b,h,s,:] * scale).
// One warp per (b, h); a lane owns keys s = lane, lane + 32, ...; fp32 accumulation; d stride must be 1.
template <typename T>
__global__ void __launch_bounds__(128)
cls_attention_rows_kernel(const T* __restrict__ q, const T* __restrict__ k, int B, int H, int S, int dh, long long qb, long long qh,
                          long long kb, long long kh, long long ks, float scale, float* __restrict__ out) {
    extern __shared__ float qs[];                       // [warps][dh]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int bh = blockIdx.x * (blockDim.x >> 5) + warp;
    if (bh >= B * H) return;
    const int b = bh / H, h = bh % H;
    float* q0 = qs + warp * dh;
    const T* qp = q + b * qb + h * qh;                  // query 0 = CLS
    for (int d = lane; d < dh; d += 32) q0[d] = static_cast<float>(qp[d]) * scale;
    __syncwarp();
    const T* kp = k + b * kb + h * kh;
    float* o = out + static_cast<size_t>(bh) * S;
    float mx = -3.0e38f;
    for (int s0 = lane; s0 < S; s0 += 32) {
        const T* kr = kp + s0 * ks;
        float acc = 0.f;
        for (int d = 0; d < dh; ++d) acc = fmaf(q0[d], static_cast<float>(kr[d]), acc);
        o[s0] = acc;                                    // scores parked in the output row
        mx = fmaxf(mx, acc);
    }
    for (int of = 16; of > 0; of >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, of));
    float sum = 0.f;
    for (int s0 = lane; s0 < S; s0 += 32) { const float e = __expf(o[s0] - mx); o[s0] = e; sum += e; }
    sum = warp_sum(sum);
    const float inv = 1.f / sum;
    for (int s0 = lane; s0 < S; s0 += 32) o[s0] *= inv;
}
cudaError_t launch_cls_attention_rows(const void* q, const void* k, int is_bf16, int B, int H, int S, int dh, const long long* qst,
                                      const long long* kst, float scale, float* out, cudaStream_t st) {
    const int warps = 4, blocks = (B * H + warps - 1) / warps;
    const size_t smem = sizeof(float) * warps * dh;
    if (is_bf16)
        cls_attention_rows_kernel<__nv_bfloat16><<<blocks, warps * 32, smem, st>>>(reinterpret_cast<const __nv_bfloat16*>(q), reinterpret_cast<const __nv_bfloat16*>(k),
                                                                                  B, H, S, dh, qst[0], qst[1], kst[0], kst[1], kst[2], scale, out);
    else
        cls_attention_rows_kernel<float><<<blocks, warps * 32, smem, st>>>(reinterpret_cast<const float*>(q), reinterpret_cast<const float*>(k), B, H, S, dh,
                                                                           qst[0], qst[1], kst[0], kst[1], kst[2], scale, out);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------- small helpers
__global__ void split_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo, size_t n) {
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const float v = src[i];
        const __nv_bfloat16 h = __float2bfloat16(v);
        hi[i] = h;
        lo[i] = __float2bfloat16(v - __bfloat162float(h));
    }
}
cudaError_t launch_split_bf16(const float* src, __nv_bfloat16* hi, __nv_bfloat16* lo, size_t n, cudaStream_t st) {
    const int blocks = static_cast<int>((n + 255) / 256 < 1184 ? (n + 255) / 256 : 1184);
    split_bf16_kernel<<<blocks, 256, 0, st>>>(src, hi, lo, n);
    return cudaGetLastError();
}

template <typename T>
__global__ void pack_bf16_kernel(const T* __restrict__ src, long long sb, long long sn, long long sd, int B, int N, int D,
                                 __nv_bfloat16* __restrict__ dst, __nv_bfloat16* __restrict__ dst_lo) {
    const size_t total = static_cast<size_t>(B) * N * D;
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int d = static_cast<int>(i % D);
        const size_t r = i / D;
        const int n = static_cast<int>(r % N), b = static_cast<int>(r / N);
        const float v = static_cast<float>(src[b * sb + n * sn + d * sd]);
        const __nv_bfloat16 h = __float2bfloat16(v);
        dst[i] = h;
        if (dst_lo) dst_lo[i] = __float2bfloat16(v - __bfloat162float(h));
    }
}
cudaError_t launch_pack_bf16(const void* src, int src_is_bf16, long long sb, long long sn, long long sd, int B, int N, int D,
                             __nv_bfloat16* dst, __nv_bfloat16* dst_lo, cudaStream_t st) {
    const size_t total = static_cast<size_t>(B) * N * D;
    const int blocks = static_cast<int>((total + 255) / 256 < 2368 ? (total + 255) / 256 : 2368);
    if (src_is_bf16)
        pack_bf16_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(src), sb, sn, sd, B, N, D, dst, dst_lo);
    else
        pack_bf16_kernel<float><<<blocks, 256, 0, st>>>(reinterpret_cast<const float*>(src), sb, sn, sd, B, N, D, dst, dst_lo);
    return cudaGetLastError();
}

// out[j][d] = sum over rows of (hi[j] + lo[j])[row][d]; D % 8 == 0.  grid = (row chunks, jobs): every CTA streams a
// contiguous chunk of rows with 16-byte loads (4 in flight per thread), reduces across its row lanes in shared
// memory and writes its D partial sums to part[job][chunk][D]; colsum_reduce_kernel adds the chunks in a fixed order
// (atomicAdd made the column sums, hence the centred Grams, differ from launch to launch).
constexpr int kColsumThreads = 256;
__global__ void __launch_bounds__(kColsumThreads)
colsum_kernel(ColsumJobs jobs, size_t rows, int D, float* __restrict__ part, int rpb, long long bstride) {
    __shared__ float red[kColsumThreads * 8];
    const int j = blockIdx.y;
    const __nv_bfloat16* Xh = jobs.hi[j];
    const __nv_bfloat16* Xl = jobs.lo[j];
    const int vpr = D / 8;                                   // 16-byte vectors per row
    const int rpp = kColsumThreads / vpr;                    // rows per pass
    const int lr = threadIdx.x / vpr, cv = threadIdx.x % vpr;
    const size_t chunk = (rows + gridDim.x - 1) / gridDim.x;
    const size_t r0 = blockIdx.x * chunk, r1 = r0 + chunk < rows ? r0 + chunk : rows;
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    // rpb > 0: row r is token r % rpb of sample r / rpb of a [B][rpb][D] tensor with batch stride bstride elements
    auto row_off = [&](size_t r) -> size_t { return rpb > 0 ? (r / rpb) * static_cast<size_t>(bstride) + (r % rpb) * static_cast<size_t>(D) : r * D; };
    if (lr < rpp) {
        size_t r = r0 + lr;
        for (; r + 3 * static_cast<size_t>(rpp) < r1; r += 4 * static_cast<size_t>(rpp)) {
            uint4 v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) v[u] = ld_nc_16(Xh + row_off(r + static_cast<size_t>(u) * rpp) + cv * 8);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                float f[8];
                bf16x8_to_float(v[u], f);
#pragma unroll
                for (int i = 0; i < 8; ++i) acc[i] += f[i];
            }
            if (Xl) {
#pragma unroll
                for (int u = 0; u < 4; ++u) v[u] = ld_nc_16(Xl + row_off(r + static_cast<size_t>(u) * rpp) + cv * 8);
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    float f[8];
                    bf16x8_to_float(v[u], f);
#pragma unroll
                    for (int i = 0; i < 8; ++i) acc[i] += f[i];
                }
            }
        }
        for (; r < r1; r += rpp) {
            float f[8];
            bf16x8_to_float(ld_nc_16(Xh + row_off(r) + cv * 8), f);
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i] += f[i];
            if (Xl) {
                bf16x8_to_float(ld_nc_16(Xl + row_off(r) + cv * 8), f);
#pragma unroll
                for (int i = 0; i < 8; ++i) acc[i] += f[i];
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) red[threadIdx.x * 8 + i] = acc[i];
    __syncthreads();
    for (int c = threadIdx.x; c < D; c += blockDim.x) {
        const int v = c / 8, e = c % 8;
        float s = 0.f;
        for (int l = 0; l < rpp; ++l) s += red[(l * vpr + v) * 8 + e];
        part[(static_cast<size_t>(j) * gridDim.x + blockIdx.x) * D + c] = s;
    }
}
__global__ void colsum_reduce_kernel(ColsumJobs jobs, const float* __restrict__ part, int chunks, int D) {
    const int j = blockIdx.x;
    for (int c = threadIdx.x; c < D; c += blockDim.x) {
        float s = 0.f;
        for (int k = 0; k < chunks; ++k) s += part[(static_cast<size_t>(j) * chunks + k) * D + c];
        jobs.out[j][c] = s;
    }
}
static int colsum_chunks(int n_jobs, size_t rows) {
    int chunks = (148 * 8 + n_jobs - 1) / n_jobs;
    if (static_cast<size_t>(chunks) * 64 > rows) chunks = static_cast<int>((rows + 63) / 64);
    return chunks;
}
size_t colsum_part_floats(int n_jobs, size_t rows, int D) { return static_cast<size_t>(n_jobs) * colsum_chunks(n_jobs, rows) * D; }
cudaError_t launch_colsum(const ColsumJobs& jobs, int n_jobs, size_t rows, int D, float* part, cudaStream_t st, int rows_per_batch,
                          long long batch_stride) {
    if (D % 8 != 0 || D > 8 * kColsumThreads || n_jobs < 1 || !part) return cudaErrorInvalidValue;
    const int chunks = colsum_chunks(n_jobs, rows);
    colsum_kernel<<<dim3(chunks, n_jobs), kColsumThreads, 0, st>>>(jobs, rows, D, part, rows_per_batch, batch_stride);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    colsum_reduce_kernel<<<n_jobs, 256, 0, st>>>(jobs, part, chunks, D);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------- importance mix
// a[i][b][n] = normalise_n( interp( sum_j w[i][j] rows[j][b][:] )[n] );  ssum[i][b] = sum before normalising
__global__ void importance_mix_kernel(const float* __restrict__ rows, const float* __restrict__ w, int Lt, int P, int B, int Nt,
                                      int Ns, float* __restrict__ a, float* __restrict__ ssum) {
    __shared__ float red[40];
    const int i = blockIdx.x / B, b = blockIdx.x % B;
    float part = 0.f;
    float* out = a + static_cast<size_t>(blockIdx.x) * Ns;
    for (int n = threadIdx.x; n < Ns; n += blockDim.x) {
        int i0, i1; float lam;
        interp_index(n, Nt, Ns, i0, i1, lam);
        float v = 0.f;
        for (int j = 0; j < Lt; ++j) {
            const float* r = rows + (static_cast<size_t>(j) * B + b) * Nt;
            v = fmaf(w[i * Lt + j], (1.f - lam) * r[i0] + lam * r[i1], v);
        }
        out[n] = v;
        part += v;
    }
    const float tot = cta_sum(part, red);
    for (int n = threadIdx.x; n < Ns; n += blockDim.x) out[n] = out[n] / tot;
    if (threadIdx.x == 0) ssum[blockIdx.x] = tot;
}
cudaError_t launch_importance_mix(const float* rows, const float* w, int Lt, int P, int B, int Nt, int Ns, float* a, float* ssum,
                                  cudaStream_t st) {
    importance_mix_kernel<<<P * B, 256, 0, st>>>(rows, w, Lt, P, B, Nt, Ns, a, ssum);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------- mix teacher
// Tbar[i][b][n][:] = sum_j w[i][j] * interp(T_j[b])[n][:]  -> bf16 hi + lo.  One thread = one 8-wide vector.
// Teacher vectors are loaded twelve layers at a time before the first use (one load and its use alternating per layer left
// one request in flight per thread: 4.0 TB/s; six at a time 4.6, twelve 5.1), 32-bit index arithmetic, no interpolation
// branch when N_t == N_s.  TSPLIT: split-bf16 teacher tokens (teacher_lo holds the lo halves, same layout), read as hi + lo;
// six layers at a time so that the doubled loads stay in registers.
constexpr int MT_JC = 12;
template <int PMAX, bool INTERP, bool TSPLIT = false>
__global__ void __launch_bounds__(256)
mix_teacher_kernel(PtrTable teacher, const float* __restrict__ w, int Lt, int P, int B, int Nt, int Ns, int Dt, long long tbs,
                   __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo, PtrTable teacher_lo) {
    constexpr int JC = TSPLIT ? MT_JC / 2 : MT_JC;
    __shared__ float ws[PMAX * kMaxLayers];
    for (int t = threadIdx.x; t < P * Lt; t += blockDim.x) ws[t] = w[t];
    __syncthreads();
    const uint32_t vpr = static_cast<uint32_t>(Dt) / 8u;
    const uint32_t total = static_cast<uint32_t>(B) * Ns * vpr;            // < 2^32 (checked by the launcher)
    const uint4 zero4 = make_uint4(0u, 0u, 0u, 0u);
    for (uint32_t v = blockIdx.x * blockDim.x + threadIdx.x; v < total; v += gridDim.x * blockDim.x) {
        const uint32_t row = v / vpr, dv = v - row * vpr;
        const uint32_t b = row / static_cast<uint32_t>(Ns), n = row - b * Ns;
        int i0, i1; float lam;
        interp_index(static_cast<int>(n), Nt, Ns, i0, i1, lam);
        float acc[PMAX][8];
#pragma unroll
        for (int i = 0; i < PMAX; ++i)
#pragma unroll
            for (int e = 0; e < 8; ++e) acc[i][e] = 0.f;
        for (int j0 = 0; j0 < Lt; j0 += JC) {
            uint4 t0[JC], t1[INTERP ? JC : 1], u0[TSPLIT ? JC : 1], u1[TSPLIT && INTERP ? JC : 1];
#pragma unroll
            for (int jj = 0; jj < JC; ++jj) {
                const bool ok = j0 + jj < Lt;
                const size_t boff = static_cast<size_t>(b) * tbs + dv * 8;
                const __nv_bfloat16* T = reinterpret_cast<const __nv_bfloat16*>(teacher.p[ok ? j0 + jj : 0]) + boff;
                t0[jj] = ok ? ld_nc_16(T + static_cast<size_t>(i0) * Dt) : zero4;
                if (INTERP) t1[jj] = ok ? ld_nc_16(T + static_cast<size_t>(i1) * Dt) : zero4;
                if (TSPLIT) {
                    const __nv_bfloat16* U = reinterpret_cast<const __nv_bfloat16*>(teacher_lo.p[ok ? j0 + jj : 0]) + boff;
                    u0[jj] = ok ? ld_nc_16(U + static_cast<size_t>(i0) * Dt) : zero4;
                    if (INTERP) u1[jj] = ok ? ld_nc_16(U + static_cast<size_t>(i1) * Dt) : zero4;
                }
            }
#pragma unroll
            for (int jj = 0; jj < JC; ++jj) {
                if (j0 + jj < Lt) {
                    float f[8];
                    bf16x8_to_float(t0[jj], f);
                    if (TSPLIT) add_bf16x8(u0[jj], f);
                    if (INTERP) {
                        float g[8];
                        bf16x8_to_float(t1[jj], g);
                        if (TSPLIT) add_bf16x8(u1[jj], g);
#pragma unroll
                        for (int e = 0; e < 8; ++e) f[e] = (1.f - lam) * f[e] + lam * g[e];
                    }
#pragma unroll
                    for (int i = 0; i < PMAX; ++i) {
                        if (i < P) {
                            const float wi = ws[i * Lt + j0 + jj];
#pragma unroll
                            for (int e = 0; e < 8; ++e) acc[i][e] = fmaf(wi, f[e], acc[i][e]);
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int i = 0; i < PMAX; ++i) {
            if (i < P) {
                const size_t off = ((static_cast<size_t>(i) * B + b) * Ns + n) * Dt + dv * 8;
                float l[8];
                uint4 h4, l4;
                uint32_t* hp = reinterpret_cast<uint32_t*>(&h4);
                uint32_t* lp = reinterpret_cast<uint32_t*>(&l4);
#pragma unroll
                for (int e = 0; e < 8; e += 2) {
                    const __nv_bfloat16 h0 = __float2bfloat16(acc[i][e]), h1 = __float2bfloat16(acc[i][e + 1]);
                    l[e] = acc[i][e] - __bfloat162float(h0);
                    l[e + 1] = acc[i][e + 1] - __bfloat162float(h1);
                    __nv_bfloat162 hv; hv.x = h0; hv.y = h1;
                    hp[e / 2] = *reinterpret_cast<uint32_t*>(&hv);
                    lp[e / 2] = pack2(l[e], l[e + 1]);
                }
                *reinterpret_cast<uint4*>(hi + off) = h4;
                *reinterpret_cast<uint4*>(lo + off) = l4;
            }
        }
    }
}
cudaError_t launch_mix_teacher(const PtrTable& teacher, const float* w, int Lt, int P, int B, int Nt, int Ns, int Dt,
                               __nv_bfloat16* hi, __nv_bfloat16* lo, cudaStream_t st, long long tbs, const PtrTable* teacher_lo) {
    if (tbs <= 0) tbs = static_cast<long long>(Nt) * Dt;
    if (Dt % 8 != 0 || P > kMaxPoints) return cudaErrorInvalidValue;
    const size_t total = static_cast<size_t>(B) * Ns * (Dt / 8);
    const int blocks = static_cast<int>((total + 255) / 256 < 148 * 8 ? (total + 255) / 256 : 148 * 8);
    if (static_cast<unsigned long long>(B) * Ns * (Dt / 8) >= (1ull << 32)) return cudaErrorInvalidValue;
    const bool interp = Nt != Ns;
    const PtrTable tl = teacher_lo ? *teacher_lo : PtrTable{};
#define MIX_LAUNCH(PM, IN, SP) mix_teacher_kernel<PM, IN, SP><<<blocks, 256, 0, st>>>(teacher, w, Lt, P, B, Nt, Ns, Dt, tbs, hi, lo, tl)
    if (teacher_lo) {
        if (P <= 4) { if (interp) MIX_LAUNCH(4, true, true); else MIX_LAUNCH(4, false, true); }
        else { if (interp) MIX_LAUNCH(8, true, true); else MIX_LAUNCH(8, false, true); }
    } else {
        if (P <= 4) { if (interp) MIX_LAUNCH(4, true, false); else MIX_LAUNCH(4, false, false); }
        else { if (interp) MIX_LAUNCH(8, true, false); else MIX_LAUNCH(8, false, false); }
    }
#undef MIX_LAUNCH
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------- d loss / d w
// gw[i][j] += sum_{b,n,d} Dtm[i][b][n][d] * interp(T_j[b])[n][d]      blockIdx.y selects a (point-chunk, layer-chunk)
constexpr int WG_PC = 4, WG_JC = 12;
// All 16-byte loads of a position (WG_PC gradient vectors, WG_JC teacher vectors, twice that when interpolating) are issued
// before the first use: with a load and its use alternating per layer the kernel ran at 2 TB/s, one L2/HBM latency per layer.
// Every CTA writes its WG_PC x WG_JC partial dots to gw_part[blockIdx.x][P][Lt]; wgrad_reduce_kernel adds the CTAs (and the
// importance partials) in a fixed order.  TSPLIT: split-bf16 teacher tokens read as hi + lo, six layers per CTA.
template <bool TSPLIT> __host__ __device__ constexpr int wgrad_jc() { return TSPLIT ? WG_JC / 2 : WG_JC; }
template <bool INTERP, bool SPLIT, bool TSPLIT = false>
__global__ void __launch_bounds__(256)
wgrad_dots_kernel(PtrTable teacher, const __nv_bfloat16* __restrict__ Dtm, const __nv_bfloat16* __restrict__ DtmLo, int Lt, int P, int B, int Nt,
                  int Ns, int Dt, long long tbs, float* __restrict__ gw_part, PtrTable teacher_lo) {
    constexpr int JC = wgrad_jc<TSPLIT>();
    const int n_jc = (Lt + JC - 1) / JC;
    const int i_base = (blockIdx.y / n_jc) * WG_PC, j_base = (blockIdx.y % n_jc) * JC;
    float acc[WG_PC][JC];
#pragma unroll
    for (int i = 0; i < WG_PC; ++i)
#pragma unroll
        for (int j = 0; j < JC; ++j) acc[i][j] = 0.f;
    const uint32_t vpr = static_cast<uint32_t>(Dt) / 8u;
    const uint32_t total = static_cast<uint32_t>(B) * Ns * vpr;            // < 2^32 (checked by the launcher)
    const uint4 zero4 = make_uint4(0u, 0u, 0u, 0u);
    for (uint32_t v = blockIdx.x * blockDim.x + threadIdx.x; v < total; v += gridDim.x * blockDim.x) {
        const uint32_t row = v / vpr, dv = v - row * vpr;
        const uint32_t b = row / static_cast<uint32_t>(Ns), n = row - b * Ns;
        int i0, i1; float lam;
        interp_index(static_cast<int>(n), Nt, Ns, i0, i1, lam);
        uint4 draw[WG_PC], dlow[SPLIT ? WG_PC : 1], t0[JC], t1[INTERP ? JC : 1], u0[TSPLIT ? JC : 1], u1[TSPLIT && INTERP ? JC : 1];
#pragma unroll
        for (int i = 0; i < WG_PC; ++i) {
            const size_t off = ((static_cast<size_t>(i_base + i < P ? i_base + i : 0) * B + b) * Ns + n) * Dt + dv * 8;
            draw[i] = i_base + i < P ? ld_nc_16(Dtm + off) : zero4;
            if (SPLIT) dlow[i] = i_base + i < P ? ld_nc_16(DtmLo + off) : zero4;
        }
#pragma unroll
        for (int j = 0; j < JC; ++j) {
            const bool ok = j_base + j < Lt;
            const size_t boff = static_cast<size_t>(b) * tbs + dv * 8;
            const __nv_bfloat16* T = reinterpret_cast<const __nv_bfloat16*>(teacher.p[ok ? j_base + j : 0]) + boff;
            t0[j] = ok ? ld_nc_16(T + static_cast<size_t>(i0) * Dt) : zero4;
            if (INTERP) t1[j] = ok ? ld_nc_16(T + static_cast<size_t>(i1) * Dt) : zero4;
            if (TSPLIT) {
                const __nv_bfloat16* U = reinterpret_cast<const __nv_bfloat16*>(teacher_lo.p[ok ? j_base + j : 0]) + boff;
                u0[j] = ok ? ld_nc_16(U + static_cast<size_t>(i0) * Dt) : zero4;
                if (INTERP) u1[j] = ok ? ld_nc_16(U + static_cast<size_t>(i1) * Dt) : zero4;
            }
        }
        float dtv[WG_PC][8];
#pragma unroll
        for (int i = 0; i < WG_PC; ++i) {
            bf16x8_to_float(draw[i], dtv[i]);
            if (SPLIT) {
                float lo8[8];
                bf16x8_to_float(dlow[i], lo8);
#pragma unroll
                for (int e = 0; e < 8; ++e) dtv[i][e] += lo8[e];
            }
        }
#pragma unroll
        for (int j = 0; j < JC; ++j) {
            float f[8];
            bf16x8_to_float(t0[j], f);
            if (TSPLIT) add_bf16x8(u0[j], f);
            if (INTERP) {
                float g[8];
                bf16x8_to_float(t1[j], g);
                if (TSPLIT) add_bf16x8(u1[j], g);
#pragma unroll
                for (int e = 0; e < 8; ++e) f[e] = (1.f - lam) * f[e] + lam * g[e];
            }
#pragma unroll
            for (int i = 0; i < WG_PC; ++i) {
                float s = 0.f;
#pragma unroll
                for (int e = 0; e < 8; ++e) s = fmaf(dtv[i][e], f[e], s);
                acc[i][j] += s;
            }
        }
    }
    __shared__ float red[8][WG_PC * JC];                  // one row per warp (256 threads)
#pragma unroll
    for (int i = 0; i < WG_PC; ++i)
#pragma unroll
        for (int j = 0; j < JC; ++j) {
            const float s = warp_sum(acc[i][j]);
            if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][i * JC + j] = s;
        }
    __syncthreads();
    for (int t = threadIdx.x; t < WG_PC * JC; t += blockDim.x) {
        const int i = i_base + t / JC, j = j_base + t % JC;
        float s = 0.f;
#pragma unroll
        for (int wv = 0; wv < 8; ++wv) s += red[wv][t];
        if (i < P && j < Lt) gw_part[(static_cast<size_t>(blockIdx.x) * P + i) * Lt + j] = s;
    }
}
// gw_part[blockIdx.y][i][j] = sum_{b in this slice, n} gwt[i][b][n] * interp(rows[j][b])[n]
__global__ void wgrad_importance_kernel(const float* __restrict__ gwt, const float* __restrict__ rows, int Lt, int P, int B, int Nt,
                                        int Ns, float* __restrict__ gw_part) {
    __shared__ float red[40];
    const int i = blockIdx.x / Lt, j = blockIdx.x % Lt;
    float part = 0.f;
    // blockIdx.y strides over the samples (48 CTAs walking 50k elements each was 0.1 ms of pure latency)
    for (int b = blockIdx.y; b < B; b += gridDim.y) {
        const float* r = rows + (static_cast<size_t>(j) * B + b) * Nt;
        const float* gq = gwt + (static_cast<size_t>(i) * B + b) * Ns;
        for (int n = threadIdx.x; n < Ns; n += blockDim.x) {
            int i0, i1; float lam;
            interp_index(n, Nt, Ns, i0, i1, lam);
            part = fmaf(gq[n], (1.f - lam) * r[i0] + lam * r[i1], part);
        }
    }
    const float tot = cta_sum(part, red);
    if (threadIdx.x == 0) gw_part[(static_cast<size_t>(blockIdx.y) * P + i) * Lt + j] = tot;
}
// gw[i][j] = sum of the n_part partial tables in a FIXED order: one warp per entry, lane l sums partials l, l + 32, ...
// ascending, then the 32 lane sums are combined by the xor-shuffle tree (the same association on every launch).
// (One thread per entry walking all ~600 partials was 54 us of dependent L2 latency at cfg2.)
__global__ void __launch_bounds__(256)
wgrad_reduce_kernel(const float* __restrict__ gw_part, int n_part, int PL, float* __restrict__ gw) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= PL) return;
    float s = 0.f;
    for (int k = lane; k < n_part; k += 32) s += gw_part[static_cast<size_t>(k) * PL + warp];
    s = warp_sum(s);
    if (lane == 0) gw[warp] = s;
}
constexpr int kWgradDotCtas = 148 * 4, kWgradImpSlices = 16;
size_t wgrad_part_floats(int P, int Lt) { return static_cast<size_t>(kWgradDotCtas + kWgradImpSlices) * P * Lt; }
cudaError_t launch_wgrad_dots(const PtrTable& teacher, const __nv_bfloat16* Dtm, const __nv_bfloat16* DtmLo, const float* gwt, const float* rows, int Lt, int P,
                              int B, int Nt, int Ns, int Dt, float* gw, float* gw_part, cudaStream_t st, bool dtm_unaligned, long long tbs,
                              const PtrTable* teacher_lo) {
    if (tbs <= 0) tbs = static_cast<long long>(Nt) * Dt;
    if (Dt % 8 != 0 || static_cast<unsigned long long>(B) * Ns * (Dt / 8) >= (1ull << 32) || !gw_part) return cudaErrorInvalidValue;
    const int jc = teacher_lo ? wgrad_jc<true>() : wgrad_jc<false>();
    const int ny = ((P + WG_PC - 1) / WG_PC) * ((Lt + jc - 1) / jc);
    const dim3 grid(kWgradDotCtas, ny);
    const PtrTable tl = teacher_lo ? *teacher_lo : PtrTable{};
    const bool aligned = Nt == Ns || dtm_unaligned;
    const int ns = aligned ? Nt : Ns;
#define WG_LAUNCH(IN, SP, TS) wgrad_dots_kernel<IN, SP, TS><<<grid, 256, 0, st>>>(teacher, Dtm, DtmLo, Lt, P, B, Nt, ns, Dt, tbs, gw_part, tl)
    if (teacher_lo) {
        if (aligned) { if (DtmLo) WG_LAUNCH(false, true, true); else WG_LAUNCH(false, false, true); }
        else { if (DtmLo) WG_LAUNCH(true, true, true); else WG_LAUNCH(true, false, true); }
    } else {
        if (aligned) { if (DtmLo) WG_LAUNCH(false, true, false); else WG_LAUNCH(false, false, false); }
        else { if (DtmLo) WG_LAUNCH(true, true, false); else WG_LAUNCH(true, false, false); }
    }
#undef WG_LAUNCH
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const int slices = B < kWgradImpSlices ? B : kWgradImpSlices;
    wgrad_importance_kernel<<<dim3(P * Lt, slices), 256, 0, st>>>(gwt, rows, Lt, P, B, Nt, Ns, gw_part + static_cast<size_t>(kWgradDotCtas) * P * Lt);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    wgrad_reduce_kernel<<<(P * Lt * 32 + 255) / 256, 256, 0, st>>>(gw_part, kWgradDotCtas + slices, P * Lt, gw);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------- loss reduce
__global__ void loss_reduce_kernel(const float* __restrict__ loss_b, const float* __restrict__ dbg, int P, int B, float* __restrict__ geo_i,
                                   float* __restrict__ geo, float* __restrict__ resid_max) {
    __shared__ float red[40];
    __shared__ float mx[8];
    if (resid_max) {                        // largest polar residual over all (point, sample) problems; NaN counts as +inf
        float m = 0.f;
        for (int t = threadIdx.x; t < P * B; t += blockDim.x) {
            const float r = dbg[t * 5 + 3];
            m = fmaxf(m, (r == r) ? r : __int_as_float(0x7f800000));
        }
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if ((threadIdx.x & 31) == 0) mx[threadIdx.x >> 5] = m;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int wv = 1; wv < (blockDim.x >> 5); ++wv) m = fmaxf(m, mx[wv]);
            *resid_max = m;
        }
    }
    float total = 0.f;
    for (int i = 0; i < P; ++i) {
        float part = 0.f;
        for (int b = threadIdx.x; b < B; b += blockDim.x) part += loss_b[i * B + b];
        const float s = cta_sum(part, red) / static_cast<float>(B);
        if (threadIdx.x == 0) geo_i[i] = s;
        total += s;
    }
    if (threadIdx.x == 0) *geo = total / static_cast<float>(P);
}
cudaError_t launch_loss_reduce(const float* loss_b, const float* dbg, int P, int B, float* geo_i, float* geo, float* resid_max, cudaStream_t st) {
    loss_reduce_kernel<<<1, 256, 0, st>>>(loss_b, dbg, P, B, geo_i, geo, resid_max);
    return cudaGetLastError();
}


// ---------------------------------------------------------------------------------------------- align_token_count (standalone)
// combined.py:9-14 on its own: out[b][n][:] = (1 - lam) in[b][i0][:] + lam in[b][i1][:] along the flattened token axis
// (interp_index: 1-D linear, align_corners = False, no anti-aliasing).  Inside the loss this resampling is fused into
// mix_teacher; these two kernels exist so that the reference's free function has a drop-in with the same gradient.
// One thread per (b, n, 8-feature octet) when D % 8 == 0 and the rows are 16-byte aligned, else per element.
template <typename T>
__global__ void __launch_bounds__(256)
align_tokens_kernel(const T* __restrict__ src, long long sb, long long sn, long long sd, int B, int Nin, int Nout, int D,
                    T* __restrict__ dst) {
    const long long total = static_cast<long long>(B) * Nout * D;
    for (long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < total; t += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int d = static_cast<int>(t % D);
        const int n = static_cast<int>((t / D) % Nout);
        const long long b = t / (static_cast<long long>(D) * Nout);
        int i0, i1; float lam;
        interp_index(n, Nin, Nout, i0, i1, lam);
        const float x0 = static_cast<float>(src[b * sb + i0 * sn + d * sd]), x1 = static_cast<float>(src[b * sb + i1 * sn + d * sd]);
        dst[t] = static_cast<T>((1.f - lam) * x0 + lam * x1);
    }
}
// adjoint: gin[b][m][:] = sum over the output tokens n that read input token m of their tap weight times gout[b][n][:]
// (gather form: every input token walks the output tokens in order - no atomics, bitwise repeatable)
template <typename T>
__global__ void __launch_bounds__(256)
align_tokens_bwd_kernel(const T* __restrict__ gout, int B, int Nin, int Nout, int D, T* __restrict__ gin) {
    const long long total = static_cast<long long>(B) * Nin * D;
    // output tokens whose taps can touch input token m lie in a window around m * Nout / Nin
    const float ratio = static_cast<float>(Nout) / static_cast<float>(Nin);
    for (long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < total; t += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int d = static_cast<int>(t % D);
        const int m = static_cast<int>((t / D) % Nin);
        const long long b = t / (static_cast<long long>(D) * Nin);
        int n_lo = static_cast<int>((m - 1) * ratio) - 2, n_hi = static_cast<int>((m + 2) * ratio) + 2;
        if (n_lo < 0) n_lo = 0;
        if (n_hi > Nout - 1) n_hi = Nout - 1;
        float acc = 0.f;
        for (int n = n_lo; n <= n_hi; ++n) {
            int i0, i1; float lam;
            interp_index(n, Nin, Nout, i0, i1, lam);
            const float g = static_cast<float>(gout[(b * Nout + n) * D + d]);
            if (i0 == m) acc = fmaf(1.f - lam, g, acc);
            if (i1 == m) acc = fmaf(lam, g, acc);           // (i0 == i1 at the clamped end: both taps land on m, weights sum to 1)
        }
        gin[t] = static_cast<T>(acc);
    }
}
cudaError_t launch_align_tokens(const void* src, int is_bf16, long long sb, long long sn, long long sd, int B, int Nin, int Nout, int D,
                                void* dst, cudaStream_t st) {
    const long long total = static_cast<long long>(B) * Nout * D;
    const int grid = static_cast<int>(total / 256 + 1 < 148 * 16 ? total / 256 + 1 : 148 * 16);
    if (is_bf16) align_tokens_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(src), sb, sn, sd, B, Nin, Nout, D, reinterpret_cast<__nv_bfloat16*>(dst));
    else align_tokens_kernel<float><<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(src), sb, sn, sd, B, Nin, Nout, D, reinterpret_cast<float*>(dst));
    return cudaGetLastError();
}
cudaError_t launch_align_tokens_bwd(const void* gout, int is_bf16, int B, int Nin, int Nout, int D, void* gin, cudaStream_t st) {
    const long long total = static_cast<long long>(B) * Nin * D;
    const int grid = static_cast<int>(total / 256 + 1 < 148 * 16 ? total / 256 + 1 : 148 * 16);
    if (is_bf16) align_tokens_bwd_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(gout), B, Nin, Nout, D, reinterpret_cast<__nv_bfloat16*>(gin));
    else align_tokens_bwd_kernel<float><<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(gout), B, Nin, Nout, D, reinterpret_cast<float*>(gin));
    return cudaGetLastError();
}
__global__ void fill_f32_kernel(float* __restrict__ p, float v, int n) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) p[i] = v;
}
cudaError_t launch_fill_f32(float* p, float v, int n, cudaStream_t st) {
    fill_f32_kernel<<<(n + 255) / 256 < 64 ? (n + 255) / 256 : 64, 256, 0, st>>>(p, v, n);
    return cudaGetLastError();
}

}  // namespace basd
