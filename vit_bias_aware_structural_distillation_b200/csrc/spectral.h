// Internal declarations shared by the kernels and the C-ABI orchestration (not part of the public ABI).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace basd {

constexpr int kSpectralThreads = 768;
constexpr int kMaxPoints = 8;         // extraction points P
constexpr int kMaxLayers = 64;        // teacher layers Lt


constexpr int kSpectralSmemMax = 224;  // largest symmetric problem whose matrix fits one SM's shared memory
bool spectral_large(int n);            // n > kSpectralSmemMax: matrices in global scratch (pooled_eig_scratch_floats)
size_t pooled_eig_scratch_floats(int n, int problems);
// mode kEigPooled: Lt + P centred eigenproblems (teacher layers, then student points); the MP rank of every teacher layer comes
// from its centred eigensystem (rank-one secular equation).  mode kEigMpOnly: Lt uncentred problems, ranks only (evals / evecs
// unused) - the free function marchenko_pastur_rank, which also takes M < D.
constexpr int kEigPooled = 1, kEigMpOnly = 2;
cudaError_t launch_pooled_eig(const float* stats, int n, int Lt, int P, float Mt, float Ms, int* ranks, float* evals,
                              float* evecs_km, float* evecs_cm, int* sweeps, float* scratch, cudaStream_t st, int mode = kEigPooled);
cudaError_t launch_angles(int n, int Lt, int P, const int* ranks, const float* evals, const float* evecs_km,
                          const float* evecs_cm, const float* proj_s, float* scratch, float* d2, float* gamma,
                          float* cos_out, const float* log_temp, float* w, cudaStream_t st);
cudaError_t launch_selector_bwd(int n, int Lt, int P, const float* gw_raw, const float* scale_ptr, float scale_host,
                                const float* w, const float* d2, const float* log_temp, const float* gamma,
                                const float* stats, float Ms, __nv_bfloat16* gam_hi, __nv_bfloat16* gam_lo, float* corr,
                                float* grad_log_temp, cudaStream_t st);

// linear resampling index along the token axis (align_corners = False), combined.py:12-14
#ifdef __CUDACC__
__device__ __forceinline__ void interp_index(int n, int n_in, int n_out, int& i0, int& i1, float& lam) {
    if (n_in == n_out) { i0 = n; i1 = n; lam = 0.f; return; }
    const float scale = static_cast<float>(n_in) / static_cast<float>(n_out);
    float x = scale * (static_cast<float>(n) + 0.5f) - 0.5f;
    x = fmaxf(x, 0.f);
    i0 = min(static_cast<int>(x), n_in - 1);
    i1 = min(i0 + 1, n_in - 1);
    lam = x - static_cast<float>(i0);
}
#endif

// ---- streaming kernels (stream_ops.cu)
struct PtrTable {                         // small by-value pointer tables for per-layer tensors
    const void* p[kMaxLayers];
};
cudaError_t launch_importance_rows(const PtrTable& attn, int attn_is_bf16, int Lt, int B, int H, int Nt, int has_cls,
                                   const long long* strides /*[b,h,q,k] elements*/, float* rows, cudaStream_t st);
cudaError_t launch_split_bf16(const float* src, __nv_bfloat16* hi, __nv_bfloat16* lo, size_t n, cudaStream_t st);
cudaError_t launch_pack_bf16(const void* src, int src_is_bf16, long long sb, long long sn, long long sd, int B, int N,
                             int D, __nv_bfloat16* dst, __nv_bfloat16* dst_lo /*null: round to bf16*/, cudaStream_t st);
struct ColsumJobs {                       // out[j][d] += sum_rows (hi[j] + lo[j])[row][d]; lo may be null
    const __nv_bfloat16* hi[kMaxLayers + kMaxPoints];
    const __nv_bfloat16* lo[kMaxLayers + kMaxPoints];
    float* out[kMaxLayers + kMaxPoints];
};
size_t colsum_part_floats(int n_jobs, size_t rows, int D);      // scratch for the per-CTA partial sums (fixed-order reduce)
// rows_per_batch > 0: the job tensors are [B][rows_per_batch][D] with batch stride batch_stride elements (CLS-stripped views)
cudaError_t launch_colsum(const ColsumJobs& jobs, int n_jobs, size_t rows, int D, float* part, cudaStream_t st, int rows_per_batch = 0,
                          long long batch_stride = 0);
cudaError_t launch_importance_mix(const float* rows, const float* w, int Lt, int P, int B, int Nt, int Ns, float* a,
                                  float* ssum, cudaStream_t st);
// teacher_lo (non-null): split-bf16 teacher tokens, read as hi + lo (BASD_DTYPE_F32_SPLIT)
cudaError_t launch_mix_teacher(const PtrTable& teacher, const float* w, int Lt, int P, int B, int Nt, int Ns, int Dt,
                               __nv_bfloat16* hi, __nv_bfloat16* lo, cudaStream_t st, long long teacher_batch_stride = 0 /*0: Nt * Dt*/,
                               const PtrTable* teacher_lo = nullptr);
// Dtm is [P][B][Nd][Dt] with Nd = Ns (gradient w.r.t. the token-aligned mixed teacher) or, with dtm_unaligned, Nd = Nt
// (gradient w.r.t. the mixed teacher on its own token grid: no resampling in the dots)
cudaError_t launch_wgrad_dots(const PtrTable& teacher, const __nv_bfloat16* Dtm, const __nv_bfloat16* Dtm_lo, const float* gwt, const float* rows,
                              int Lt, int P, int B, int Nt, int Ns, int Dt, float* gw /*[P][Lt]*/,
                              float* gw_part /*wgrad_part_floats(P, Lt) floats: per-CTA partials, summed in a fixed order*/,
                              cudaStream_t st, bool dtm_unaligned = false, long long teacher_batch_stride = 0 /*0: Nt * Dt*/,
                              const PtrTable* teacher_lo = nullptr /*split-bf16 teachers: read as hi + lo*/);
size_t wgrad_part_floats(int P, int Lt);
cudaError_t launch_cls_attention_rows(const void* q, const void* k, int is_bf16, int B, int H, int S, int dh,
                                      const long long* q_strides /*[b,h]*/, const long long* k_strides /*[b,h,s]*/, float scale,
                                      float* out /*[B,H,S]*/, cudaStream_t st);
// (attention_rows.cu) out[b,h,s] = mean over queries of softmax(scale q k^T)[., s], fp32 [B,H,S]; q, k [B,H,S,dh] with (b,h,s)
// element strides, d stride 1.  bf16: 16-byte aligned base and strides; fp32: 16-byte aligned base, strides multiples of 4.
constexpr int kQueryMeanMaxTokens = 2048, kQueryMeanMaxHeadDim = 256;
cudaError_t launch_query_mean_attention(const void* q, const void* k, int is_bf16, int B, int H, int S, int dh,
                                        const long long* q_strides /*[b,h,s]*/, const long long* k_strides /*[b,h,s]*/, float scale,
                                        float* out /*[B,H,S]*/, cudaStream_t st);
// standalone combined.py:9-14 (tokens [B,Nin,D] with element strides -> dense [B,Nout,D]) and its adjoint (dense in, dense out)
cudaError_t launch_align_tokens(const void* src, int is_bf16, long long sb, long long sn, long long sd, int B, int Nin, int Nout, int D,
                                void* dst, cudaStream_t st);
cudaError_t launch_align_tokens_bwd(const void* gout, int is_bf16, int B, int Nin, int Nout, int D, void* gin, cudaStream_t st);
cudaError_t launch_fill_f32(float* p, float v, int n, cudaStream_t st);
// geo_i[P], *geo = mean; resid_max = max over the problems of dbg[.][3] (polar residual)
cudaError_t launch_loss_reduce(const float* loss_b, const float* dbg, int P, int B, float* geo_i, float* geo, float* resid_max, cudaStream_t st);

// ---- tcgen05 GEMM launchers (gemm_ops.cu)
int gemm_init_driver_api();               // resolves cuTensorMapEncodeTiled; 0 on success
// Z[j] = X[j] P^T for n_layers separate [M][Dt] bf16 tensors; Zhi / Zlo are [n_layers][M][Ds]
// gap_period > 0: rows r of X with r % gap_period >= gap_valid lie between two samples (CLS-stripped view of a
// [B][N+1][Dt] buffer read as a dense matrix of M rows): their Z rows are written as zeros
// Xlo non-null (split-bf16 teachers): X[0] is the hi block [n_layers][M][Dt], Xlo the lo block; Z = X_hi P_hi^T + X_hi P_lo^T + X_lo P_hi^T
cudaError_t gemm_project(const void* const* X, int n_layers, size_t M, int Dt, const __nv_bfloat16* Phi, const __nv_bfloat16* Plo,
                         int Ds, __nv_bfloat16* Zhi, __nv_bfloat16* Zlo, int gap_period, int gap_valid, cudaStream_t st,
                         const __nv_bfloat16* Xlo = nullptr);
// Zlo may be null (exact bf16 input); otherwise Z = Zhi + Zlo and the Gram uses hi*hi + hi*lo + lo*hi
// G[i] (stride g_stride floats) += S_i^T S_i for n separate exact-bf16 [M][Ds] tensors, one launch
// Split-K slices go to `part` (gemm_gram_part_floats floats) and are summed in a fixed order: bitwise repeatable Grams.
size_t gemm_gram_part_floats(size_t M, int Ds, int batches);
// with_colsum: the column sums of every operand come out of the same pass (an N = 16 ones-operand MMA per k-step) and are written
// behind its Gram, G[i] + Ds * Ds - the layout of the pooled statistics; g_stride >= Ds * Ds + Ds then.
bool gemm_gram_colsum_fused(int Ds, bool split);         // false: that shape keeps the separate column-sum kernel
cudaError_t gemm_gram_table(const void* const* S, int n, size_t M, int Ds, float* G, long long g_stride, float* part, int rows_per_batch,
                            long long batch_stride, cudaStream_t st, bool with_colsum = false);
cudaError_t gemm_gram(const __nv_bfloat16* Z, const __nv_bfloat16* Zlo, size_t M, int Ds, float* G /*[Ds][Ds]*/, float* part,
                      cudaStream_t st);
cudaError_t gemm_gram_batched(const __nv_bfloat16* Z, const __nv_bfloat16* Zlo, size_t M, int Ds, int batches, float* G,
                              long long g_stride, float* part, cudaStream_t st, bool with_colsum = false);
cudaError_t gemm_token_gram(const __nv_bfloat16* Thi, const __nv_bfloat16* Tlo, int batches, int Ns, int Dt, float* Ktt,
                            cudaStream_t st);
cudaError_t gemm_theta_apply(const __nv_bfloat16* theta_hi, const __nv_bfloat16* theta_lo, int NsPad, const __nv_bfloat16* Thi,
                             const __nv_bfloat16* Tlo, int batches, int Ns, int Dt, __nv_bfloat16* Dtm, __nv_bfloat16* Dtm_lo, cudaStream_t st);
cudaError_t gemm_student_grad(const __nv_bfloat16* S, size_t M, int Ds, const __nv_bfloat16* Ghi, const __nv_bfloat16* Glo,
                              const float* gdir, const float* corr, const float* scale_ptr, float scale_host, void* out,
                              int out_is_bf16, int gap_period, int gap_valid, cudaStream_t st,
                              const __nv_bfloat16* S_lo = nullptr /*split-bf16 students: adds the term S_lo Gamma'_hi*/);
// generic test hook: C[M][N] (fp32) = A[M][K] * B[N][K]^T or with MN-major operands (see basd_b200.h selftest)
cudaError_t gemm_selftest(int variant, const __nv_bfloat16* A, const __nv_bfloat16* B, float* C, int M, int N, int K,
                          cudaStream_t st);
const char* gemm_last_error();

// CUDA-event bracket + launch counter of basd_capi.cu (live timing for bench.py), usable from every translation unit
struct TimingScope {
    void* impl;
    TimingScope(int slot, cudaStream_t st, int n_launches);
    ~TimingScope();
    TimingScope(const TimingScope&) = delete;
    TimingScope& operator=(const TimingScope&) = delete;
};
constexpr int kSlotPolarPrep = 10, kSlotPolarGemm = 16, kSlotPolarFinish = 17;

// ---- Newton-Schulz polar iteration of the Procrustes core (polar.cu + polar_gemm.cuh)
struct SplitMat {                         // bf16 hi/lo pair, column-block tiled: [batch][col / 64][row][col % 64]
    __nv_bfloat16* hi; __nv_bfloat16* lo;
    int rows, inner;                      // valid rows / columns
    long long batch_stride;               // elements per problem = ceil(inner / 64) * rows * 64
    __host__ __device__ size_t at(int r, int c) const { return (static_cast<size_t>(c >> 6) * rows + r) * 64 + (c & 63); }
};
struct PolarFusedArgs {
    int n;                           // D_s: rows of T and W, order of A
    int k_total;                     // N_s
    int bn;                          // n rounded up to 16 (UMMA N)
    int rows_ld;                     // n rounded up to 64 (rows loaded / copied per k-block)
    int n_mt;                        // 128-row tiles (1 or 2)
    int n_problems, reverse;
    float ca, cb, cc;                // Bm = ca I + cb (rA) + cc (rA)^2
    int first;                       // step 0: r = 1 / trace(A) (written to fro2); otherwise r = 1
    float* fro2;                     // [problem][fro_slots]: slot 0 written here
    int fro_slots;
    float* resid;                    // last step only: [problem][fro_slots] per-warp partial sums of ||A - I||_F^2 (else null)
};
// Bm = ca I + cb (rA) + cc (rA)^2 with A = T W^T kept on chip (polar_fused.cuh); needs polar_fused_supported(D_s, N_s)
bool polar_fused_supported(int n, int k);
cudaError_t polar_fused_abm(const SplitMat& T, const SplitMat& W, const SplitMat& Bm, int batches, PolarFusedArgs& args, cudaStream_t st);
struct PolarGemmArgs;
// out = A (rows x K, K-major) * B^T; B is K-major ([n_cols][K]) or, with b_mn, the row-major [K][n_cols] buffer.
cudaError_t polar_gemm(bool b_mn, const SplitMat& A, const SplitMat& B, int batches, PolarGemmArgs& args, cudaStream_t st);

struct PolarArgs {
    int Ns, Ds, B, P, NsPad;
    int n_problems;                       // P * B
    // teacher-token-space form (launch_polar_procrustes_vt): D_s > min(N_s, N_t) - 1, N_t <= N_s
    int vt;                               // 1: this form is running (prep_student skips W_0)
    int Nt, NtPad;                        // unaligned teacher tokens; row pitch of theta in this form
    int Dsp;                              // feature columns of X: D_s rounded up to 16, + 8 (the decoupled augmentation column sits at Ds16)
    SplitMat FG, FGt;                     // F G [Ns][Nt] and its transpose [Nt][Ns]   (F = diag(q)(I - 1 a^T)E, G G^T = K_R)
    SplitMat GinvC, GinvT;                // G^-1 (I - 1 1^T / Nt) [Nt][Nt] and G^-T [Nt][Nt]
    SplitMat X0, X1, X2;                  // [Nt][Dsp]: whitened cross-covariance and the two iterates
    SplitMat Hm, M2;                      // [Nt][Nt]
    float* ginv;                          // [P*B][Nt*Nt] fp32 scratch (column-major inverse of the Cholesky factor)
    float* thraw;                         // [P*B][Nt][Nt]
    float* ftf;                           // [P*B][Nt][Nt]   F^T F
    const __nv_bfloat16* student[kMaxPoints];   // [B][Ns][Ds] bf16, batch stride student_bs elements (Ns * Ds when dense)
    const __nv_bfloat16* student_lo[kMaxPoints];  // split-bf16 students: lo halves (dense), s = hi + lo; null otherwise
    long long student_bs;
    const float* Ktt;                     // [P*B][Ns][Ns]   uncentred token Gram of the mixed teacher
    const float* a;                       // [P*B][Ns]       normalised importance
    const float* ssum;                    // [P*B]
    // scratch (all per problem)
    SplitMat W, W2, T, A, Bm, Kt, SW;
    float* Gsw;                           // [P*B][Ns][Ds]   d nuc / d s_w
    float* vec;                           // [P*B][4][Ns]    ksd, ktd, (spare), (spare)
    float* scal;                          // [P*B][4]        (spare), tr_s, tr_t, (spare)
    float* fro2;                          // [P*B][fro_slots]  partial traces of A_0; their sum = ||C||_F^2
    int fro_slots;
    float* resid;                         // [P*B][fro_slots]  partial sums of ||A - I||_F^2 at the last step (A = X X^T before the last update)
    int steps;                            // Newton-Schulz steps (kPolarStepsDefault .. kPolarStepsMax)
    // outputs
    float* gdir;                          // [P*B][Ns][Ds]
    __nv_bfloat16* theta;                 // [P*B][Ns][NsPad] hi
    __nv_bfloat16* theta_lo;              // [P*B][Ns][NsPad] lo
    float* gwt;                           // [P*B][Ns]
    float* loss_b;                        // [P*B]
    float* dbg;                           // [P*B][5]
};
cudaError_t launch_polar_procrustes(const PolarArgs& args, cudaStream_t st);
cudaError_t launch_polar_procrustes_vt(const PolarArgs& args, cudaStream_t st);
constexpr int kVtMaxTokens = 224;         // teacher tokens of the token-space form (Cholesky factor held in shared memory)
int polar_fro_slots(int core);            // partial-trace slots per problem for a core (D_s or N_t) of this size
constexpr int kPolarStepsDefault = 10, kPolarStepsMin = 7, kPolarStepsMax = 16;   // (fewer than the default: caller override only, rows of the schedule skipped from the front)
int polar_steps();                        // default number of Newton-Schulz steps (the final iterate lives in W2 when odd, W when even)

}  // namespace basd
