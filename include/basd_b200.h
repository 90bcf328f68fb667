/* basd_b200.h — C ABI of the B200-native BASD distillation-loss hot path.
 *
 * The reference (indrajeetadityaroy9/vit-bias-aware-structural-distillation) has no FFI: its boundary is the Python
 * call BASDLoss.forward (src/losses/combined.py:48-85) plus the free function marchenko_pastur_rank
 * (src/losses/layer_selector.py:8-20, second consumer src/models/teacher.py:177).  This header is what a binding for
 * that path binds to; the drop-in Python module (vit_bias_aware_structural_distillation_b200/loss.py) is such a binding
 * (ctypes).  INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - every pointer is DEVICE memory owned by the caller (the library never allocates or frees);
 *   - every call is asynchronous on `stream` and never synchronises with the host;
 *   - return value 0 = success, non-zero = error; basd_last_error() gives a thread-local message;
 *   - one workspace (basd_workspace_bytes) carries all intermediates from the forward phases to the backward
 *     phases of the same step; it must stay untouched in between;
 *   - the four phases are separate entry points so the host language can place the two collectives
 *     (sum all-reduce of basd_view "stats" after phase 1, of "gw" after phase 3) with its own NCCL binding.
 */
#ifndef BASD_B200_H
#define BASD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BASD_DTYPE_F32 0
#define BASD_DTYPE_BF16 1
/* basd_shape.act_dtype only: fp32 tokens carried as split-bf16 pairs hi = bf16(x), lo = bf16(x - hi) instead of being rounded
 * to bf16 on entry (every product reads them as hi*hi + hi*lo + lo*hi, every streaming kernel as hi + lo; fp32-class accuracy) */
#define BASD_DTYPE_F32_SPLIT 2
#define BASD_MAX_POINTS 8
#define BASD_MAX_LAYERS 64

typedef struct basd_shape {
    int B;          /* local (per-rank) batch                                         */
    int Ns, Nt;     /* student / teacher tokens without CLS   (trainer.py:29, teacher.py:156-157) */
    int Ds, Dt;     /* student / teacher width                                        */
    int Lt;         /* teacher layers handed over (sorted keys, layer_selector.py:123) */
    int P;          /* student extraction points (combined.py:34-40)                  */
    int H;          /* attention heads (1 for CNN teachers, teacher.py:188-191)       */
    int has_cls;    /* teacher_has_cls_token (combined.py:27), or BASD_ATTN_QUERY_MEAN  */
    int act_dtype;  /* BASD_DTYPE_* of student and teacher tokens: BASD_DTYPE_BF16 (read in place), BASD_DTYPE_F32 (rounded
                       to bf16 on entry) or BASD_DTYPE_F32_SPLIT (fp32 tokens kept as split-bf16 pairs; more workspace) */
    int attn_dtype; /* BASD_DTYPE_F32 or BASD_DTYPE_BF16 of attention maps                                          */
    int world_size; /* ranks whose pooled statistics are summed (equal local batches) */
    int polar_steps;/* Newton-Schulz steps of the Procrustes polar iteration: 0 = default (10: singular values of the
                       cross-covariance down to 3e-5 ||C||_F), up to 16 (each step more divides that floor by ~4);
                       the residual of the last forward is in basd_view "polar_resid" */
    int mode;       /* BASD_MODE_*: which part of the path the four phases run (0 = the whole loss)                     */
} basd_shape;

/* basd_shape.mode
 *   BASD_MODE_LOSS      BASDLoss.forward's geometric term (combined.py:58-76): selector + alignment + Procrustes.
 *   BASD_MODE_PAIR      geometric_relational_loss (relational.py:5-50) of ONE student / teacher pair on its own: Lt = P = 1, the
 *                       layer selector is bypassed (mixing weight 1), proj_s / proj_t / log_temperatures are not read (may be
 *                       null); grad_log_temperatures comes back as zeros.
 *   BASD_MODE_SELECTOR  GrassmannianLayerSelector.forward's mixing weights (layer_selector.py:116-152 up to :108) on their own:
 *                       phases 1-2 stop at view "w" [P*Lt] (attention pointers are not read, geo_loss = 0); phase 3 is a no-op;
 *                       phase 4 takes d(total)/d(w) from view "gw" (written by the caller, *grad_geo multiplies it) and returns
 *                       the gradients w.r.t. the student tensors and log_temperatures through the closed-form selector backward. */
/* basd_shape.has_cls
 *   0                     no CLS token: every attention pointer holds the full map [B,H,Nt,Nt] (relational.py:27 averages it
 *                         over heads and queries).
 *   1                     CLS token: the full map [B,H,Nt+1,Nt+1] or its CLS query row [B,H,1,Nt+1] (relational.py:24).
 *   BASD_ATTN_QUERY_MEAN  no CLS token, and every attention pointer holds the query-mean row per head [B,H,1,Nt]
 *                         (basd_query_mean_attention): what relational.py:27 reads of the full map, without the map. */
#define BASD_ATTN_QUERY_MEAN 2

#define BASD_MODE_LOSS 0
#define BASD_MODE_PAIR 1
#define BASD_MODE_SELECTOR 2

typedef struct basd_inputs {
    const void* student[BASD_MAX_POINTS];   /* P  tensors [B,Ns,Ds]; element strides below            */
    const void* teacher[BASD_MAX_LAYERS];   /* Lt tensors [B,Nt,Dt]                                   */
    const void* attn[BASD_MAX_LAYERS];      /* Lt tensors [B,H,Nt+1,Nt+1] (has_cls) or [B,H,Nt,Nt]; rows: see has_cls */
    int64_t student_strides[3];             /* (batch, token, feature) in elements, same for all P    */
    int64_t teacher_strides[3];
    int64_t attn_strides[4];                /* (batch, head, query, key)                              */
    const float* proj_s;                    /* [Ds,Ds] row-major  (layer_selector.py:51,55)           */
    const float* proj_t;                    /* [Ds,Dt] row-major  (layer_selector.py:52,56)           */
    const float* log_temperatures;          /* [P]                (layer_selector.py:58-63)           */
} basd_inputs;

/* Bytes of workspace needed for one forward+backward step of `shape`. */
int basd_workspace_bytes(const basd_shape* shape, size_t* bytes);

/* Phase 1 (replaces layer_selector.py:69-74,86-91,131-136 and relational.py:22-27 up to the pooled statistics):
 * attention importance rows, teacher projection (tcgen05), per-layer token Gram + column sums (tcgen05). */
int basd_forward_stats(const basd_shape* shape, const basd_inputs* in, void* workspace, void* stream);

/* Phase 2 (layer_selector.py:16-19,36-37,92-112; combined.py:63-76; relational.py:29-50): MP ranks, eigenbases,
 * principal angles, mixing weights, mixed teacher, per-sample Procrustes.  geo_loss: device float (mean over the local batch). */
int basd_forward_solve(const basd_shape* shape, const basd_inputs* in, void* workspace, float* geo_loss, void* stream);

/* Phase 3 (closed-form backward, SURVEY.md B.1-B.2): d loss / d mixing weights, unscaled, into view "gw". */
int basd_backward_dots(const basd_shape* shape, const basd_inputs* in, void* workspace, void* stream);

/* Phase 4 (SURVEY.md B.3-B.5): gradients w.r.t. the P student tensors (dense [B,Ns,Ds], dtype grad_dtype) and
 * log_temperatures [P] (fp32).  grad_geo: device float, upstream d(total)/d(geo_loss). */
int basd_backward_finish(const basd_shape* shape, const basd_inputs* in, void* workspace, const float* grad_geo,
                         void* const* grad_student, int grad_dtype, float* grad_log_temperatures, void* stream);

/* Named views into the workspace (for the collectives and for tests).  Names: "stats" [(Lt+P)*(Ds*Ds+Ds)] f32,
 * "gw" [P*Lt] f32, "ranks" [Lt] i32, "w" [P*Lt], "d2" [P*Lt], "geo_i" [P], "loss_b" [P*B], "rows" [Lt*B*Nt],
 * "a" [P*B*Ns], "evals" [(Lt+P)*Ds], "cos" [P*Lt*Ds], "dbg" [P*B*5] (nuc, tr_s, tr_t, polar residual ||X X^T - I||_F going into the
 * last Newton-Schulz step, ||C||_F^2), "polar_resid" [1] (largest residual over all problems: <= 0.1 means converged), "gdir", "ktt",
 * "polar_*" (state of the polar iteration; bf16 views count hi then lo elements). */
int basd_view(const basd_shape* shape, void* workspace, const char* name, void** ptr, size_t* count);

/* marchenko_pastur_rank(features[M,D]) (layer_selector.py:8-20), rank written to device int; D a multiple of 8 up to 4096
 * (teacher.py:177 passes unprojected D_t-wide features: D <= 224 runs in shared memory, <= 384 on the cluster solver, larger on
 * the one-CTA global-memory solver); either branch of :12-15 (M >= D, M < D).
 * workspace: at least basd_mp_rank_workspace_bytes(M, D). */
int basd_mp_rank_workspace_bytes(int64_t M, int D, size_t* bytes);
int basd_mp_rank(const void* features, int64_t M, int D, int dtype, int64_t row_stride, int* rank_out, void* workspace,
                 void* stream);

/* SURVEY.md section 8(f) rank 1 - teacher attention capture (src/models/teacher.py:27-39 recomputes the full
 * softmax(Q K^T * scale) map per block; the loss reads only its CLS query row, relational.py:24).  Emits that row:
 * out[b,h,:] = softmax_s(q[b,h,0,:] . k[b,h,s,:] * scale), fp32 [B,H,S].  q, k: [B,H,S,dh] with element strides
 * (b,h,s,d), d stride 1 (views into a fused qkv tensor are fine).  The result, viewed as [B,H,1,S], is accepted
 * by basd_forward_stats in place of the [B,H,S,S] map (attn_strides accordingly). */
int basd_cls_attention_rows(const void* q, const void* k, int dtype, int B, int H, int S, int dh, const int64_t* q_strides,
                            const int64_t* k_strides, float scale, float* out, void* stream);

/* The same for teachers WITHOUT a CLS token (relational.py:27 reads attn.mean over heads and all queries): emits the
 * query mean of every head's map, out[b,h,:] = (1/S) sum_q softmax_s(q[b,h,q,:] . k[b,h,s,:] * scale), fp32 [B,H,S], and never
 * stores an S x S map (two passes of tcgen05 products over q and k: row max / sum of exps per query, then the normalised
 * probabilities summed per key; fixed-order sums, bitwise repeatable).  q, k: [B,H,S,dh] with element strides (b,h,s,d),
 * d stride 1 (views into a fused qkv tensor are fine); dtype BASD_DTYPE_BF16, or BASD_DTYPE_F32 (split-bf16 products,
 * fp32-class accuracy).  dh a multiple of 8 up to 256, 1 <= S <= 2048; base 16-byte aligned, (b,h,s) strides multiples of 8
 * (bf16) or 4 (fp32) elements.  The result, viewed as [B,H,1,S], is accepted by basd_forward_stats with
 * has_cls = BASD_ATTN_QUERY_MEAN in place of the [B,H,S,S] map. */
int basd_query_mean_attention(const void* q, const void* k, int dtype, int B, int H, int S, int dh, const int64_t* q_strides,
                              const int64_t* k_strides, float scale, float* out, void* stream);

/* Host-resident teacher attention (an offline / CPU-resident teacher): copies the CLS query rows of a HOST map [B,H,S,S]
 * (element strides (b,h,q,k), k stride 1, 2- or 4-byte elements) to a dense DEVICE tensor [B,H,1,S] with one pitched DMA -
 * the only part of the map relational.py:24 reads.  Asynchronous on `stream` when the host memory is pinned. */
int basd_copy_cls_rows_h2d(const void* host_attn, int elem_bytes, int B, int H, int S, const int64_t* strides, void* dev_rows,
                           void* stream);

/* _align_token_count (combined.py:9-14) on its own: 1-D linear resampling along the token axis (align_corners = False) of
 * tokens [B,Nin,D] (element strides (b,n,d)) to a dense [B,Nout,D] tensor of the same dtype, and its adjoint
 * (grad_out dense [B,Nout,D] -> grad_in dense [B,Nin,D]).  Inside the loss the resampling is fused into the teacher mix. */
int basd_align_tokens(const void* tokens, int dtype, const int64_t* strides, int B, int Nin, int Nout, int D, void* out, void* stream);
int basd_align_tokens_bwd(const void* grad_out, int dtype, int B, int Nin, int Nout, int D, void* grad_in, void* stream);

/* UW-SO weighting of the two loss terms (combined.py:78-85) in one launch: with the DETACHED values d_i (det_ce, det_geo: the
 * terms themselves, or their means over the ranks of a batch-sharded job) and eps = the dtype's machine epsilon,
 *     w_i = (1 / max(d_i, eps)) / sum_j (1 / max(d_j, eps)),      out = [w_ce * ce + w_geo * geo, w_ce, w_geo].
 * All pointers are fp32 device scalars; the weights are what the backward multiplies the incoming gradient by. */
int basd_uwso_combine(const float* ce, const float* geo, const float* det_ce, const float* det_geo, float eps, float* out3, void* stream);

/* Test hooks (used by tests/ only). */
int basd_selftest_gemm(int variant, const void* A, const void* B, float* C, int M, int N, int K, void* stream);
int basd_selftest_eig(const float* G, int n, float* evals, float* evecs, int* sweeps, void* workspace, void* stream);

/* Live timing (CUDA events on the launching stream around each kernel group) and launch counting, for bench.py.
 * A single-caller measurement facility: the event brackets are process-global and NOT re-entrant (off by default; the
 * launch counter is atomic).  The compute entry points themselves keep no mutable process state. */
void basd_timing_enable(int on);
void basd_timing_reset(void);
long long basd_launch_count(void);
int basd_timing_slots(void);
const char* basd_timing_name(int slot);
int basd_timing_read(int slot, float* ms_total, int* brackets);

/* Number of Newton-Schulz steps of the Procrustes polar iteration. */
int basd_polar_steps(void);
/* Products launched per Newton-Schulz step for these sizes: 3 when A = T W^T and the polynomial in A are fused into one
 * kernel (D_s <= 192), 4 otherwise.  For bench.py's launch and byte counts. */
int basd_polar_launches_per_step(int Ds, int Ns);

const char* basd_last_error(void);
const char* basd_version(void);

#ifdef __cplusplus
}
#endif
#endif /* BASD_B200_H */
