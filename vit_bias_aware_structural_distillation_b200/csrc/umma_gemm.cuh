// Warp-specialised tcgen05 GEMM for sm_100a: TMA (SWIZZLE_128B) -> shared memory ring -> tcgen05.mma
// (bf16 x bf16 -> fp32 in TMEM) -> tcgen05.ld epilogue.  One CTA = MT x (128 x BN) output tiles.
//
// Instances on the BASD loss path (see gemm_ops.cu):
//   gram         G += Z_chunk^T Z_chunk      (replaces layer_selector.py:13,36,92)    A,B MN-major, split-K
//   token_gram   K = T T^T per sample        (relational.py:47 moved to token space)  A,B K-major, B aliases A; N_s < 16 only
//   student_grad dS = S Gamma + ...          (SURVEY.md B.5)                          A,B K-major; views, fp32 or split students
//   (project, the other token Grams, theta_apply and the dense bf16 student gradient run on the persistent polar_gemm kernel)
// "Split-bf16" terms (hi/lo operand pairs) accumulate into the same TMEM tile to recover fp32-class
// accuracy from bf16 tensor-core passes.
#pragma once
#include "ptx.cuh"

namespace basd {

constexpr int GEMM_BK = 64;           // bf16 elements per k-block = one 128-byte swizzle row
constexpr int GEMM_THREADS = 192;     // warp0 TMA, warp1 MMA, warps2-5 epilogue

constexpr int GEMM_MAX_A_TABLE = 16;
struct GemmMaps {                     // up to two A and two B operand buffers (hi / lo)
    CUtensorMap a[2];
    CUtensorMap b[2];
    CUtensorMap a_table[GEMM_MAX_A_TABLE];   // GemmArgs::a_table: A operand of batch z when the batches are separate allocations
};

struct GemmArgs {
    int kb_total;        // number of 64-wide k-blocks
    int kb_per_split;    // split-K: k-blocks per split (0 = no split, blockIdx.z is the batch index)
    int n_splits;        // split-K: blockIdx.z = batch * n_splits + split
    int a_batched;       // A uses blockIdx.z as 3rd TMA coordinate
    int b_batched;       // B uses blockIdx.z as 3rd TMA coordinate
    int a_table;         // A (single buffer) comes from maps.a_table[batch] (teacher layers live in separate tensors)
    int b_table;         // B (single buffer) comes from maps.a_table[batch] too (Gram of separate tensors: B = A)
    // epilogue
    void* out;           // primary output
    long long out_batch_stride;   // elements
    int ld_out;          // elements
    int rows_valid;      // rows of the (per-batch) output that exist
    int cols_valid;
    const void* aux0;    // epilogue specific
    const void* aux1;
    const void* aux2;
    long long aux_batch_stride;
    float alpha;
    float beta;
    // Row-gapped A operand (K-major, rows = M): a [B][N+1][D] buffer read through its CLS-stripped view [:,1:,:] is a dense
    // 2-D matrix whose rows r with r % gap_period >= gap_valid belong to no sample (trainer.py:29, teacher.py:157 hand such
    // views over).  gap_period == 0: no gaps.  The student_grad epilogue skips those rows.
    int gap_period, gap_valid;
    // MN-major operands whose K dimension runs over the rows of a [B][N][D] tensor with an arbitrary batch stride: the tensor
    // map is 3-D (D, N, B) and k-block kb covers rows (kb % kb_per_batch) * 64.. of sample kb / kb_per_batch; rows past N are
    // zero-filled by TMA.  kb_per_batch == 0: flat rows.
    int kb_per_batch;
};

// COLSUM (Gram configurations, A MN-major): the column sums of the A operand over the K rows of this CTA's split-K slice come out
// of the same pass as the Gram - one extra N = 16 MMA per k-step against a constant "ones" tile (row 0 = 1, K-major), i.e.
// sum_k A[k][m] * 1, into 16 more TMEM columns per row tile.  The separate colsum kernel re-read every Gram operand (540 MB,
// 0.1 ms at cfg2).
template <bool A_MN, bool B_MN, int BN, int MT, int NA, int NB, int NTERMS, bool B_ALIAS_A, int STAGES, bool COLSUM = false>
struct GemmCfg {
    static constexpr bool kAMN = A_MN, kBMN = B_MN, kAlias = B_ALIAS_A, kColsum = COLSUM;
    static constexpr int kBN = BN, kMT = MT, kNA = NA, kNB = NB, kTerms = NTERMS, kStages = STAGES;
    static constexpr int kABytes = MT * 128 * 128;                    // per A buffer per stage
    static constexpr int kBBytes = B_ALIAS_A ? 0 : BN * 128;          // per B buffer per stage
    static constexpr int kStageBytes = NA * kABytes + NB * kBBytes;
    static constexpr int kAccCols = MT * BN + (COLSUM ? MT * 16 : 0);
    static constexpr int kTmemCols = (kAccCols <= 32) ? 32 : (kAccCols <= 64) ? 64 : (kAccCols <= 128) ? 128 : (kAccCols <= 256) ? 256 : 512;
    static constexpr int kOnesBytes = COLSUM ? 2048 : 0;              // [16 rows][64 k] bf16, 128-byte rows (row 0 is not moved by the swizzle)
    static constexpr int kSmemBytes = STAGES * kStageBytes + kOnesBytes + 1024 /*align*/ + 256 /*barriers*/;
    static_assert(kAccCols <= 512, "accumulators exceed TMEM");
    static_assert(!COLSUM || A_MN, "COLSUM sums an MN-major A operand over its K rows");
    static_assert(BN % 16 == 0 && BN <= 256, "invalid UMMA N");
    static_assert(!B_MN || BN % 64 == 0, "MN-major B needs 64-wide groups");
    static_assert(!B_ALIAS_A || (A_MN == B_MN && BN <= MT * 128), "alias: B = the first BN rows / columns of the A tile, same major");
    static_assert(kSmemBytes <= 232448, "shared memory budget");
};

// term t multiplies A[a_sel] by B[b_sel]:  t=0 (0,0)  t=1 (0,1)  t=2 (1,0)   (hi*hi, hi*lo, lo*hi)
__device__ __forceinline__ int term_a(int t) { return t == 2 ? 1 : 0; }
__device__ __forceinline__ int term_b(int t) { return t == 1 ? 1 : 0; }

template <class Cfg, class Epi>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
umma_gemm_kernel(const __grid_constant__ GemmMaps maps, const GemmArgs args) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* ones_tile = smem + Cfg::kStages * Cfg::kStageBytes;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + Cfg::kStages * Cfg::kStageBytes + Cfg::kOnesBytes);
    uint64_t* empty_bar = full_bar + Cfg::kStages;
    uint64_t* tmem_full_bar = empty_bar + Cfg::kStages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int z = blockIdx.z;
    int kb0 = 0, kb1 = args.kb_total;
    int batch = z;
    if (args.kb_per_split > 0) {
        batch = z / args.n_splits;
        kb0 = (z % args.n_splits) * args.kb_per_split;
        kb1 = min(args.kb_total, kb0 + args.kb_per_split);
    }
    const int a_row0 = blockIdx.y * (Cfg::kMT * 128);
    const int b_row0 = blockIdx.x * Cfg::kBN;

    if (threadIdx.x == 0) {
        for (int s = 0; s < Cfg::kStages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        mbar_init(tmem_full_bar, 1);
        fence_mbar_init();
        for (int i = 0; i < Cfg::kNA; ++i) tma_prefetch_desc(args.a_table ? &maps.a_table[batch] : &maps.a[i]);
        if (!Cfg::kAlias)
            for (int i = 0; i < Cfg::kNB; ++i) tma_prefetch_desc(&maps.b[i]);
    }
    if (warp == 1) tmem_alloc(tmem_slot, Cfg::kTmemCols);
    if constexpr (Cfg::kColsum) {                            // ones tile: row 0 = 1.0 (64 bf16), rows 1..15 = 0
        for (int t = threadIdx.x; t < Cfg::kOnesBytes / 4; t += blockDim.x)
            reinterpret_cast<uint32_t*>(ones_tile)[t] = t < 32 ? 0x3F803F80u : 0u;
        fence_proxy_async_smem();                            // generic-proxy writes -> visible to the tensor core
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer
        if (lane == 0) {
            const int za = args.a_batched ? batch : 0;
            const int zb = args.b_batched ? batch : 0;
            for (int kb = kb0; kb < kb1; ++kb) {
                const int it = kb - kb0;
                const int s = it % Cfg::kStages;
                const uint32_t ph = (it / Cfg::kStages) & 1;
                mbar_wait(&empty_bar[s], ph ^ 1);
                mbar_arrive_expect_tx(&full_bar[s], Cfg::kStageBytes);
                uint8_t* st = smem + s * Cfg::kStageBytes;
#pragma unroll
                for (int i = 0; i < Cfg::kNA; ++i) {
                    uint8_t* dst = st + i * Cfg::kABytes;
                    const CUtensorMap* amap = args.a_table ? &maps.a_table[batch] : &maps.a[i];
                    if (Cfg::kAMN) {
                        const int krow = args.kb_per_batch ? (kb % args.kb_per_batch) * GEMM_BK : kb * GEMM_BK;
                        const int kz = args.kb_per_batch ? kb / args.kb_per_batch : za;
#pragma unroll
                        for (int g = 0; g < Cfg::kMT * 2; ++g)
                            tma_load_3d(dst + g * 8192, amap, &full_bar[s], a_row0 + g * 64, krow, kz);
                    } else {
#pragma unroll
                        for (int mt = 0; mt < Cfg::kMT; ++mt)
                            tma_load_3d(dst + mt * 16384, amap, &full_bar[s], kb * GEMM_BK, a_row0 + mt * 128, za);
                    }
                }
                if (!Cfg::kAlias) {
#pragma unroll
                    for (int i = 0; i < Cfg::kNB; ++i) {
                        uint8_t* dst = st + Cfg::kNA * Cfg::kABytes + i * Cfg::kBBytes;
                        const CUtensorMap* bmap = args.b_table ? &maps.a_table[batch] : &maps.b[i];
                        if (Cfg::kBMN) {
                            const int krow = args.kb_per_batch ? (kb % args.kb_per_batch) * GEMM_BK : kb * GEMM_BK;
                            const int kz = args.kb_per_batch ? kb / args.kb_per_batch : zb;
#pragma unroll
                            for (int g = 0; g < Cfg::kBN / 64; ++g)
                                tma_load_3d(dst + g * 8192, bmap, &full_bar[s], b_row0 + g * 64, krow, kz);
                        } else {
                            tma_load_3d(dst, bmap, &full_bar[s], kb * GEMM_BK, b_row0, zb);
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (one elected lane)
        constexpr uint32_t idesc = umma_idesc_bf16(128, Cfg::kBN, Cfg::kAMN, Cfg::kBMN);
        for (int kb = kb0; kb < kb1; ++kb) {
            const int it = kb - kb0;
            const int s = it % Cfg::kStages;
            const uint32_t ph = (it / Cfg::kStages) & 1;
            mbar_wait(&full_bar[s], ph);
            tc_fence_after();
            if (lane == 0) {
                const uint32_t st = smem_u32(smem + s * Cfg::kStageBytes);
#pragma unroll
                for (int mt = 0; mt < Cfg::kMT; ++mt) {
#pragma unroll
                    for (int t = 0; t < Cfg::kTerms; ++t) {
                        const uint32_t a_base = st + term_a(t) * Cfg::kABytes + mt * 16384;
                        const uint32_t b_base = Cfg::kAlias ? (st + term_b(t) * Cfg::kABytes)
                                                            : (st + Cfg::kNA * Cfg::kABytes + term_b(t) * Cfg::kBBytes);
#pragma unroll
                        for (int ks = 0; ks < GEMM_BK / 16; ++ks) {
                            const uint64_t adesc = Cfg::kAMN ? umma_smem_desc(a_base + ks * 2048, 8192, 1024)
                                                             : umma_smem_desc(a_base + ks * 32, 16, 1024);
                            const uint64_t bdesc = Cfg::kBMN ? umma_smem_desc(b_base + ks * 2048, 8192, 1024)
                                                             : umma_smem_desc(b_base + ks * 32, 16, 1024);
                            umma_bf16(tmem_base + mt * Cfg::kBN, adesc, bdesc, idesc, (it > 0 || t > 0 || ks > 0) ? 1u : 0u);
                        }
                    }
                    if constexpr (Cfg::kColsum) {            // column sums of every A buffer (hi, lo) of this row tile
                        constexpr uint32_t idesc_cs = umma_idesc_bf16(128, 16, true, false);
#pragma unroll
                        for (int i = 0; i < Cfg::kNA; ++i) {
                            const uint32_t a_base = st + i * Cfg::kABytes + mt * 16384;
#pragma unroll
                            for (int ks = 0; ks < GEMM_BK / 16; ++ks)
                                umma_bf16(tmem_base + Cfg::kMT * Cfg::kBN + mt * 16, umma_smem_desc(a_base + ks * 2048, 8192, 1024),
                                          umma_smem_desc(smem_u32(ones_tile) + ks * 32, 16, 1024), idesc_cs, (it > 0 || i > 0 || ks > 0) ? 1u : 0u);
                        }
                    }
                }
                umma_commit(&empty_bar[s]);                 // frees the smem slot when these MMAs retire
                if (kb == kb1 - 1) umma_commit(tmem_full_bar);
            }
            __syncwarp();
        }
    } else {
        // ------------------------------------------------------------------ epilogue (4 warps = 128 TMEM lanes)
        if (kb1 > kb0) {
            mbar_wait(tmem_full_bar, 0);
            tc_fence_after();
            const int q = warp & 3;                          // TMEM lane quadrant this warp may read
            Epi epi(args, batch, z);
#pragma unroll 1
            for (int mt = 0; mt < Cfg::kMT; ++mt) {
                const int row = a_row0 + mt * 128 + q * 32 + lane;
#pragma unroll 1
                for (int c = 0; c < Cfg::kBN; c += 16) {
                    float v[16];
                    tmem_ld16(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + mt * Cfg::kBN + c, v);
                    epi(row, b_row0 + c, v);
                }
                if constexpr (Cfg::kColsum) {
                    float v[16];
                    tmem_ld16(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + Cfg::kMT * Cfg::kBN + mt * 16, v);
                    if (blockIdx.x == 0) epi.colsum(row, v[0]);      // (every column tile computes it; one stores it)
                }
            }
            tc_fence_before();
        }
    }
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, Cfg::kTmemCols);
    }
}

// ---------------------------------------------------------------------------------------------------
// Epilogues.  operator()(row, col0, v[16]) handles 16 consecutive columns of one output row.
// ---------------------------------------------------------------------------------------------------
struct EpiStoreF32 {                      // out[batch][row][col] = alpha * acc
    float* out; int ld, rows, cols; float alpha;
    __device__ EpiStoreF32(const GemmArgs& a, int batch, int) {
        out = reinterpret_cast<float*>(a.out) + batch * a.out_batch_stride;
        ld = a.ld_out; rows = a.rows_valid; cols = a.cols_valid; alpha = a.alpha;
    }
    __device__ void operator()(int row, int col0, const float* v) const {
        if (row >= rows || col0 >= cols) return;
        float* p = out + static_cast<long long>(row) * ld + col0;
        if (col0 + 16 <= cols && (ld & 3) == 0) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
                reinterpret_cast<float4*>(p)[i] = make_float4(alpha * v[4 * i], alpha * v[4 * i + 1], alpha * v[4 * i + 2], alpha * v[4 * i + 3]);
        } else {
            for (int i = 0; i < 16 && col0 + i < cols; ++i) p[i] = alpha * v[i];
        }
    }
};

// split-K partial of slice z = batch * n_splits + split, stored (not added): out[z][row][col] = acc.  The slices are summed
// in a fixed order by splitk_reduce_kernel (gemm_ops.cu), so the result does not depend on the order CTAs finish in
// (fp32 atomicAdd made the pooled Gram - and every eigenvector downstream - differ from launch to launch).
struct EpiStoreSplitK {
    float* out; float* csum; int ld, rows, cols;
    __device__ EpiStoreSplitK(const GemmArgs& a, int, int z) {
        out = reinterpret_cast<float*>(a.out) + z * a.out_batch_stride; ld = a.ld_out; rows = a.rows_valid; cols = a.cols_valid;
        csum = a.aux0 ? reinterpret_cast<float*>(const_cast<void*>(a.aux0)) + static_cast<long long>(z) * a.rows_valid : nullptr;
    }
    // COLSUM configurations: this slice's column sum of A's column `row` (aux0 = [slices][rows] partials, summed in slice order)
    __device__ void colsum(int row, float v) const { if (csum && row < rows) csum[row] = v; }
    __device__ void operator()(int row, int col0, const float* v) const {
        if (row >= rows || col0 >= cols) return;
        float* p = out + static_cast<long long>(row) * ld + col0;
        if (col0 + 16 <= cols && (ld & 3) == 0) {
#pragma unroll
            for (int i = 0; i < 4; ++i) reinterpret_cast<float4*>(p)[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
        } else {
            for (int i = 0; i < 16 && col0 + i < cols; ++i) p[i] = v[i];
        }
    }
};

struct EpiAtomicAddF32 {                  // split-K partial: out[row][col] += acc   (out pre-zeroed; self test only)
    float* out; int ld, rows, cols;
    __device__ EpiAtomicAddF32(const GemmArgs& a, int batch, int) {
        out = reinterpret_cast<float*>(a.out) + batch * a.out_batch_stride; ld = a.ld_out; rows = a.rows_valid; cols = a.cols_valid;
    }
    __device__ void operator()(int row, int col0, const float* v) const {
        if (row >= rows) return;
        float* p = out + static_cast<long long>(row) * ld + col0;
        for (int i = 0; i < 16 && col0 + i < cols; ++i) atomicAdd(p + i, v[i]);
    }
};

// student_grad: out[row][col] = alpha * gdir[row][col] + acc - corr[col]
//   aux0 = gdir fp32 [rows][cols] (direct-path gradient, unscaled), aux1 = corr fp32 [cols] (= mu^T Gamma)
//   out dtype: beta == 0 -> fp32, beta == 1 -> bf16
struct EpiStudentGrad {
    void* out; const float* gdir; const float* corr; int ld, rows, cols, gap_period, gap_valid; float alpha; bool bf16_out;
    __device__ EpiStudentGrad(const GemmArgs& g, int, int) {
        out = g.out; gdir = reinterpret_cast<const float*>(g.aux0); corr = reinterpret_cast<const float*>(g.aux1);
        ld = g.ld_out; rows = g.rows_valid; cols = g.cols_valid; bf16_out = g.beta != 0.f;
        gap_period = g.gap_period; gap_valid = g.gap_valid;
        alpha = g.alpha * (g.aux2 ? *reinterpret_cast<const float*>(g.aux2) : 1.f);
    }
    __device__ void operator()(int row_in, int col0, const float* v) const {
        if (row_in >= rows || col0 >= cols) return;
        int row = row_in;
        if (gap_period) {                  // input rows are the CLS-stripped view of a [B][N+1][D] buffer; the gradient is dense [B][N][D]
            const int b = row_in / gap_period, n = row_in - b * gap_period;
            if (n >= gap_valid) return;
            row = b * gap_valid + n;
        }
        const long long off = static_cast<long long>(row) * ld + col0;
        float r[16];
        const float* gp = gdir + static_cast<long long>(row) * cols + col0;
        if (col0 + 16 <= cols && (cols & 3) == 0) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float4 g4 = __ldg(reinterpret_cast<const float4*>(gp) + i);
                const float4 c4 = __ldg(reinterpret_cast<const float4*>(corr + col0) + i);
                r[4 * i] = alpha * g4.x + v[4 * i] - c4.x;         r[4 * i + 1] = alpha * g4.y + v[4 * i + 1] - c4.y;
                r[4 * i + 2] = alpha * g4.z + v[4 * i + 2] - c4.z; r[4 * i + 3] = alpha * g4.w + v[4 * i + 3] - c4.w;
            }
            if (bf16_out) {
                __nv_bfloat16* p = reinterpret_cast<__nv_bfloat16*>(out) + off;
                uint4 w0, w1;
                w0.x = pack_bf16x2(r[0], r[1]);   w0.y = pack_bf16x2(r[2], r[3]);   w0.z = pack_bf16x2(r[4], r[5]);   w0.w = pack_bf16x2(r[6], r[7]);
                w1.x = pack_bf16x2(r[8], r[9]);   w1.y = pack_bf16x2(r[10], r[11]); w1.z = pack_bf16x2(r[12], r[13]); w1.w = pack_bf16x2(r[14], r[15]);
                reinterpret_cast<uint4*>(p)[0] = w0;
                reinterpret_cast<uint4*>(p)[1] = w1;
            } else {
                float* p = reinterpret_cast<float*>(out) + off;
#pragma unroll
                for (int i = 0; i < 4; ++i) reinterpret_cast<float4*>(p)[i] = make_float4(r[4 * i], r[4 * i + 1], r[4 * i + 2], r[4 * i + 3]);
            }
            return;
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) r[i] = 0.f;
        for (int i = 0; i < 16 && col0 + i < cols; ++i) r[i] = alpha * gp[i] + v[i] - corr[col0 + i];
        if (bf16_out) {
            __nv_bfloat16* p = reinterpret_cast<__nv_bfloat16*>(out) + off;
            for (int i = 0; i < 16 && col0 + i < cols; ++i) p[i] = __float2bfloat16(r[i]);
        } else {
            float* p = reinterpret_cast<float*>(out) + off;
            for (int i = 0; i < 16 && col0 + i < cols; ++i) p[i] = r[i];
        }
    }
};

}  // namespace basd
