// Persistent batched small-matrix tcgen05 GEMM with run-time tile sizes, for the Newton-Schulz polar iteration of
// the Procrustes core (polar.cu).  A launch computes, for every problem z of a batch,
//     out[z] (m_rows x n_cols)  =  A[z] (m_rows x K)  *  B[z] (n_cols x K)^T
// on bf16 "split" operand pairs (hi, lo = bf16(x - hi)): the three MMAs hi*hi + hi*lo + lo*hi accumulate into the
// same TMEM tile and give fp32-class products (relative error ~2^-17) at bf16 tensor-core rate.
//   A : K-major ([m_rows][K]), loaded as 64-row TMA boxes, SWIZZLE_128B
//   B : K-major ([n_cols][K]) or MN-major ([K][n_cols]: the same buffer used transposed)
// Global layout of every split matrix is COLUMN-BLOCK TILED: [problem][col / 64][row][col % 64], so that each TMA box
// (rows x 64 columns) is one contiguous run of HBM (row-major storage with a 400-byte pitch measured 37 % of the
// copy bandwidth: every 128-byte box row opened its own DRAM page).
// Work item = (problem, 128-row tile, column tile of at most 256 columns) of the output - any m_rows, n_cols, K.
// One CTA per SM loops over its items; the shared-memory operand
// ring and two TMEM accumulator buffers are carried across items, so the TMA loads and MMAs of item i+1 overlap the
// epilogue of item i.  Warp 0 = TMA producer, warp 1 = MMA issuer, warps 2-5 = epilogue (one TMEM lane quadrant each).
// Epilogues only store (no global reads on the critical path) except the one-off Frobenius trace of step 0; the split
// outputs go through a 128B-swizzled shared-memory staging tile per warp and leave as TMA tensor stores (per-lane
// 16-byte stores of one row each saturated the L1TEX->XBAR request path: 32 requests per instruction; coalesced
// 512-byte-per-instruction stores out of the same staging tile measured the same as the TMA stores).
#pragma once
#include "ptx.cuh"

namespace basd {

constexpr int PG_THREADS = 192;
constexpr int PG_BK = 64;

enum PolarEpi : int {
    PG_EPI_SPLIT = 0,       // out = split(scale * acc + aux_scale * aux + diag_add * I); optional trace
    PG_EPI_F32 = 2,         // out_f32 = acc
    PG_EPI_THETA = 3,       // out = split(2 (diag(a) - q acc q^T - a a^T)), ROW-MAJOR [m_rows][ld_out]   (SURVEY.md B.1, teacher side)
    PG_EPI_ROWMAJOR = 4,    // out = bf16(scale * acc) or its split pair (out_lo != null), ROW-MAJOR [m_rows][ld_out]
    PG_EPI_SGRAD = 5,       // out = bf16(alpha * gdir + acc - corr[col]), ROW-MAJOR [m_rows][n_cols]   (student gradient, SURVEY.md B.5)
};

struct PolarGemmMaps {
    CUtensorMap a[2];
    CUtensorMap b[2];
    CUtensorMap o[4];                // SPLIT: out hi, out lo (TMA stores), aux hi, aux lo (TMA loads); box = 32 rows x 64 columns
};
// A_TABLE instantiations: the A operand of problem z is its own allocation with its own tensor map (the teacher layers of the
// projection are separate tensors); only those instantiations carry the table in their kernel parameters.
constexpr int PG_MAX_A_TABLE = 16;
struct PolarGemmMapsT : PolarGemmMaps {
    CUtensorMap a_tab[PG_MAX_A_TABLE];
};

struct PolarGemmArgs {
    int m_rows, n_cols, k_total;     // valid sizes
    int k_override;                  // > 0: contract over the first k_override columns of A / B only
    int n_override;                  // > 0: only the first n_override output columns (rows of B / columns of an MN-major B) exist
    int n_mt;                        // 128-row tiles per problem
    int n_nt;                        // column tiles per problem (bn_mma columns each; bn_mma is a multiple of 64 when n_nt > 1)
    int n_items;                     // batches * n_mt * n_nt
    int bn_mma;                      // UMMA N = columns per tile (multiple of 16; >= n_cols when n_nt == 1)
    int b_groups;                    // MN-major B: 64-column groups loaded per k-block
    int stages;
    int epi;
    // primary output (split pair, per-problem stride in elements)
    __nv_bfloat16* out_hi; __nv_bfloat16* out_lo; long long out_stride; int ld_out;   // tiled (SPLIT) or row-major with ld_out (THETA)
    const float* norm2;              // if non-null r = 1 / sum(norm2[z][0 .. fro_slots)), else r = 1
    int fro_slots;                   // partial-trace slots per problem (>= 4 n_mt n_nt of the launch that writes `trace`)
    float scale_c, scale_p;          // scale = scale_c * r^scale_p
    float diag_add;
    // auxiliary split matrix laid out like the output, added in the epilogue: out += aux_c * r^aux_p * aux (TMA-loaded)
    int aux_mode; float aux_c, aux_p;
    int a_alias_b;                   // A == B (K-major, same matrix): the A tile is read out of the B tile, no A loads
    int reverse, n_batches;          // reverse: walk the problems last-to-first (what the previous launch wrote last is still in L2)
    float* trace;                    // if non-null: trace[z][(mt n_nt + nt) 4 + warp] = this warp's share of sum(diag(acc)) (stored, not
                                     // added: the consumer sums the slots in order, so the norm is bitwise repeatable)
    float* resid;                    // aux epilogue only: resid[z][(mt n_nt + nt) 4 + warp] = sum (aux - I)^2 over this warp's part of the tile
    const __nv_bfloat16* aux_hi; const __nv_bfloat16* aux_lo;
    float* out_f32; long long out_f32_stride; int ld_f32;
    const float* vec_a;              // THETA: importance a [z][m_rows]
    // operands that are NOT column-block tiled (3-D tensor maps over row-major storage, 64 x 64 boxes):
    int a_rm;                        // A: row-major [z][m_rows][K]                 (K-major operand)
    int b_rm;                        // B: row-major [z][K][n_cols] (MN-major operand) or [z][n_cols][K] (K-major operand)
    int a_single;                    // A is one exact bf16 buffer (no lo half): terms A * B_hi + A * B_lo
    // SGRAD: direct-path gradient gdir fp32 [m_rows][n_cols], centring correction corr fp32 [n_cols], alpha = sg_alpha * *sg_scale (if non-null)
    const float* sg_gdir; const float* sg_corr; const float* sg_scale; float sg_alpha;
    int b_shared;                    // row-major K-major B: one matrix for every problem (batch coordinate 0)
    // ROWMAJOR: rows r with r % gap_period >= gap_valid are written as zeros (the CLS rows between the samples of a [:,1:,:] view
    // read as one dense matrix, umma_gemm.cuh GemmArgs::gap_period); 0 = no gaps
    int gap_period, gap_valid;
};

// 16 fp32 values -> bf16 hi / lo halves of staging row `row` (32 rows x 128 B, SWIZZLE_128B: 16-byte chunk j of row r
// lives at chunk position j ^ (r & 7)); chunk0 = first of the two 16-byte chunks the 16 columns occupy.
// Packed conversions (two values per cvt) and st.shared with 32-bit addresses: the epilogue runs one warp per scheduler,
// so its cost is its instruction count.
__device__ __forceinline__ void st_shared_v4(uint32_t saddr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void pg_stage_split16(uint32_t stg_hi, uint32_t stg_lo, int row, int chunk0, const float* v) {
    uint32_t hw[8], lw[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const __nv_bfloat162 hv = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
        const float2 hf = __bfloat1622float2(hv);
        const __nv_bfloat162 lv = __floats2bfloat162_rn(v[2 * i] - hf.x, v[2 * i + 1] - hf.y);
        hw[i] = *reinterpret_cast<const uint32_t*>(&hv);
        lw[i] = *reinterpret_cast<const uint32_t*>(&lv);
    }
    const uint32_t base = row * 128, p0 = base + ((chunk0 ^ (row & 7)) << 4), p1 = base + (((chunk0 + 1) ^ (row & 7)) << 4);
    st_shared_v4(stg_hi + p0, hw[0], hw[1], hw[2], hw[3]);
    st_shared_v4(stg_hi + p1, hw[4], hw[5], hw[6], hw[7]);
    st_shared_v4(stg_lo + p0, lw[0], lw[1], lw[2], lw[3]);
    st_shared_v4(stg_lo + p1, lw[4], lw[5], lw[6], lw[7]);
}
// 16 fp32 values -> staging row `row` of a 32 rows x 32 fp32 tile (128-byte rows, SWIZZLE_128B); chunk0 = first of the four
// 16-byte chunks they occupy
__device__ __forceinline__ void pg_stage_f32x16(uint32_t stg, int row, int chunk0, const float* v) {
    const uint32_t base = stg + row * 128;
#pragma unroll
    for (int i = 0; i < 4; ++i)
        st_shared_v4(base + (((chunk0 + i) ^ (row & 7)) << 4), __float_as_uint(v[4 * i]), __float_as_uint(v[4 * i + 1]),
                     __float_as_uint(v[4 * i + 2]), __float_as_uint(v[4 * i + 3]));
}
__device__ __forceinline__ void pg_stage_zero16(uint32_t stg_hi, uint32_t stg_lo, int row, int chunk0) {
    const uint32_t base = row * 128, p0 = base + ((chunk0 ^ (row & 7)) << 4), p1 = base + (((chunk0 + 1) ^ (row & 7)) << 4);
    st_shared_v4(stg_hi + p0, 0u, 0u, 0u, 0u);
    st_shared_v4(stg_hi + p1, 0u, 0u, 0u, 0u);
    st_shared_v4(stg_lo + p0, 0u, 0u, 0u, 0u);
    st_shared_v4(stg_lo + p1, 0u, 0u, 0u, 0u);
}
// inverse of pg_stage_split16: 16 values hi + lo of a TMA-loaded (swizzled) 32 x 64 tile
__device__ __forceinline__ void pg_read_split16(const uint8_t* t_hi, const uint8_t* t_lo, int row, int chunk0, float* x) {
    const int p0 = (chunk0 ^ (row & 7)) * 16, p1 = ((chunk0 + 1) ^ (row & 7)) * 16;
    const uint4 h0 = *reinterpret_cast<const uint4*>(t_hi + row * 128 + p0), h1 = *reinterpret_cast<const uint4*>(t_hi + row * 128 + p1);
    const uint4 l0 = *reinterpret_cast<const uint4*>(t_lo + row * 128 + p0), l1 = *reinterpret_cast<const uint4*>(t_lo + row * 128 + p1);
    const __nv_bfloat162* a0 = reinterpret_cast<const __nv_bfloat162*>(&h0);
    const __nv_bfloat162* a1 = reinterpret_cast<const __nv_bfloat162*>(&h1);
    const __nv_bfloat162* b0 = reinterpret_cast<const __nv_bfloat162*>(&l0);
    const __nv_bfloat162* b1 = reinterpret_cast<const __nv_bfloat162*>(&l1);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 u0 = __bfloat1622float2(a0[i]), w0 = __bfloat1622float2(b0[i]);
        const float2 u1 = __bfloat1622float2(a1[i]), w1 = __bfloat1622float2(b1[i]);
        x[2 * i] = u0.x + w0.x; x[2 * i + 1] = u0.y + w0.y;
        x[8 + 2 * i] = u1.x + w1.x; x[8 + 2 * i + 1] = u1.y + w1.y;
    }
}
// work item w -> (problem z, row tile mt, column tile nt); the tiles of one problem are consecutive (operands stay in L2)
struct PgItem { int z, mt, nt; };
__device__ __forceinline__ PgItem pg_item(const PolarGemmArgs& a, int w) {
    const int per = a.n_mt * a.n_nt;
    const int zi = w / per, r = w - zi * per;
    PgItem it;
    it.z = a.reverse ? a.n_batches - 1 - zi : zi;
    it.mt = r / a.n_nt;
    it.nt = r - it.mt * a.n_nt;
    return it;
}
// rows of A loaded for row tile mt (a multiple of 64, at most 128)
__device__ __forceinline__ int pg_a_rows(const PolarGemmArgs& a, int mt) {
    const int left = a.m_rows - mt * 128;
    return left >= 128 ? 128 : (left + 63) & ~63;
}
// KIND specialises the epilogue at compile time (one compact code path per instantiation: with every variant in one
// body the epilogue was ~3900 SASS instructions of mostly-skipped branches executed by a single warp per scheduler):
//   0 = SPLIT (scale, diagonal, optional trace of the diagonal)   1 = SPLIT + auxiliary tile   2 = THETA   3 = F32
//   4 = ROWMAJOR (scale; one bf16 or a split pair, row-major)   5 = SGRAD (direct gradient + product - correction, bf16 row-major)
//   6 = F32 through the staging tiles: the warp's two 4 KB tiles hold 32 rows x 32 fp32 columns each and leave as TMA stores
//       (maps.o[0] = fp32 map of the row-major output; needs a 16-byte row pitch).  The per-lane row stores of kind 3 (32 rows x
//       16 bytes per instruction) cost ~20 k cycles per 128 x 192 item - more than the item's MMAs.
template <bool A_TABLE> struct PgMapsOf { using type = PolarGemmMaps; };
template <> struct PgMapsOf<true> { using type = PolarGemmMapsT; };
template <bool B_MN, int KIND, bool A_TABLE = false>
__global__ void __launch_bounds__(PG_THREADS, 1)
polar_gemm_kernel(const __grid_constant__ typename PgMapsOf<A_TABLE>::type maps, const PolarGemmArgs args) {
    constexpr bool kStaged = KIND != 3, kTheta = KIND == 2, kAux = KIND == 1, kSgrad = KIND == 5, kF32Staged = KIND == 6;
    constexpr bool kRowMajor = KIND == 4 || kSgrad || kF32Staged;
    extern __shared__ uint8_t pg_smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(pg_smem_raw) + 1023) & ~uintptr_t(1023));
    const int kABytes = args.a_alias_b ? 0 : 128 * 128;    // one 128-row A tile per operand buffer (none when aliased)
    const int b_bytes = B_MN ? args.b_groups * 8192 : args.bn_mma * 128;
    const int a_bufs = args.a_single ? 1 : 2;
    const int stage_bytes = a_bufs * kABytes + 2 * b_bytes;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + args.stages * stage_bytes);
    uint64_t* empty_bar = full_bar + args.stages;
    uint64_t* tmem_full_bar = empty_bar + args.stages;         // [2]
    uint64_t* tmem_empty_bar = tmem_full_bar + 2;              // [2]
    uint64_t* aux_bar = tmem_empty_bar + 2;                    // [4] one per epilogue warp
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(aux_bar + 4);
    uint8_t* staging = smem + args.stages * stage_bytes + 1024;          // 4 warps x (hi 4 KB + lo 4 KB), 1024-aligned
    uint8_t* aux_staging = staging + 4 * 8192;                           // [4 warps][col blocks][hi 4 KB + lo 4 KB], only with aux_mode

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_kb = (args.k_total + PG_BK - 1) / PG_BK;

    if (threadIdx.x == 0) {
        for (int s = 0; s < args.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full_bar[i], 1); mbar_init(&tmem_empty_bar[i], 4); }
        for (int i = 0; i < 4; ++i) mbar_init(&aux_bar[i], 1);
        fence_mbar_init();
        if constexpr (!A_TABLE) { tma_prefetch_desc(&maps.a[0]); tma_prefetch_desc(&maps.a[1]); }
        tma_prefetch_desc(&maps.b[0]); tma_prefetch_desc(&maps.b[1]);
        if (kStaged) { tma_prefetch_desc(&maps.o[0]); if (!kF32Staged) tma_prefetch_desc(&maps.o[1]); }
    }
    uint32_t tmem_cols = 32;
    while (tmem_cols < static_cast<uint32_t>(2 * args.bn_mma)) tmem_cols <<= 1;
    if (warp == 1) tmem_alloc(tmem_slot, tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer
        if (lane == 0) {
            int it = 0;
            for (int w = blockIdx.x; w < args.n_items; w += gridDim.x) {
                const PgItem itm = pg_item(args, w);
                const int mt = itm.mt, z = itm.z;
                const int a_rows = pg_a_rows(args, mt);
                const uint32_t tx = (args.a_alias_b ? 0 : a_bufs * a_rows * 128) + 2 * b_bytes;
                for (int kb = 0; kb < n_kb; ++kb, ++it) {
                    const int s = it % args.stages;
                    const uint32_t ph = (it / args.stages) & 1;
                    mbar_wait(&empty_bar[s], ph ^ 1);
                    mbar_arrive_expect_tx(&full_bar[s], tx);
                    uint8_t* st = smem + s * stage_bytes;
                    for (int i = 0; i < a_bufs && !args.a_alias_b; ++i) {
                        uint8_t* dst = st + i * kABytes;
                        for (int g = 0; g < a_rows / 64; ++g) {
                            if constexpr (A_TABLE) tma_load_3d(dst + g * 8192, &maps.a_tab[z], &full_bar[s], kb * PG_BK, mt * 128 + g * 64, 0);
                            else if (args.a_rm) tma_load_3d(dst + g * 8192, &maps.a[i], &full_bar[s], kb * PG_BK, mt * 128 + g * 64, z);
                            else tma_load_4d(dst + g * 8192, &maps.a[i], &full_bar[s], 0, mt * 128 + g * 64, kb, z);
                        }
                    }
                    for (int i = 0; i < 2; ++i) {
                        uint8_t* dst = st + a_bufs * kABytes + i * b_bytes;
                        if (B_MN) {
                            for (int g = 0; g < args.b_groups; ++g) {
                                if (args.b_rm) tma_load_3d(dst + g * 8192, &maps.b[i], &full_bar[s], (itm.nt * args.b_groups + g) * 64, kb * PG_BK, z);
                                else tma_load_4d(dst + g * 8192, &maps.b[i], &full_bar[s], 0, kb * PG_BK, itm.nt * args.b_groups + g, z);
                            }
                        } else if (args.b_rm) {
                            tma_load_3d(dst, &maps.b[i], &full_bar[s], kb * PG_BK, itm.nt * args.bn_mma, args.b_shared ? 0 : z);
                        } else {
                            tma_load_4d(dst, &maps.b[i], &full_bar[s], 0, itm.nt * args.bn_mma, kb, z);
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer
        const uint32_t idesc = umma_idesc_bf16(128, args.bn_mma, false, B_MN);
        int it = 0, item = 0;
        for (int w = blockIdx.x; w < args.n_items; w += gridDim.x, ++item) {
            const int acc = item & 1;
            const uint32_t acc_ph = (item >> 1) & 1;
            const int mt_mma = pg_item(args, w).mt;
            mbar_wait(&tmem_empty_bar[acc], acc_ph ^ 1);           // epilogue has drained this accumulator
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + acc * args.bn_mma;
            for (int kb = 0; kb < n_kb; ++kb, ++it) {
                const int s = it % args.stages;
                const uint32_t ph = (it / args.stages) & 1;
                mbar_wait(&full_bar[s], ph);
                tc_fence_after();
                if (lane == 0) {
                    const uint32_t st = smem_u32(smem + s * stage_bytes);
                    int ksteps = (args.k_total - kb * PG_BK + 15) / 16;
                    if (ksteps > 4) ksteps = 4;
#pragma unroll
                    for (int t = 0; t < 3; ++t) {                // hi*hi, hi*lo, lo*hi
                        if (t == 2 && args.a_single) break;      // exact bf16 A: no lo*hi term
                        const uint32_t b_base = st + a_bufs * kABytes + (t == 1 ? b_bytes : 0);
                        // aliased: rows mt*128.. of the (hi or lo) B tile are the A tile
                        const uint32_t a_base = args.a_alias_b ? st + (t == 2 ? b_bytes : 0) + mt_mma * 16384 : st + (t == 2 ? kABytes : 0);
                        for (int ks = 0; ks < ksteps; ++ks) {
                            const uint64_t adesc = umma_smem_desc(a_base + ks * 32, 16, 1024);
                            const uint64_t bdesc = B_MN ? umma_smem_desc(b_base + ks * 2048, 8192, 1024)
                                                        : umma_smem_desc(b_base + ks * 32, 16, 1024);
                            umma_bf16(d_tmem, adesc, bdesc, idesc, (kb > 0 || t > 0 || ks > 0) ? 1u : 0u);
                        }
                    }
                    umma_commit(&empty_bar[s]);
                    if (kb == n_kb - 1) umma_commit(&tmem_full_bar[acc]);
                }
                __syncwarp();
            }
        }
    } else {
        // ------------------------------------------------------------------ epilogue (4 warps = 128 TMEM lanes)
        const int q = warp & 3;
        int item = 0;
        uint32_t aux_phase = 0;
        for (int w = blockIdx.x; w < args.n_items; w += gridDim.x, ++item) {
            const PgItem itm = pg_item(args, w);
            const int mt = itm.mt, z = itm.z;
            const int c0 = itm.nt * args.bn_mma;                              // first output column of this tile
            const int cb0 = c0 >> 6;                                          // ... as a 64-column block index
            const int acc = item & 1;
            const uint32_t acc_ph = (item >> 1) & 1;
            const bool warp_rows_ok = mt * 128 + q * 32 < args.m_rows;       // uniform: this warp owns at least one valid row
            const int n_cb_aux = (args.bn_mma + 63) / 64;
            uint8_t* aux_base = aux_staging + (warp - 2) * n_cb_aux * 8192;
            const bool use_aux = kAux && warp_rows_ok;
            if (use_aux && lane == 0) {                                    // the whole auxiliary tile of this item, hidden behind the main loop
                mbar_arrive_expect_tx(&aux_bar[warp - 2], n_cb_aux * 8192);
                for (int cb = 0; cb < n_cb_aux; ++cb) {
                    tma_load_4d(aux_base + cb * 8192, &maps.o[2], &aux_bar[warp - 2], 0, mt * 128 + q * 32, cb0 + cb, z);
                    tma_load_4d(aux_base + cb * 8192 + 4096, &maps.o[3], &aux_bar[warp - 2], 0, mt * 128 + q * 32, cb0 + cb, z);
                }
            }
            // SGRAD: the direct-path gradient tile of this warp (32 rows x 64 fp32 columns per block: two 32 x 32 SWIZZLE_128B boxes)
            // arrives by TMA - block 0 behind the main loop, block b + 1 while block b is converted.  (Read straight from global
            // memory one row per lane, every 128-bit load touched 32 different lines: the load pipe, not DRAM, set the pace - 29 k
            // cycles per item against 8 k of main loop.)
            uint8_t* sg_tile = aux_staging + (warp - 2) * 8192;
            if (kSgrad && warp_rows_ok && lane == 0) {
                mbar_arrive_expect_tx(&aux_bar[warp - 2], 8192);
                tma_load_3d(sg_tile, &maps.o[2], &aux_bar[warp - 2], c0, mt * 128 + q * 32, z);
                tma_load_3d(sg_tile + 4096, &maps.o[2], &aux_bar[warp - 2], c0 + 32, mt * 128 + q * 32, z);
            }
            mbar_wait(&tmem_full_bar[acc], acc_ph);
            tc_fence_after();
            const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * args.bn_mma;
            const int row = mt * 128 + q * 32 + lane;
            const bool row_ok = row < args.m_rows;
            const bool gap_row = KIND == 4 && args.gap_period > 0 && row % args.gap_period >= args.gap_valid;
            float r = 1.f;
            if (args.norm2) {
                float tsum = 0.f;
                for (int sl = 0; sl < args.fro_slots; ++sl) tsum += args.norm2[static_cast<long long>(z) * args.fro_slots + sl];
                r = tsum > 0.f ? 1.f / tsum : 0.f;        // C == 0 (constant tokens): r = 0, the nuclear norm is 0, gradients stay finite
            }
            const float scale = args.scale_c * (args.scale_p == 0.f ? 1.f : powf(r, args.scale_p));
            const float sg_alpha = kSgrad ? args.sg_alpha * (args.sg_scale ? *args.sg_scale : 1.f) : 0.f;
            const float aux_scale = args.aux_c * (args.aux_p == 0.f ? 1.f : powf(r, args.aux_p));
            float a_row = 0.f, q_row = 0.f;
            // THETA: a and sqrt(a) of this tile's columns, once per item into the warp's strip of shared memory (the per-element
            // global load + IEEE sqrtf this replaces made the launch three times as long as a plain product: 0.31 ms at cfg2)
            float* th_a = reinterpret_cast<float*>(aux_staging) + (warp - 2) * 512;
            float* th_q = th_a + 256;
            if (kTheta) {
                if (row_ok) {
                    a_row = args.vec_a[static_cast<long long>(z) * args.m_rows + row];
                    q_row = sqrtf(a_row);
                }
                const float* avz = args.vec_a + static_cast<long long>(z) * args.m_rows;
                for (int cl = lane; cl < args.bn_mma; cl += 32) {
                    const float ac = c0 + cl < args.n_cols ? avz[c0 + cl] : 0.f;
                    th_a[cl] = ac;
                    th_q[cl] = sqrtf(ac);
                }
                __syncwarp();
            }
            float tr_part = 0.f, rs_part = 0.f;
            if constexpr (kStaged) {
                constexpr bool theta = kTheta;
                // convert into the warp's swizzled staging tile; every 64-column block leaves as one TMA store per half
                uint8_t* stg_hi = staging + (warp - 2) * 8192;
                uint8_t* stg_lo = stg_hi + 4096;
                const uint32_t stg_hi_s = smem_u32(stg_hi), stg_lo_s = smem_u32(stg_lo);
                const bool diag_work = args.diag_add != 0.f;           // uniform: most launches have no diagonal term
                const int n_cb = (args.bn_mma + 63) / 64;
                if (use_aux) {
                    mbar_wait(&aux_bar[warp - 2], aux_phase);
                    aux_phase ^= 1;
                }
                for (int cbk = 0; cbk < n_cb; ++cbk) {
                    if (c0 + cbk * 64 >= ((args.n_cols + 63) & ~63)) break;    // column blocks past the matrix (last tile)
                    if (kRowMajor && c0 + cbk * 64 >= args.n_cols) break;
                    const uint8_t* aux_hi_s = aux_base + cbk * 8192;
                    const uint8_t* aux_lo_s = aux_hi_s + 4096;
                    // whole 64-column block in one tcgen05.ld (the last block of a 208-wide tile has 16 columns)
                    float vb[64];
                    const int cols_here = min(64, args.bn_mma - cbk * 64);
                    float4 sg_g[kSgrad ? 16 : 1];
                    if constexpr (kSgrad) {
                        if (warp_rows_ok) {
                            mbar_wait(&aux_bar[warp - 2], aux_phase);
                            aux_phase ^= 1;
#pragma unroll
                            for (int j = 0; j < 16; ++j)      // chunk j of this lane's row: box j / 8, 16-byte chunk (j % 8) ^ (row % 8) of its 128-byte row
                                sg_g[j] = *reinterpret_cast<const float4*>(sg_tile + (j >> 3) * 4096 + lane * 128 + (((j & 7) ^ (lane & 7)) << 4));
                            __syncwarp();                     // tile consumed by every lane: the next block may land on it
                            const int cn = c0 + (cbk + 1) * 64;
                            if (lane == 0 && cbk + 1 < n_cb && cn < args.n_cols) {
                                mbar_arrive_expect_tx(&aux_bar[warp - 2], 8192);
                                tma_load_3d(sg_tile, &maps.o[2], &aux_bar[warp - 2], cn, mt * 128 + q * 32, z);
                                tma_load_3d(sg_tile + 4096, &maps.o[2], &aux_bar[warp - 2], cn + 32, mt * 128 + q * 32, z);
                            }
                        }
                    }
                    if (cols_here == 64) {
                        tmem_ld64(t_addr + cbk * 64, vb);
                    } else {
#pragma unroll
                        for (int jc = 0; jc < 4; ++jc) {
                            if (jc * 16 < cols_here) tmem_ld16(t_addr + cbk * 64 + jc * 16, vb + jc * 16);
                        }
                    }
#pragma unroll
                    for (int jc = 0; jc < 4; ++jc) {
                        const int c = c0 + cbk * 64 + jc * 16;                  // global column of v[0]
                        float* v = vb + jc * 16;
                        if constexpr (kF32Staged) {                             // plain fp32 result (scale_c == 1): columns 0-31 -> tile "hi", 32-63 -> tile "lo"
                            if (cbk * 64 + jc * 16 < args.bn_mma) pg_stage_f32x16(jc < 2 ? stg_hi_s : stg_lo_s, lane, (jc & 1) * 4, v);
                            continue;
                        }
                        if (cbk * 64 + jc * 16 < args.bn_mma) {
                            if (KIND == 0 && args.trace && row_ok) {
#pragma unroll
                                for (int i = 0; i < 16; ++i) tr_part += (c + i == row) ? v[i] : 0.f;
                            }
                            if constexpr (theta) {
#pragma unroll
                                for (int i = 0; i < 16; ++i) {
                                    const int cl = cbk * 64 + jc * 16 + i;          // column inside the tile (zero a / q past n_cols)
                                    float t = -q_row * v[i] * th_q[cl] - a_row * th_a[cl];
                                    if (c + i == row) t += a_row;
                                    v[i] = c + i < args.n_cols ? 2.f * t : 0.f;
                                }
                            } else if constexpr (kAux) {
                                float x[16];
                                pg_read_split16(aux_hi_s, aux_lo_s, lane, jc * 2, x);
                                if (args.resid && row_ok) {                     // last step: ||A - I||_F^2 (convergence evidence)
#pragma unroll
                                    for (int i = 0; i < 16; ++i) {
                                        const float dv = (c + i < args.n_cols) ? x[i] - ((c + i == row) ? 1.f : 0.f) : 0.f;
                                        rs_part = fmaf(dv, dv, rs_part);
                                    }
                                }
#pragma unroll
                                for (int i = 0; i < 16; ++i) v[i] = fmaf(aux_scale, x[i], scale * v[i]) + ((c + i == row) ? args.diag_add : 0.f);
                            } else if constexpr (kSgrad) {
                                if (row_ok && c < args.n_cols) {             // (n_cols is a multiple of 8; chunks are 16 wide)
                                    const float* cp = args.sg_corr + static_cast<long long>(z) * args.n_cols + c;
                                    const int nq = min(4, (args.n_cols - c) >> 2);
#pragma unroll
                                    for (int i4 = 0; i4 < 4; ++i4) {
                                        if (i4 < nq) {
                                            const float4 g4 = sg_g[jc * 4 + i4];
                                            const float4 c4 = __ldg(reinterpret_cast<const float4*>(cp) + i4);
                                            v[4 * i4] = sg_alpha * g4.x + v[4 * i4] - c4.x;         v[4 * i4 + 1] = sg_alpha * g4.y + v[4 * i4 + 1] - c4.y;
                                            v[4 * i4 + 2] = sg_alpha * g4.z + v[4 * i4 + 2] - c4.z; v[4 * i4 + 3] = sg_alpha * g4.w + v[4 * i4 + 3] - c4.w;
                                        }
                                    }
                                }
                            } else if (diag_work) {
#pragma unroll
                                for (int i = 0; i < 16; ++i) v[i] = scale * v[i] + ((c + i == row) ? args.diag_add : 0.f);
                            } else if (KIND == 4 && gap_row) {
#pragma unroll
                                for (int i = 0; i < 16; ++i) v[i] = 0.f;
                            } else {
#pragma unroll
                                for (int i = 0; i < 16; ++i) v[i] *= scale;
                            }
                            pg_stage_split16(stg_hi_s, stg_lo_s, lane, jc * 2, v);
                        } else {
                            pg_stage_zero16(stg_hi_s, stg_lo_s, lane, jc * 2);      // padding columns of the last block
                        }
                    }
                    fence_proxy_async_smem();
                    __syncwarp();                                               // staging complete; aux tile fully consumed
                    if (lane == 0 && warp_rows_ok) {
                        if constexpr (kF32Staged) {                             // two 32 x 32 fp32 boxes; columns past n_cols / rows past m_rows are clipped
                            tma_store_3d(&maps.o[0], stg_hi, c0 + cbk * 64, mt * 128 + q * 32, z);
                            if (c0 + cbk * 64 + 32 < args.n_cols && cbk * 64 + 32 < args.bn_mma)
                                tma_store_3d(&maps.o[0], stg_lo, c0 + cbk * 64 + 32, mt * 128 + q * 32, z);
                        } else if constexpr (theta) {                           // row-major output, columns past n_cols are clipped
                            tma_store_3d(&maps.o[0], stg_hi, c0 + cbk * 64, mt * 128 + q * 32, z);
                            tma_store_3d(&maps.o[1], stg_lo, c0 + cbk * 64, mt * 128 + q * 32, z);
                        } else if constexpr (kRowMajor) {
                            tma_store_3d(&maps.o[0], stg_hi, c0 + cbk * 64, mt * 128 + q * 32, z);
                            if (args.out_lo) tma_store_3d(&maps.o[1], stg_lo, c0 + cbk * 64, mt * 128 + q * 32, z);
                        } else {
                            tma_store_4d(&maps.o[0], stg_hi, 0, mt * 128 + q * 32, cb0 + cbk, z);
                            tma_store_4d(&maps.o[1], stg_lo, 0, mt * 128 + q * 32, cb0 + cbk, z);
                        }
                        tma_store_commit();
                        tma_store_wait_read();
                    }
                    __syncwarp();
                }
            } else {
                for (int cl = 0; cl < args.bn_mma; cl += 16) {
                    float v[16];
                    tmem_ld16(t_addr + cl, v);
                    const int c = c0 + cl;
                    if (!row_ok || c >= args.n_cols) continue;
                    const int nv = min(16, args.n_cols - c);
                    if (args.epi == PG_EPI_F32) {
                        float* p = args.out_f32 + z * args.out_f32_stride + static_cast<long long>(row) * args.ld_f32 + c;
                        if (nv == 16 && (args.ld_f32 & 3) == 0) {
#pragma unroll
                            for (int i = 0; i < 4; ++i)
                                reinterpret_cast<float4*>(p)[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
                        } else {
                            for (int i = 0; i < nv; ++i) p[i] = v[i];
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);
            if (args.trace) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) tr_part += __shfl_xor_sync(0xffffffffu, tr_part, o);
                if (lane == 0) args.trace[static_cast<long long>(z) * args.fro_slots + (mt * args.n_nt + itm.nt) * 4 + q] = tr_part;
            }
            if (kAux && args.resid) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) rs_part += __shfl_xor_sync(0xffffffffu, rs_part, o);
                if (lane == 0) args.resid[static_cast<long long>(z) * args.fro_slots + (mt * args.n_nt + itm.nt) * 4 + q] = rs_part;
            }
        }
        if (lane == 0) tma_store_wait_all();          // global writes of this CTA complete before it exits
    }
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, tmem_cols);
    }
}

}  // namespace basd
