// Fused G2 + G3 of a Newton-Schulz step (polar.cu):   A = T W^T   and   Bm = a I + b (rA) + c (rA)^2   in ONE kernel, A never
// leaving the SM.  The two-launch version wrote A (split pair) to global memory, read it back twice (operand + auxiliary
// tile) and paid a second launch; the polar launches sit at ~90 % of the chip's L2 throughput (DESIGN.md section 5), so
// the lever is L2 traffic per flop.
// One work item = one problem; a CTA (320 threads) keeps both 128-row tiles of A in TMEM (2 x bn columns):
//   phase 1   warp 0 streams T (A operand) and W (B operand) k-blocks through a 2-stage ring, warp 1 accumulates A;
//   copy      warps 2-9 (one per 32-row slab of a tile) read A from TMEM WITHOUT draining it, scale it by
//             s = sqrt(c r / |b|) and write it as a split bf16 pair in the canonical K-major SWIZZLE_128B operand layout
//             into the (now idle) ring memory; at step 0 they first reduce trace(A) = ||C||_F^2 -> r;
//   phase 2   warp 1 issues (-A~) A~ on top of the accumulator (negate-A bit of the instruction descriptor when b < 0,
//             A~ is both operands: the A tile is read out of the B tile), so TMEM holds  A - (c r / |b|) A^2 = A + (c r / b) A^2;
//   store     warps 2-9:  Bm = a I + (b r) acc  -> split pair -> SWIZZLE_64B staging (32 x 32) -> TMA store.
// The loads of the next problem start as soon as phase 2 has retired (they overlap the store phase); its MMAs wait for the
// accumulators to be drained.  Phase 2 cannot start before the WHOLE copy is written: its MMAs update every accumulator
// column, including the ones the copy still has to read.  Timeline of one problem on B200 (cfg2, cycles): phase 1 10-12 k
// (tensor bound), copy 3.8 k, phase 2 8 k (tensor bound), store 7.8 k, hand-overs 1-2 k.  Requires m = n = D_s <= 192 (the operand copy must fit the ring) - larger D_s keeps the
// two-launch path.
#pragma once
#include "polar_gemm.cuh"
#include "spectral.h"

namespace basd {

constexpr int PF_THREADS = 320;
constexpr int PF_STAGES = 2;

struct PolarFusedMaps {
    CUtensorMap t[2];                // T hi / lo   (A operand: 64-row x 64-column boxes)
    CUtensorMap w[2];                // W hi / lo   (B operand: bn-row x 64-column boxes)
    CUtensorMap o[2];                // Bm hi / lo  (stores: 32 rows x 32 columns, SWIZZLE_64B)
};

// 32 rows x 32 bf16 columns (64-byte rows), SWIZZLE_64B: 16-byte chunk c of row r sits at chunk c ^ ((r >> 1) & 3)
__device__ __forceinline__ void pf_stage_split16_sw64(uint32_t stg_hi, uint32_t stg_lo, int row, int chunk0, const float* v) {
    uint32_t hw[8], lw[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const __nv_bfloat162 hv = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
        const float2 hf = __bfloat1622float2(hv);
        const __nv_bfloat162 lv = __floats2bfloat162_rn(v[2 * i] - hf.x, v[2 * i + 1] - hf.y);
        hw[i] = *reinterpret_cast<const uint32_t*>(&hv);
        lw[i] = *reinterpret_cast<const uint32_t*>(&lv);
    }
    const uint32_t sw = (row >> 1) & 3, base = row * 64, p0 = base + ((chunk0 ^ sw) << 4), p1 = base + (((chunk0 + 1) ^ sw) << 4);
    st_shared_v4(stg_hi + p0, hw[0], hw[1], hw[2], hw[3]);
    st_shared_v4(stg_hi + p1, hw[4], hw[5], hw[6], hw[7]);
    st_shared_v4(stg_lo + p0, lw[0], lw[1], lw[2], lw[3]);
    st_shared_v4(stg_lo + p1, lw[4], lw[5], lw[6], lw[7]);
}
__device__ __forceinline__ void pf_stage_zero16_sw64(uint32_t stg_hi, uint32_t stg_lo, int row, int chunk0) {
    const uint32_t sw = (row >> 1) & 3, base = row * 64, p0 = base + ((chunk0 ^ sw) << 4), p1 = base + (((chunk0 + 1) ^ sw) << 4);
    st_shared_v4(stg_hi + p0, 0u, 0u, 0u, 0u);
    st_shared_v4(stg_hi + p1, 0u, 0u, 0u, 0u);
    st_shared_v4(stg_lo + p0, 0u, 0u, 0u, 0u);
    st_shared_v4(stg_lo + p1, 0u, 0u, 0u, 0u);
}

__global__ void __launch_bounds__(PF_THREADS, 1)
polar_fused_abm_kernel(const __grid_constant__ PolarFusedMaps maps, const PolarFusedArgs args) {
    extern __shared__ uint8_t pf_smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(pf_smem_raw) + 1023) & ~uintptr_t(1023));
    const int a_bytes = args.rows_ld * 128;                    // one half (hi or lo) of a T k-block
    const int b_bytes = args.bn * 128;                         // one half of a W k-block
    const int stage_bytes = 2 * a_bytes + 2 * b_bytes;
    const int ring_bytes = PF_STAGES * stage_bytes;
    const int n_kb = (args.k_total + 63) / 64;                 // phase 1 k-blocks
    const int n_kb2 = (args.n + 63) / 64;                      // phase 2 k-blocks = 64-column blocks of A
    const int blk_bytes = args.rows_ld * 128;                  // operand copy: [half][k-block][rows_ld rows x 128 B]
    const int half_bytes = n_kb2 * blk_bytes;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + ring_bytes);
    uint64_t* empty_bar = full_bar + PF_STAGES;
    uint64_t* acc1_bar = empty_bar + PF_STAGES;                // [2] row tile mt of A complete in TMEM
    uint64_t* copy_bar = acc1_bar + 2;                         // [4] 64-column block kb of the operand copy written (4 n_mt warps)
    uint64_t* acc2_bar = copy_bar + 4;                         // [2] row tile mt of A + (c r / b) A^2 complete in TMEM
    uint64_t* p2done_bar = acc2_bar + 2;                       // phase 2 retired: the ring memory is free again
    uint64_t* tmem_empty_bar = p2done_bar + 1;                 // [2] accumulator of row tile mt drained (its 4 warps)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);
    float* trace_s = reinterpret_cast<float*>(tmem_slot + 2);  // [2][8]: per item parity, one slot per epilogue warp
    uint8_t* staging = smem + ring_bytes + 1024;               // 8 warps x (hi 2 KB + lo 2 KB)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < PF_STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&acc1_bar[i], 1); mbar_init(&acc2_bar[i], 1); mbar_init(&tmem_empty_bar[i], 4); }
        mbar_init(p2done_bar, 1);
        for (int i = 0; i < 4; ++i) mbar_init(&copy_bar[i], 4 * args.n_mt);
        fence_mbar_init();
        tma_prefetch_desc(&maps.t[0]); tma_prefetch_desc(&maps.t[1]);
        tma_prefetch_desc(&maps.w[0]); tma_prefetch_desc(&maps.w[1]);
        tma_prefetch_desc(&maps.o[0]); tma_prefetch_desc(&maps.o[1]);
    }
    uint32_t tmem_cols = 32;
    while (tmem_cols < static_cast<uint32_t>(2 * args.bn)) tmem_cols <<= 1;
    if (warp == 1) tmem_alloc(tmem_slot, tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer
        if (lane == 0) {
            const uint32_t tx = stage_bytes;
            int it = 0, item = 0;
            for (int w = blockIdx.x; w < args.n_problems; w += gridDim.x, ++item) {
                const int z = args.reverse ? args.n_problems - 1 - w : w;
                if (item > 0) mbar_wait(p2done_bar, (item - 1) & 1);       // the operand copy of the previous problem is dead
                for (int kb = 0; kb < n_kb; ++kb, ++it) {
                    const int s = it % PF_STAGES;
                    const uint32_t ph = (it / PF_STAGES) & 1;
                    mbar_wait(&empty_bar[s], ph ^ 1);
                    mbar_arrive_expect_tx(&full_bar[s], tx);
                    uint8_t* st = smem + s * stage_bytes;
                    for (int i = 0; i < 2; ++i) {
                        for (int g = 0; g < args.rows_ld / 64; ++g)
                            tma_load_4d(st + i * a_bytes + g * 8192, &maps.t[i], &full_bar[s], 0, g * 64, kb, z);
                        tma_load_4d(st + 2 * a_bytes + i * b_bytes, &maps.w[i], &full_bar[s], 0, 0, kb, z);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer
        const uint32_t idesc1 = umma_idesc_bf16(128, args.bn, false, false);
        const uint32_t idesc2 = idesc1 | (args.cb < 0.f ? (1u << 13) : 0u);       // negate A:  acc -= A~ A~  when c r / b < 0
        int it = 0, item = 0;
        for (int w = blockIdx.x; w < args.n_problems; w += gridDim.x, ++item) {
            const uint32_t ph_item = item & 1;
            for (int kb = 0; kb < n_kb; ++kb, ++it) {             // phase 1: A = T W^T
                const int s = it % PF_STAGES;
                const uint32_t ph = (it / PF_STAGES) & 1;
                mbar_wait(&full_bar[s], ph);
                tc_fence_after();
                const uint32_t st = smem_u32(smem + s * stage_bytes);
                int ksteps = (args.k_total - kb * 64 + 15) / 16;
                if (ksteps > 4) ksteps = 4;
                for (int mt = 0; mt < args.n_mt; ++mt) {
                    if (kb == 0) {                                // the store phase of the previous problem has drained THIS tile's accumulator
                        mbar_wait(&tmem_empty_bar[mt], ph_item ^ 1);   // (tile 1 is still being stored while tile 0's first MMAs run)
                        tc_fence_after();
                    }
                    if (lane == 0) {
#pragma unroll
                        for (int t = 0; t < 3; ++t) {            // hi*hi, hi*lo, lo*hi
                            const uint32_t a_base = st + (t == 2 ? a_bytes : 0) + mt * 16384;
                            const uint32_t b_base = st + 2 * a_bytes + (t == 1 ? b_bytes : 0);
                            for (int ks = 0; ks < ksteps; ++ks)
                                umma_bf16(tmem_base + mt * args.bn, umma_smem_desc(a_base + ks * 32, 16, 1024),
                                          umma_smem_desc(b_base + ks * 32, 16, 1024), idesc1, (kb > 0 || t > 0 || ks > 0) ? 1u : 0u);
                        }
                        if (kb == n_kb - 1) umma_commit(&acc1_bar[mt]);       // tile 0's copy starts under tile 1's last MMAs
                    }
                    __syncwarp();
                }
                if (lane == 0) umma_commit(&empty_bar[s]);
                __syncwarp();
            }
            if (lane == 0) {                                      // phase 2: acc += (-A~) A~
                const uint32_t cp = smem_u32(smem);
                // every block of A~ must be in shared memory first: the MMAs overwrite the accumulator columns the copy
                // is still reading (generic-proxy writes, fenced by the writers)
                for (int kb = 0; kb < n_kb2; ++kb) mbar_wait(&copy_bar[kb], ph_item);
                tc_fence_after();
                // row tile by row tile (every operand is resident): tile 0 is stored while tile 1 is still being multiplied
                for (int mt = 0; mt < args.n_mt; ++mt) {
                    for (int kb = 0; kb < n_kb2; ++kb) {
                        int ksteps = (args.n - kb * 64 + 15) / 16;
                        if (ksteps > 4) ksteps = 4;
#pragma unroll
                        for (int t = 0; t < 3; ++t) {
                            const uint32_t b_base = cp + (t == 1 ? half_bytes : 0) + kb * blk_bytes;
                            const uint32_t a_base = cp + (t == 2 ? half_bytes : 0) + kb * blk_bytes + mt * 16384;
                            for (int ks = 0; ks < ksteps; ++ks)
                                umma_bf16(tmem_base + mt * args.bn, umma_smem_desc(a_base + ks * 32, 16, 1024),
                                          umma_smem_desc(b_base + ks * 32, 16, 1024), idesc2, 1u);
                        }
                    }
                    umma_commit(&acc2_bar[mt]);
                }
                umma_commit(p2done_bar);
            }
            __syncwarp();
        }
    } else if (((warp - 2) >> 2) < args.n_mt) {
        // ------------------------------------------------------------------ copy + store warps (4 per tile = 128 TMEM lanes)
        const int e = warp - 2, mt = e >> 2, q = warp & 3;
        const int row0 = mt * 128 + q * 32;
        const int row = row0 + lane;
        const bool warp_rows_ok = row0 < args.n;
        const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + mt * args.bn;
        const int n_epi_threads = 128 * args.n_mt;
        uint8_t* stg_hi = staging + e * 4096;
        uint8_t* stg_lo = stg_hi + 2048;
        const uint32_t stg_hi_s = smem_u32(stg_hi), stg_lo_s = smem_u32(stg_lo);
        int item = 0;
        for (int w = blockIdx.x; w < args.n_problems; w += gridDim.x, ++item) {
            const int z = args.reverse ? args.n_problems - 1 - w : w;
            const uint32_t ph_item = item & 1;
            mbar_wait(&acc1_bar[mt], ph_item);
            tc_fence_after();
            float r = 1.f;
            if (args.first) {                                     // trace(A) = ||C||_F^2 of this problem
                float tr = 0.f;
                if (warp_rows_ok) {
                    float d[32];
                    tmem_ld32(t_addr + row0, d);                  // columns row0 .. row0+31 of this warp's rows: the diagonal block
#pragma unroll
                    for (int i = 0; i < 32; ++i) tr += (i == lane && row < args.n) ? d[i] : 0.f;
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) tr += __shfl_xor_sync(0xffffffffu, tr, o);
                if (lane == 0) trace_s[ph_item * 8 + e] = tr;           // stored per warp, summed in order: bitwise repeatable
                asm volatile("bar.sync 2, %0;" ::"r"(n_epi_threads) : "memory");
                float trace = 0.f;
#pragma unroll
                for (int e2 = 0; e2 < 8; ++e2) trace += e2 * 32 < n_epi_threads ? trace_s[ph_item * 8 + e2] : 0.f;
                r = trace > 0.f ? 1.f / trace : 0.f;
                if (e == 0 && lane == 0) args.fro2[static_cast<long long>(z) * args.fro_slots] = trace;
            }
            // ---- copy: A~ = s A as a split pair, K-major SWIZZLE_128B operand layout [half][64-column block][row]
            const float s_copy = sqrtf(args.cc * r / fabsf(args.cb));
            float rs_part = 0.f;                                  // last step: this warp's share of ||A - I||_F^2
            for (int cbk = 0; cbk < n_kb2; ++cbk) {
                if (row0 < args.rows_ld) {
                    float vb[64];
                    const int cols_here = min(64, args.bn - cbk * 64);
                    if (cols_here == 64) {
                        tmem_ld64(t_addr + cbk * 64, vb);
                    } else {
#pragma unroll
                        for (int jc = 0; jc < 4; ++jc)
                            if (jc * 16 < cols_here) tmem_ld16(t_addr + cbk * 64 + jc * 16, vb + jc * 16);
                    }
                    const uint32_t dst_hi = smem_u32(smem + cbk * blk_bytes + row0 * 128), dst_lo = dst_hi + half_bytes;
#pragma unroll
                    for (int jc = 0; jc < 4; ++jc) {
                        float* v = vb + jc * 16;
                        if (jc * 16 < cols_here) {
                            if (args.resid && row < args.n) {
                                const int cg = cbk * 64 + jc * 16;
#pragma unroll
                                for (int i = 0; i < 16; ++i) {
                                    const float dv = (cg + i < args.n) ? v[i] - ((cg + i == row) ? 1.f : 0.f) : 0.f;
                                    rs_part = fmaf(dv, dv, rs_part);
                                }
                            }
#pragma unroll
                            for (int i = 0; i < 16; ++i) v[i] *= s_copy;
                            pg_stage_split16(dst_hi, dst_lo, lane, jc * 2, v);
                        } else {
                            pg_stage_zero16(dst_hi, dst_lo, lane, jc * 2);
                        }
                    }
                }
                fence_proxy_async_smem();                         // generic-proxy writes -> visible to the tensor core
                __syncwarp();
                if (lane == 0) mbar_arrive(&copy_bar[cbk]);
            }
            if (args.resid) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) rs_part += __shfl_xor_sync(0xffffffffu, rs_part, o);
                if (lane == 0) args.resid[static_cast<long long>(z) * args.fro_slots + e] = rs_part;
            }
            // ---- store: Bm = ca I + (cb r) acc
            mbar_wait(&acc2_bar[mt], ph_item);
            tc_fence_after();
            const float sc = args.cb * r;
            const int n_ch = (args.bn + 31) / 32;
            for (int ch = 0; ch < n_ch; ++ch) {
                float vb[32];
                const int c0 = ch * 32;
                if (c0 + 32 <= args.bn) tmem_ld32(t_addr + c0, vb);
                else tmem_ld16(t_addr + c0, vb);
#pragma unroll
                for (int jc = 0; jc < 2; ++jc) {
                    const int c = c0 + jc * 16;
                    float* v = vb + jc * 16;
                    if (c < args.bn) {
                        if (c0 == row0) {                          // the only chunk of this warp that holds diagonal entries
#pragma unroll
                            for (int i = 0; i < 16; ++i) v[i] = sc * v[i] + ((c + i == row) ? args.ca : 0.f);
                        } else {
#pragma unroll
                            for (int i = 0; i < 16; ++i) v[i] *= sc;
                        }
                    }
                }
                // the TMA store of the previous chunk may still be reading the staging tile: wait only now, after this
                // chunk's TMEM load and arithmetic
                if (ch > 0) {
                    if (lane == 0 && warp_rows_ok) tma_store_wait_read();
                    __syncwarp();
                }
#pragma unroll
                for (int jc = 0; jc < 2; ++jc) {
                    if (c0 + jc * 16 < args.bn) pf_stage_split16_sw64(stg_hi_s, stg_lo_s, lane, jc * 2, vb + jc * 16);
                    else pf_stage_zero16_sw64(stg_hi_s, stg_lo_s, lane, jc * 2);
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0 && warp_rows_ok) {
                    tma_store_4d(&maps.o[0], stg_hi, (ch & 1) * 32, row0, ch >> 1, z);
                    tma_store_4d(&maps.o[1], stg_lo, (ch & 1) * 32, row0, ch >> 1, z);
                    tma_store_commit();
                }
            }
            if (lane == 0 && warp_rows_ok) tma_store_wait_read();     // (the next problem's first chunk overwrites the tile)
            __syncwarp();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty_bar[mt]);
        }
        if (lane == 0) tma_store_wait_all();
    }
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, tmem_cols);
    }
}

}  // namespace basd
