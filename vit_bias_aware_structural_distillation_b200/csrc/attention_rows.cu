// Query-mean attention rows for teachers without a CLS token (SURVEY.md section 8(f) rank 1, the no-CLS half).
//
// relational.py:27 reads a no-CLS teacher's attention only as attn.mean((1, 2)) - over heads and ALL queries - yet the
// reference hook (src/models/teacher.py:27-39) materialises the full softmax(q k^T * scale) map [B,H,S,S] per block.  This
// kernel emits the per-head query mean straight from q and k and never stores an S x S map:
//     out[b,h,s] = (1/S) sum_q softmax_s'(scale q[b,h,q,:] . k[b,h,s',:])[s]                    fp32 [B,H,S]
//
// One CTA per (b, h), 128 threads, one TMEM lane (= one row of a 128-row tile) per thread.  Two passes over the same
// operand tiles, both K-major (q and k rows are dh-contiguous):
//   pass 1  S_tile = Q_tile K_tile^T (tcgen05, fp32 in TMEM): a thread owns a QUERY row and keeps its running max and sum of
//           exps over the key tiles; the max (log2 domain) and 1 / sum of every query go to shared memory.
//   pass 2  S_tile = K_tile Q_tile^T: a thread owns a KEY row and sums exp2(x - m_q) / l_q over the query tiles in registers.
// Rows past S come in as zeros from the TMA zero fill (score 0, not -inf): padded keys are skipped in pass 1, padded queries in
// pass 2.  Every sum runs in a fixed order inside one thread - no atomics, bitwise repeatable.
// bf16 operands go global -> shared by TMA (4-D tensor map over (d, s, h, b) strides: views into a fused qkv work in place;
// dh past a multiple of 64 is padded by the zero fill).  fp32 operands follow the project's split-bf16 convention: the threads
// load them, split each value into hi = bf16(x), lo = bf16(x - hi) and write both into the same swizzled layout; the product
// is hi*hi + hi*lo + lo*hi in one TMEM accumulator.
#include <cuda.h>

#include <cstring>

#include "ptx.cuh"
#include "spectral.h"

namespace basd {

int tensor_map_encode_bf16(CUtensorMap* map, int rank, const void* ptr, const uint64_t* dims, const uint64_t* strides_bytes,
                           const uint32_t* box);   // gemm_ops.cu

namespace {

constexpr int QM_THREADS = 128;
constexpr int QM_TILE = 128;                    // rows of a tile: UMMA M = N = 128
constexpr int QM_KB_BYTES = QM_TILE * 128;      // one 64-wide bf16 k-block of a tile (128-byte swizzled rows): 16 KB

struct QmMaps { CUtensorMap q, k; };
struct QmArgs {
    const float* q; const float* k;             // fp32 operands (the bf16 ones come through the tensor maps)
    long long qs[3], ks[3];                     // (b, h, s) element strides
    int B, H, S, dh;
    int kb_total, kb_chunk, n_chunks;           // 64-wide k-blocks; k-blocks held in shared memory at once
    int hq_inner, hk_inner;                     // tensor map of q / k ordered (d, h, s, b): its head stride is the smaller one
    float scale_log2;                           // scale * log2(e)
    float* out;                                 // [B][H][S]
};

// split-bf16 product terms: t = 0 hi*hi, 1 hi*lo, 2 lo*hi.  Operand tiles: 0 A hi, 1 B hi, 2 A lo, 3 B lo.
__device__ __forceinline__ int qm_term_a(int t) { return t == 2 ? 2 : 0; }
__device__ __forceinline__ int qm_term_b(int t) { return t == 1 ? 3 : 1; }

// fp32 rows [row0, row0 + 128) x k-blocks [kb0, kb0 + nkb) of one (b, h) -> hi / lo bf16 tiles in the SWIZZLE_128B K-major
// layout TMA would produce (16-byte chunk c of row r at r * 128 + (c ^ (r & 7)) * 16).  Rows past S and columns past dh: zeros.
__device__ __forceinline__ void qm_stage_f32(uint8_t* hi, uint8_t* lo, const float* src, long long ss, int row0, int S, int dh, int kb0,
                                             int nkb) {
    for (int i = 0; i < nkb; ++i)
#pragma unroll 2
    for (int u = threadIdx.x; u < QM_TILE * 8; u += QM_THREADS) {
        const int ch = u & 7, r = u >> 3;
        const int row = row0 + r, col = (kb0 + i) * 64 + ch * 8;
        float f[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (row < S && col < dh) {                      // dh % 8 == 0: a chunk is valid as a whole
            const float4* p = reinterpret_cast<const float4*>(src + row * ss + col);
            const float4 x0 = __ldg(p), x1 = __ldg(p + 1);
            f[0] = x0.x; f[1] = x0.y; f[2] = x0.z; f[3] = x0.w; f[4] = x1.x; f[5] = x1.y; f[6] = x1.z; f[7] = x1.w;
        }
        uint32_t hw[4], lw[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const __nv_bfloat16 h0 = __float2bfloat16(f[2 * e]), h1 = __float2bfloat16(f[2 * e + 1]);
            __nv_bfloat162 hv; hv.x = h0; hv.y = h1;
            hw[e] = *reinterpret_cast<uint32_t*>(&hv);
            lw[e] = pack_bf16x2(f[2 * e] - __bfloat162float(h0), f[2 * e + 1] - __bfloat162float(h1));
        }
        const uint32_t off = i * QM_KB_BYTES + r * 128 + ((ch ^ (r & 7)) << 4);
        *reinterpret_cast<uint4*>(hi + off) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
        *reinterpret_cast<uint4*>(lo + off) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
    }
}

template <bool F32>
__global__ void __launch_bounds__(QM_THREADS)
query_mean_attention_kernel(const __grid_constant__ QmMaps maps, const QmArgs a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* tiles = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    constexpr int kOps = F32 ? 4 : 2, kTerms = F32 ? 3 : 1;
    const int n_tiles = (a.S + QM_TILE - 1) / QM_TILE;
    float* m2 = reinterpret_cast<float*>(tiles + kOps * a.kb_chunk * QM_KB_BYTES);   // per query: running max, log2 domain
    float* il = m2 + n_tiles * QM_TILE;                                              // per query: 1 / sum of exps
    uint64_t* load_bar = reinterpret_cast<uint64_t*>(il + n_tiles * QM_TILE);
    uint64_t* mma_bar = load_bar + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mma_bar + 1);

    const int tid = threadIdx.x, warp = tid >> 5;
    const int bh = blockIdx.x, b = bh / a.H, h = bh - b * a.H;
    if (tid == 0) {
        mbar_init(load_bar, 1);
        mbar_init(mma_bar, 1);
        fence_mbar_init();
        if constexpr (!F32) { tma_prefetch_desc(&maps.q); tma_prefetch_desc(&maps.k); }
    }
    if (warp == 0) tmem_alloc(tmem_slot, QM_TILE);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t tm_row = tmem + (static_cast<uint32_t>(warp * 32) << 16);     // this warp's TMEM lane quadrant
    uint32_t load_phase = 0, mma_phase = 0;
    const float* qp = F32 ? a.q + b * a.qs[0] + h * a.qs[1] : nullptr;
    const float* kp = F32 ? a.k + b * a.ks[0] + h * a.ks[1] : nullptr;

    // TMEM[128 x 128] = rows [a_row0, +128) of A times rows [b_row0, +128) of B, over dh; A = q (pass 1) or k (pass 2), B the other.
    // The A tile stays in shared memory across the column tiles when all of dh fits there at once.
    auto product = [&](bool a_is_q, int a_row0, int b_row0, bool first_col_tile) {
        const bool load_a = first_col_tile || a.n_chunks > 1;
        for (int c = 0; c < a.n_chunks; ++c) {
            const int kb0 = c * a.kb_chunk, nkb = min(a.kb_chunk, a.kb_total - kb0);
            if constexpr (!F32) {
                if (tid == 0) {
                    mbar_arrive_expect_tx(load_bar, (load_a ? 2u : 1u) * nkb * QM_KB_BYTES);
                    const CUtensorMap* am = a_is_q ? &maps.q : &maps.k;
                    const CUtensorMap* bm = a_is_q ? &maps.k : &maps.q;
                    const int ah = a_is_q ? a.hq_inner : a.hk_inner, bh_ = a_is_q ? a.hk_inner : a.hq_inner;
                    for (int i = 0; i < nkb; ++i) {
                        const int d0 = (kb0 + i) * 64;
                        if (load_a) tma_load_4d(tiles + i * QM_KB_BYTES, am, load_bar, d0, ah ? h : a_row0, ah ? a_row0 : h, b);
                        tma_load_4d(tiles + (a.kb_chunk + i) * QM_KB_BYTES, bm, load_bar, d0, bh_ ? h : b_row0, bh_ ? b_row0 : h, b);
                    }
                    mbar_wait(load_bar, load_phase);
                }
                load_phase ^= 1;
            } else {
                if (load_a)
                    qm_stage_f32(tiles, tiles + 2 * a.kb_chunk * QM_KB_BYTES, a_is_q ? qp : kp, a_is_q ? a.qs[2] : a.ks[2], a_row0, a.S, a.dh, kb0, nkb);
                qm_stage_f32(tiles + a.kb_chunk * QM_KB_BYTES, tiles + 3 * a.kb_chunk * QM_KB_BYTES, a_is_q ? kp : qp,
                             a_is_q ? a.ks[2] : a.qs[2], b_row0, a.S, a.dh, kb0, nkb);
                fence_proxy_async_smem();                 // generic-proxy writes -> visible to the tensor core
                __syncthreads();
            }
            if (tid == 0) {
                tc_fence_after();
                constexpr uint32_t idesc = umma_idesc_bf16(QM_TILE, QM_TILE, false, false);
                for (int i = 0; i < nkb; ++i)
#pragma unroll
                    for (int t = 0; t < kTerms; ++t) {
                        const uint32_t ab = smem_u32(tiles + (qm_term_a(t) * a.kb_chunk + i) * QM_KB_BYTES);
                        const uint32_t bb = smem_u32(tiles + (qm_term_b(t) * a.kb_chunk + i) * QM_KB_BYTES);
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks)
                            umma_bf16(tmem, umma_smem_desc(ab + ks * 32, 16, 1024), umma_smem_desc(bb + ks * 32, 16, 1024), idesc,
                                      (c > 0 || i > 0 || t > 0 || ks > 0) ? 1u : 0u);
                    }
                umma_commit(mma_bar);
            }
            __syncwarp();
            mbar_wait(mma_bar, mma_phase);                // the tiles may be overwritten, the accumulator read
            mma_phase ^= 1;
            tc_fence_after();
        }
    };
    // every thread is done reading the accumulator before the next product overwrites it
    auto release_acc = [&]() { tc_fence_before(); __syncthreads(); };

    // ---- pass 1: per query, max and sum of exps over all keys
    for (int mt = 0; mt < n_tiles; ++mt) {
        float m = -INFINITY, l = 0.f;
        for (int nt = 0; nt < n_tiles; ++nt) {
            product(true, mt * QM_TILE, nt * QM_TILE, nt == 0);
            const int kvalid = min(QM_TILE, a.S - nt * QM_TILE);
            for (int c0 = 0; c0 < kvalid; c0 += 32) {     // (uniform over the CTA)
                float v[32];
                tmem_ld32(tm_row + c0, v);
                float cm = m;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    v[j] *= a.scale_log2;
                    if (c0 + j < kvalid) cm = fmaxf(cm, v[j]);
                }
                float s = 0.f;
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    if (c0 + j < kvalid) s += exp2f(v[j] - cm);
                l = l * exp2f(m - cm) + s;
                m = cm;
            }
            release_acc();
        }
        const int row = mt * QM_TILE + tid;
        if (row < a.S) { m2[row] = m; il[row] = 1.f / l; }
    }
    __syncthreads();

    // ---- pass 2: per key, sum over the queries of its normalised probability
    for (int mt = 0; mt < n_tiles; ++mt) {
        float acc = 0.f;
        for (int nt = 0; nt < n_tiles; ++nt) {
            product(false, mt * QM_TILE, nt * QM_TILE, nt == 0);
            const int qvalid = min(QM_TILE, a.S - nt * QM_TILE);
            for (int c0 = 0; c0 < qvalid; c0 += 32) {
                float v[32];
                tmem_ld32(tm_row + c0, v);
                const int q0 = nt * QM_TILE + c0;
                float s = 0.f;
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    if (c0 + j < qvalid) s += exp2f(fmaf(v[j], a.scale_log2, -m2[q0 + j])) * il[q0 + j];
                acc += s;
            }
            release_acc();
        }
        const int key = mt * QM_TILE + tid;
        if (key < a.S) a.out[static_cast<size_t>(bh) * a.S + key] = acc / static_cast<float>(a.S);
    }
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem, QM_TILE);
    }
}

}  // namespace

static size_t query_mean_attention_smem_bytes(int is_bf16, int S, int dh) {
    const int kb_total = (dh + 63) / 64, kb_chunk = is_bf16 ? kb_total : (kb_total < 2 ? kb_total : 2);
    const int n_tiles = (S + QM_TILE - 1) / QM_TILE;
    return 1024 + static_cast<size_t>(is_bf16 ? 2 : 4) * kb_chunk * QM_KB_BYTES + 2 * sizeof(float) * n_tiles * QM_TILE + 64;
}

cudaError_t launch_query_mean_attention(const void* q, const void* k, int is_bf16, int B, int H, int S, int dh, const long long* qst,
                                        const long long* kst, float scale, float* out, cudaStream_t st) {
    QmArgs a;
    memset(&a, 0, sizeof a);
    a.B = B; a.H = H; a.S = S; a.dh = dh;
    a.kb_total = (dh + 63) / 64;
    a.kb_chunk = is_bf16 ? a.kb_total : (a.kb_total < 2 ? a.kb_total : 2);    // fp32: hi + lo of both operands, two k-blocks at a time
    a.n_chunks = (a.kb_total + a.kb_chunk - 1) / a.kb_chunk;
    a.scale_log2 = static_cast<float>(static_cast<double>(scale) * 1.4426950408889634);
    a.out = out;
    for (int i = 0; i < 3; ++i) { a.qs[i] = qst[i]; a.ks[i] = kst[i]; }
    a.hq_inner = qst[1] < qst[2] ? 1 : 0;
    a.hk_inner = kst[1] < kst[2] ? 1 : 0;
    QmMaps maps;
    memset(&maps, 0, sizeof maps);
    if (is_bf16) {
        // 4-D maps over (d, s, h, b) - or (d, h, s, b) when the head stride is the smaller (fused qkv: s stride 3 H dh, h stride dh)
        const void* ptrs[2] = {q, k};
        const long long* strides[2] = {qst, kst};
        CUtensorMap* m[2] = {&maps.q, &maps.k};
        const int h_inner[2] = {a.hq_inner, a.hk_inner};
        for (int i = 0; i < 2; ++i) {
            const long long* s = strides[i];
            const uint64_t dims_s[4] = {static_cast<uint64_t>(dh), static_cast<uint64_t>(S), static_cast<uint64_t>(H), static_cast<uint64_t>(B)};
            const uint64_t str_s[3] = {2ull * s[2], 2ull * s[1], 2ull * s[0]};
            const uint32_t box_s[4] = {64, QM_TILE, 1, 1};
            const uint64_t dims_h[4] = {static_cast<uint64_t>(dh), static_cast<uint64_t>(H), static_cast<uint64_t>(S), static_cast<uint64_t>(B)};
            const uint64_t str_h[3] = {2ull * s[1], 2ull * s[2], 2ull * s[0]};
            const uint32_t box_h[4] = {64, 1, QM_TILE, 1};
            if (tensor_map_encode_bf16(m[i], 4, ptrs[i], h_inner[i] ? dims_h : dims_s, h_inner[i] ? str_h : str_s, h_inner[i] ? box_h : box_s))
                return cudaErrorInvalidValue;
        }
    } else {
        a.q = reinterpret_cast<const float*>(q);
        a.k = reinterpret_cast<const float*>(k);
    }
    const size_t smem = query_mean_attention_smem_bytes(is_bf16, S, dh);
    cudaError_t e;
    if (is_bf16) {
        e = cudaFuncSetAttribute(query_mean_attention_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
        if (e != cudaSuccess) return e;
        query_mean_attention_kernel<false><<<B * H, QM_THREADS, smem, st>>>(maps, a);
    } else {
        e = cudaFuncSetAttribute(query_mean_attention_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
        if (e != cudaSuccess) return e;
        query_mean_attention_kernel<true><<<B * H, QM_THREADS, smem, st>>>(maps, a);
    }
    return cudaGetLastError();
}

}  // namespace basd
