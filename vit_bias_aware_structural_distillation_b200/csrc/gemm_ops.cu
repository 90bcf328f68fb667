// Host launchers for the tcgen05 GEMM instances used by the BASD loss path (see umma_gemm.cuh).
// Tensor maps are encoded on the host per call (cuTensorMapEncodeTiled, resolved at run time through
// cudaGetDriverEntryPoint so the library links and loads on a machine without a driver).
#include <cudaTypedefs.h>

#include <cstdio>
#include <cstring>

#include "spectral.h"
#include "polar_gemm.cuh"

#include "polar_fused.cuh"
#include "umma_gemm.cuh"

namespace basd {

static thread_local char g_gemm_err[256] = "";
const char* gemm_last_error() { return g_gemm_err; }

using EncodeFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                              const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                              CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeFn g_encode = nullptr;

int gemm_init_driver_api() {
    if (g_encode) return 0;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
        snprintf(g_gemm_err, sizeof g_gemm_err, "cuTensorMapEncodeTiled unavailable: %s", cudaGetErrorString(e));
        return 1;
    }
    g_encode = reinterpret_cast<EncodeFn>(fn);
    return 0;
}

// bf16 tensor viewed as [batch][rows][inner]; box = [1][box_rows][64]; SWIZZLE_128B; OOB -> zeros.
static int make_map(CUtensorMap* map, const void* ptr, uint64_t inner, uint64_t rows, uint64_t batch, uint64_t row_pitch_elems,
                    uint64_t batch_pitch_elems, uint32_t box_rows) {
    if (gemm_init_driver_api()) return 1;
    if ((reinterpret_cast<uintptr_t>(ptr) & 15) || (row_pitch_elems * 2) % 16 || (batch_pitch_elems * 2) % 16) {
        snprintf(g_gemm_err, sizeof g_gemm_err, "TMA operand misaligned: ptr=%p row_pitch=%llu batch_pitch=%llu", ptr,
                 (unsigned long long)row_pitch_elems, (unsigned long long)batch_pitch_elems);
        return 1;
    }
    cuuint64_t dims[3] = {inner, rows, batch};
    cuuint64_t strides[2] = {row_pitch_elems * 2, batch_pitch_elems * 2};
    cuuint32_t box[3] = {64, box_rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        snprintf(g_gemm_err, sizeof g_gemm_err, "cuTensorMapEncodeTiled failed (%d) inner=%llu rows=%llu batch=%llu box_rows=%u", (int)r,
                 (unsigned long long)inner, (unsigned long long)rows, (unsigned long long)batch, box_rows);
        return 1;
    }
    return 0;
}

// bf16 tensor of any rank with explicit byte strides (dims[0] contiguous); box[0] = 64 (128-byte rows); SWIZZLE_128B; OOB -> zeros.
// For the other translation units (attention_rows.cu: 4-D maps over strided q / k views).
int tensor_map_encode_bf16(CUtensorMap* map, int rank, const void* ptr, const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box) {
    if (gemm_init_driver_api()) return 1;
    cuuint64_t d[5], s[4];
    cuuint32_t bx[5], estr[5];
    for (int i = 0; i < rank; ++i) { d[i] = dims[i]; bx[i] = box[i]; estr[i] = 1; }
    for (int i = 0; i + 1 < rank; ++i) s[i] = strides_bytes[i];
    CUresult r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, const_cast<void*>(ptr), d, s, bx, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        snprintf(g_gemm_err, sizeof g_gemm_err, "cuTensorMapEncodeTiled (rank %d) failed (%d) ptr=%p dims=%llu,%llu strides=%llu,%llu", rank, (int)r, ptr,
                 (unsigned long long)dims[0], (unsigned long long)dims[1], (unsigned long long)strides_bytes[0], (unsigned long long)strides_bytes[1]);
        return 1;
    }
    return 0;
}

// fp32 tensor viewed as [batch][rows][inner]; box = [1][32][32] (128-byte rows); SWIZZLE_128B; OOB -> zeros.
static int make_map_f32(CUtensorMap* map, const void* ptr, uint64_t inner, uint64_t rows, uint64_t batch, uint64_t row_pitch_elems,
                        uint64_t batch_pitch_elems) {
    if (gemm_init_driver_api()) return 1;
    if ((reinterpret_cast<uintptr_t>(ptr) & 15) || (row_pitch_elems * 4) % 16 || (batch_pitch_elems * 4) % 16) {
        snprintf(g_gemm_err, sizeof g_gemm_err, "TMA fp32 operand misaligned: ptr=%p row_pitch=%llu", ptr, (unsigned long long)row_pitch_elems);
        return 1;
    }
    cuuint64_t dims[3] = {inner, rows, batch};
    cuuint64_t strides[2] = {row_pitch_elems * 4, batch_pitch_elems * 4};
    cuuint32_t box[3] = {32, 32, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        snprintf(g_gemm_err, sizeof g_gemm_err, "cuTensorMapEncodeTiled (fp32) failed (%d) inner=%llu rows=%llu", (int)r,
                 (unsigned long long)inner, (unsigned long long)rows);
        return 1;
    }
    return 0;
}

// bf16 split matrix stored column-block tiled: [batch][col / 64][row][col % 64]; box = [1][1][box_rows][64].
static int make_map_tiled(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t col_blocks, uint64_t batch, uint64_t batch_pitch_elems,
                          uint32_t box_rows, uint32_t box_inner = 64) {
    if (gemm_init_driver_api()) return 1;
    if ((reinterpret_cast<uintptr_t>(ptr) & 127) || (batch_pitch_elems * 2) % 16) {
        snprintf(g_gemm_err, sizeof g_gemm_err, "tiled TMA operand misaligned: ptr=%p batch_pitch=%llu", ptr, (unsigned long long)batch_pitch_elems);
        return 1;
    }
    cuuint64_t dims[4] = {64, rows, col_blocks, batch};
    cuuint64_t strides[3] = {128, rows * 128, batch_pitch_elems * 2};
    cuuint32_t box[4] = {box_inner, box_rows, 1, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, box_inner == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        snprintf(g_gemm_err, sizeof g_gemm_err, "cuTensorMapEncodeTiled (tiled) failed (%d) rows=%llu blocks=%llu batch=%llu box_rows=%u", (int)r,
                 (unsigned long long)rows, (unsigned long long)col_blocks, (unsigned long long)batch, box_rows);
        return 1;
    }
    return 0;
}

// Function attributes and the SM count are per DEVICE: caches are indexed by the current device (a process may drive
// several GPUs); the flags are only ever set, so concurrent callers at worst repeat an idempotent call.
constexpr int kMaxDevices = 64;
static int current_device() {
    int dev = 0;
    cudaGetDevice(&dev);
    return dev >= 0 && dev < kMaxDevices ? dev : 0;
}
static int device_sm_count() {
    static int sm_count[kMaxDevices] = {0};
    const int dev = current_device();
    if (!sm_count[dev]) {
        int n = 0;
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        sm_count[dev] = n > 0 ? n : 148;
    }
    return sm_count[dev];
}

template <class Cfg, class Epi>
static cudaError_t launch(const GemmMaps& maps, const GemmArgs& args, dim3 grid, cudaStream_t st) {
    auto kern = umma_gemm_kernel<Cfg, Epi>;
    static bool configured[kMaxDevices] = {false};
    const int dev = current_device();
    if (!configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes);
        if (e != cudaSuccess) return e;
        configured[dev] = true;
    }
    kern<<<grid, GEMM_THREADS, Cfg::kSmemBytes, st>>>(maps, args);
    return cudaGetLastError();
}

static inline int cdiv(long long a, long long b) { return static_cast<int>((a + b - 1) / b); }

//                      A_MN   B_MN   BN   MT NA NB T  alias  stages
using CfgStudentGrad = GemmCfg<false, false, 192, 1, 1, 2, 2, false, 1>;   // one stage (65 KB), 256 TMEM columns: two CTAs per SM overlap each other
using CfgStudentGrad3 = GemmCfg<false, false, 192, 1, 2, 2, 3, false, 1>;  // split-bf16 students: + S_lo Gamma'_hi (one 81 KB stage)
using CfgGram    = GemmCfg<true,  true,  192, 2, 1, 1, 1, false, 3>;
using CfgGramA   = GemmCfg<true,  true,  192, 2, 1, 1, 1, true,  3>;      // D_s <= 192 (one output tile): the B tile is the A tile, one load per k-block
using CfgGram3   = GemmCfg<true,  true,  192, 2, 2, 2, 3, false, 2>;      // split operands: hi*hi + hi*lo + lo*hi
using CfgGram3A  = GemmCfg<true,  true,  192, 2, 2, 2, 3, true,  3>;      // the same with B aliased onto A (D_s <= 192)
// ... with the column sums of the operand from the same pass (umma_gemm.cuh: COLSUM)
using CfgGramAC  = GemmCfg<true,  true,  192, 2, 1, 1, 1, true,  3, true>;
// (two-tile Grams, D_s > 192, keep the separate column-sum kernel: gemm_gram_colsum_fused())
using CfgGram3AC = GemmCfg<true,  true,  192, 2, 2, 2, 3, true,  3, true>;
using CfgTheta   = GemmCfg<false, true,  128, 2, 1, 1, 1, false, 4>;      // self test (single operands)
template <int BN> using CfgTokenGram = GemmCfg<false, false, BN, 2, 2, 2, 3, true, 3>;
using CfgTestTN  = GemmCfg<false, false, 192, 1, 1, 1, 1, false, 4>;

// fp32 row-major outputs can leave the persistent kernel as TMA stores (epilogue kind 6) when base, row pitch and batch pitch are
// 16-byte aligned; otherwise (e.g. N_s = 50) as per-lane stores (kind 3)
static bool f32_tma_ok(const float* out, int ld, long long batch_stride) {
    return (reinterpret_cast<uintptr_t>(out) & 15) == 0 && ld % 4 == 0 && batch_stride % 4 == 0;
}

// Z[j] = X[j] P_t^T for all L_t teacher layers in ONE launch (the layers are separate tensors, so each has its own tensor map
// in maps.a_tab).  12 launches of 392 CTAs each left the last wave of every launch 65 % empty.
// The projection on the persistent polar_gemm kernel: work item = (layer, 128-row tile, column tile of <= 256 columns), A = the
// teacher tokens of that layer through the layer's own tensor map (one exact bf16 buffer: two split terms against P_t hi / lo),
// operand ring and two TMEM accumulators carried across items, Z leaves as a row-major split pair through swizzled staging and
// TMA stores (ROWMAJOR epilogue; the rows between the samples of a CLS-stripped view are written as zeros).  The one-tile-per-CTA
// kernel it replaced ran a two-stage ring and per-lane 32-byte row stores with nothing overlapped: 59 k cycles per 256-row tile
// against 18 k of MMAs (0.48 ms at cfg2).
// Split-bf16 teachers (Xlo non-null; X[0] = the hi block [n_layers][M][Dt], Xlo the lo block, both packed): the layers are one
// batched tensor map per half and the third term X_lo P_hi^T joins the two (a_single = 0).
static cudaError_t project_persistent(const void* const* X, const __nv_bfloat16* Xlo, int n_layers, size_t M, int Dt, const __nv_bfloat16* Phi,
                                      const __nv_bfloat16* Plo, int Ds, __nv_bfloat16* Z, __nv_bfloat16* Zlo, int gap_period, int gap_valid,
                                      cudaStream_t st) {
    PolarGemmArgs a;
    memset(&a, 0, sizeof a);
    a.epi = PG_EPI_ROWMAJOR; a.scale_c = 1.f; a.a_rm = 1; a.b_rm = 1; a.a_single = Xlo ? 0 : 1; a.b_shared = 1;
    a.gap_period = gap_period; a.gap_valid = gap_valid;
    a.ld_out = Ds; a.out_stride = static_cast<long long>(M) * Ds;
    a.m_rows = static_cast<int>(M); a.n_cols = Ds; a.k_total = Dt;
    a.n_mt = static_cast<int>((M + 127) / 128);
    if (Ds <= 256) {
        a.n_nt = 1; a.bn_mma = (Ds + 15) / 16 * 16;
    } else {
        a.n_nt = (Ds + 255) / 256;
        a.bn_mma = ((Ds + a.n_nt - 1) / a.n_nt + 63) / 64 * 64;
        a.n_nt = (Ds + a.bn_mma - 1) / a.bn_mma;
    }
    a.b_groups = (a.bn_mma + 63) / 64;
    const int stage_bytes = (Xlo ? 2 : 1) * 16384 + 2 * a.bn_mma * 128;
    const int kTail = 1024 /*alignment*/ + 1024 /*barriers*/ + 4 * 8192 /*epilogue staging*/;
    int stages = (232448 - kTail) / stage_bytes;
    if (stages > 4) stages = 4;
    if (stages < 1) return cudaErrorInvalidValue;
    a.stages = stages;
    const int smem = stages * stage_bytes + kTail;
    const int sm_count = device_sm_count();
    if (Xlo) {
        PolarGemmMaps maps;
        memset(&maps, 0, sizeof maps);
        if (make_map(&maps.a[0], X[0], Dt, M, n_layers, Dt, M * Dt, 64)) return cudaErrorInvalidValue;
        if (make_map(&maps.a[1], Xlo, Dt, M, n_layers, Dt, M * Dt, 64)) return cudaErrorInvalidValue;
        if (make_map(&maps.b[0], Phi, Dt, Ds, 1, Dt, static_cast<uint64_t>(Ds) * Dt, a.bn_mma)) return cudaErrorInvalidValue;
        if (make_map(&maps.b[1], Plo, Dt, Ds, 1, Dt, static_cast<uint64_t>(Ds) * Dt, a.bn_mma)) return cudaErrorInvalidValue;
        a.out_hi = Z; a.out_lo = Zlo;
        if (make_map(&maps.o[0], Z, Ds, M, n_layers, Ds, M * Ds, 32)) return cudaErrorInvalidValue;
        if (make_map(&maps.o[1], Zlo, Ds, M, n_layers, Ds, M * Ds, 32)) return cudaErrorInvalidValue;
        a.n_items = n_layers * a.n_mt * a.n_nt; a.n_batches = n_layers;
        auto kern = polar_gemm_kernel<false, 4>;
        static bool configured_split[kMaxDevices] = {};
        const int dev = current_device();
        if (!configured_split[dev]) {
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
            if (e != cudaSuccess) return e;
            configured_split[dev] = true;
        }
        kern<<<a.n_items < sm_count ? a.n_items : sm_count, PG_THREADS, smem, st>>>(maps, a);
        return cudaGetLastError();
    }
    auto kern = polar_gemm_kernel<false, 4, true>;
    static bool configured[kMaxDevices] = {};
    const int dev = current_device();
    if (!configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
        if (e != cudaSuccess) return e;
        configured[dev] = true;
    }
    for (int j0 = 0; j0 < n_layers; j0 += PG_MAX_A_TABLE) {
        const int nl = n_layers - j0 < PG_MAX_A_TABLE ? n_layers - j0 : PG_MAX_A_TABLE;
        PolarGemmMapsT maps;
        memset(&maps, 0, sizeof maps);
        for (int j = 0; j < nl; ++j)
            if (make_map(&maps.a_tab[j], X[j0 + j], Dt, M, 1, Dt, M * Dt, 64)) return cudaErrorInvalidValue;
        if (make_map(&maps.b[0], Phi, Dt, Ds, 1, Dt, static_cast<uint64_t>(Ds) * Dt, a.bn_mma)) return cudaErrorInvalidValue;
        if (make_map(&maps.b[1], Plo, Dt, Ds, 1, Dt, static_cast<uint64_t>(Ds) * Dt, a.bn_mma)) return cudaErrorInvalidValue;
        a.out_hi = Z + static_cast<size_t>(j0) * M * Ds; a.out_lo = Zlo + static_cast<size_t>(j0) * M * Ds;
        if (make_map(&maps.o[0], a.out_hi, Ds, M, nl, Ds, M * Ds, 32)) return cudaErrorInvalidValue;
        if (make_map(&maps.o[1], a.out_lo, Ds, M, nl, Ds, M * Ds, 32)) return cudaErrorInvalidValue;
        a.n_items = nl * a.n_mt * a.n_nt; a.n_batches = nl;
        kern<<<a.n_items < sm_count ? a.n_items : sm_count, PG_THREADS, smem, st>>>(maps, a);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

cudaError_t gemm_project(const void* const* X, int n_layers, size_t M, int Dt, const __nv_bfloat16* Phi, const __nv_bfloat16* Plo, int Ds,
                         __nv_bfloat16* Z, __nv_bfloat16* Zlo, int gap_period, int gap_valid, cudaStream_t st, const __nv_bfloat16* Xlo) {
    if (M >= (size_t(1) << 31) - 128) {             // the kernel's row indices are ints
        snprintf(g_gemm_err, sizeof g_gemm_err, "project: %zu teacher rows, at most 2^31 - 129 supported", M);
        return cudaErrorInvalidValue;
    }
    if (Xlo && gap_period) {                        // split-bf16 teachers arrive packed: dense layers
        snprintf(g_gemm_err, sizeof g_gemm_err, "project: split-bf16 teachers need dense packed layers");
        return cudaErrorInvalidValue;
    }
    return project_persistent(X, Xlo, n_layers, M, Dt, Phi, Plo, Ds, Z, Zlo, gap_period, gap_valid, st);
}

// out[b][e] = sum over the n_splits slices of part[(b * n_splits + s) * elems + e], s ascending: fixed order
__global__ void __launch_bounds__(256)
splitk_reduce_kernel(const float* __restrict__ part, int n_splits, int elems4, float* __restrict__ out, long long out_stride) {
    const int b = blockIdx.y;
    const float4* p = reinterpret_cast<const float4*>(part) + static_cast<size_t>(b) * n_splits * elems4;
    float4* o = reinterpret_cast<float4*>(out + b * out_stride);
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < elems4; e += gridDim.x * blockDim.x) {
        float4 acc = p[e];
        for (int s2 = 1; s2 < n_splits; ++s2) {
            const float4 v = p[static_cast<size_t>(s2) * elems4 + e];
            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
        o[e] = acc;
    }
}
// split-K geometry of a Gram over M rows: at most kGramMaxSplits slices.  The Gram kernels run one CTA per SM, so the launch lasts
// (waves of CTAs) x (k-blocks per slice + the fixed cost of a CTA: set-up and the unoverlapped epilogue, ~10 k-blocks' worth) plus
// the fixed-order reduction over the slices; ctas_per_slice = output tiles x batches.  (32 k-blocks per slice whatever the grid
// gave 12 layers x 25 slices = 300 CTAs at cfg2: two full waves and a third of four CTAs - a third of the launch.)
constexpr int kGramMaxSplits = 32;
static void gram_splits(size_t M, int ctas_per_slice, int* kb_total, int* kb_per_split, int* n_splits) {
    *kb_total = cdiv(M, GEMM_BK);
    const int sms = device_sm_count();
    int best_per = *kb_total;
    double best_cost = 1e300;
    for (int ns = 1; ns <= kGramMaxSplits && ns <= *kb_total; ++ns) {
        const int per = cdiv(*kb_total, ns);
        if (cdiv(*kb_total, per) != ns) continue;                       // the same geometry as a smaller ns
        const double waves = static_cast<double>(cdiv(static_cast<long long>(ctas_per_slice) * ns, sms));
        const double cost = waves * (per + 10.0) + 0.08 * ns * ctas_per_slice;
        if (cost < best_cost) { best_cost = cost; best_per = per; }
    }
    *kb_per_split = best_per;
    *n_splits = cdiv(*kb_total, best_per);
}
static int gram_tiles(int Ds) { return cdiv(Ds, CfgGram::kBN) * cdiv(Ds, CfgGram::kMT * 128); }
size_t gemm_gram_part_floats(size_t M, int Ds, int batches) {      // sized for the largest slice count (device independent)
    const int ns = cdiv(M, GEMM_BK) < kGramMaxSplits ? cdiv(M, GEMM_BK) : kGramMaxSplits;
    return static_cast<size_t>(ns > 0 ? ns : 1) * batches * (static_cast<size_t>(Ds) * Ds + Ds);       // Gram slices, then column-sum slices
}
// Fused where it was measured to pay: the single-tile (aliased) Grams, D_s <= 192 (cfg2: gram + colsum 0.33 -> 0.27 ms).  Two-tile
// Grams (D_s = 384) got SLOWER with the extra MMAs in every column tile (cfg4: gram 1.27 -> 1.59 ms against 0.04 saved).
bool gemm_gram_colsum_fused(int Ds, bool split) { (void)split; return Ds <= CfgGram::kBN; }
static cudaError_t gram_reduce(const float* part, int n_splits, int Ds, int batches, float* G, long long g_stride, cudaStream_t st) {
    if ((Ds * Ds) % 4 || (g_stride % 4)) return cudaErrorInvalidValue;
    const int elems4 = Ds * Ds / 4;
    int gx = (elems4 + 255) / 256;
    if (gx > 64) gx = 64;
    splitk_reduce_kernel<<<dim3(gx, batches), 256, 0, st>>>(part, n_splits, elems4, G, g_stride);
    return cudaGetLastError();
}
// column sums: csum[b][d] = sum over the slices of cpart[(b * n_splits + s) * Ds + d], s ascending, written behind the Gram of batch b
static cudaError_t csum_reduce(const float* cpart, int n_splits, int Ds, int batches, float* G, long long g_stride, cudaStream_t st) {
    if (Ds % 4 || (g_stride % 4)) return cudaErrorInvalidValue;
    splitk_reduce_kernel<<<dim3(1, batches), 256, 0, st>>>(cpart, n_splits, Ds / 4, G + static_cast<size_t>(Ds) * Ds, g_stride);
    return cudaGetLastError();
}

// G[batch] = Z[batch]^T Z[batch]; Z = [batches][M][Ds] contiguous (optionally a split hi/lo pair); G batch stride in floats.
// part: gemm_gram_part_floats(M, Ds, batches) floats of scratch for the split-K slices.
// with_colsum: the column sums of Z (hi + lo) are written behind each Gram (G[b] + Ds * Ds: the layout of the pooled statistics)
static cudaError_t gram_impl(const __nv_bfloat16* Z, const __nv_bfloat16* Zlo, size_t M, int Ds, int batches, float* G, long long g_stride,
                             float* part, cudaStream_t st, bool with_colsum = false) {
    GemmMaps maps;
    memset(&maps, 0, sizeof maps);
    if (make_map(&maps.a[0], Z, Ds, M, batches, Ds, M * Ds, 64)) return cudaErrorInvalidValue;
    maps.b[0] = maps.a[0];
    if (Zlo) {
        if (make_map(&maps.a[1], Zlo, Ds, M, batches, Ds, M * Ds, 64)) return cudaErrorInvalidValue;
        maps.b[1] = maps.a[1];
    }
    GemmArgs a;
    memset(&a, 0, sizeof a);
    gram_splits(M, gram_tiles(Ds) * batches, &a.kb_total, &a.kb_per_split, &a.n_splits);
    a.a_batched = 1; a.b_batched = 1;
    a.out = part; a.out_batch_stride = static_cast<long long>(Ds) * Ds; a.ld_out = Ds; a.rows_valid = Ds; a.cols_valid = Ds;
    float* cpart = part + static_cast<size_t>(a.n_splits) * batches * Ds * Ds;
    a.aux0 = with_colsum ? cpart : nullptr;
    const dim3 grid(cdiv(Ds, CfgGram::kBN), cdiv(Ds, CfgGram::kMT * 128), batches * a.n_splits);
    const bool alias = Ds <= CfgGram::kBN;                    // a single output tile: A tile == B tile
    cudaError_t e;
    if (with_colsum && !gemm_gram_colsum_fused(Ds, Zlo != nullptr)) return cudaErrorInvalidValue;
    if (with_colsum) {
        if (Zlo) e = launch<CfgGram3AC, EpiStoreSplitK>(maps, a, grid, st);
        else e = launch<CfgGramAC, EpiStoreSplitK>(maps, a, grid, st);
    } else {
        if (Zlo) e = alias ? launch<CfgGram3A, EpiStoreSplitK>(maps, a, grid, st) : launch<CfgGram3, EpiStoreSplitK>(maps, a, grid, st);
        else e = alias ? launch<CfgGramA, EpiStoreSplitK>(maps, a, grid, st) : launch<CfgGram, EpiStoreSplitK>(maps, a, grid, st);
    }
    if (e != cudaSuccess) return e;
    e = gram_reduce(part, a.n_splits, Ds, batches, G, g_stride, st);
    if (e != cudaSuccess || !with_colsum) return e;
    return csum_reduce(cpart, a.n_splits, Ds, batches, G, g_stride, st);
}
cudaError_t gemm_gram(const __nv_bfloat16* Z, const __nv_bfloat16* Zlo, size_t M, int Ds, float* G, float* part, cudaStream_t st) {
    return gram_impl(Z, Zlo, M, Ds, 1, G, 0, part, st);
}
// G[i] += S_i^T S_i for n separate [M][Ds] bf16 tensors in ONE launch (blockIdx.z = tensor x split; a single Gram is 25
// CTAs - four of them back to back were 4 x 50 us of latency)
// rows_per_batch > 0: the tensors are [B][rows_per_batch][Ds] with batch stride batch_stride elements (CLS-stripped views):
// the K dimension walks 64-row blocks per sample (GemmArgs::kb_per_batch), M = B * rows_per_batch
cudaError_t gemm_gram_table(const void* const* S, int n, size_t M, int Ds, float* G, long long g_stride, float* part, int rows_per_batch,
                            long long batch_stride, cudaStream_t st, bool with_colsum) {
    if (n > GEMM_MAX_A_TABLE) return cudaErrorInvalidValue;
    GemmMaps maps;
    memset(&maps, 0, sizeof maps);
    GemmArgs a;
    memset(&a, 0, sizeof a);
    if (rows_per_batch > 0) {
        const size_t B = M / rows_per_batch;
        for (int i = 0; i < n; ++i)
            if (make_map(&maps.a_table[i], S[i], Ds, rows_per_batch, B, Ds, batch_stride, 64)) return cudaErrorInvalidValue;
        a.kb_per_batch = cdiv(rows_per_batch, GEMM_BK);
        gram_splits(B * a.kb_per_batch * GEMM_BK, gram_tiles(Ds) * n, &a.kb_total, &a.kb_per_split, &a.n_splits);
    } else {
        for (int i = 0; i < n; ++i)
            if (make_map(&maps.a_table[i], S[i], Ds, M, 1, Ds, M * Ds, 64)) return cudaErrorInvalidValue;
        gram_splits(M, gram_tiles(Ds) * n, &a.kb_total, &a.kb_per_split, &a.n_splits);
    }
    a.a_table = 1; a.b_table = 1;
    a.out = part; a.out_batch_stride = static_cast<long long>(Ds) * Ds; a.ld_out = Ds; a.rows_valid = Ds; a.cols_valid = Ds;
    float* cpart = part + static_cast<size_t>(a.n_splits) * n * Ds * Ds;
    a.aux0 = with_colsum ? cpart : nullptr;
    const dim3 grid(cdiv(Ds, CfgGram::kBN), cdiv(Ds, CfgGram::kMT * 128), n * a.n_splits);
    cudaError_t e;
    if (with_colsum && !gemm_gram_colsum_fused(Ds, false)) return cudaErrorInvalidValue;
    if (with_colsum) e = launch<CfgGramAC, EpiStoreSplitK>(maps, a, grid, st);
    else e = Ds <= CfgGram::kBN ? launch<CfgGramA, EpiStoreSplitK>(maps, a, grid, st) : launch<CfgGram, EpiStoreSplitK>(maps, a, grid, st);
    if (e != cudaSuccess) return e;
    e = gram_reduce(part, a.n_splits, Ds, n, G, g_stride, st);
    if (e != cudaSuccess || !with_colsum) return e;
    return csum_reduce(cpart, a.n_splits, Ds, n, G, g_stride, st);
}
cudaError_t gemm_gram_batched(const __nv_bfloat16* Z, const __nv_bfloat16* Zlo, size_t M, int Ds, int batches, float* G, long long g_stride,
                              float* part, cudaStream_t st, bool with_colsum) {
    return gram_impl(Z, Zlo, M, Ds, batches, G, g_stride, part, st, with_colsum);
}

template <int BN>
static cudaError_t token_gram_impl(const __nv_bfloat16* Thi, const __nv_bfloat16* Tlo, int batches, int Ns, int Dt, float* Ktt,
                                   cudaStream_t st) {
    GemmMaps maps;
    memset(&maps, 0, sizeof maps);
    if (make_map(&maps.a[0], Thi, Dt, Ns, batches, Dt, static_cast<uint64_t>(Ns) * Dt, 128)) return cudaErrorInvalidValue;
    if (make_map(&maps.a[1], Tlo, Dt, Ns, batches, Dt, static_cast<uint64_t>(Ns) * Dt, 128)) return cudaErrorInvalidValue;
    GemmArgs a;
    memset(&a, 0, sizeof a);
    a.kb_total = cdiv(Dt, GEMM_BK);
    a.a_batched = 1;
    a.out = Ktt; a.out_batch_stride = static_cast<long long>(Ns) * Ns; a.ld_out = Ns; a.rows_valid = Ns; a.cols_valid = Ns; a.alpha = 1.f;
    return launch<CfgTokenGram<BN>, EpiStoreF32>(maps, a, dim3(1, 1, batches), st);
}
// K[z] = T[z] T[z]^T on the persistent polar_gemm kernel: T (row-major split pair [Ns][Dt]) is both operands, work item =
// (sample, 128-row tile, column tile); with one column tile (Ns <= 256) the A tile is read out of the B tile (no A loads; the
// second row tile of a sample re-reads the B tile from L2), the fp32 result leaves from the epilogue warps while the next item's
// MMAs fill the other TMEM accumulator.  The one-tile-per-CTA kernel above (both row tiles against one load of T, nothing
// overlapped) took 69 k cycles per sample against 30 k of MMAs (0.24 ms at cfg2).
static cudaError_t token_gram_persistent(const __nv_bfloat16* Thi, const __nv_bfloat16* Tlo, int batches, int Ns, int Dt, float* Ktt,
                                         cudaStream_t st) {
    PolarGemmArgs a;
    memset(&a, 0, sizeof a);
    a.epi = PG_EPI_F32; a.scale_c = 1.f; a.a_rm = 1; a.b_rm = 1;
    a.out_f32 = Ktt; a.out_f32_stride = static_cast<long long>(Ns) * Ns; a.ld_f32 = Ns;
    a.m_rows = Ns; a.n_cols = Ns; a.k_total = Dt;
    a.n_mt = (Ns + 127) / 128;
    if (Ns <= 256) {
        a.n_nt = 1; a.bn_mma = (Ns + 15) / 16 * 16; a.a_alias_b = 1;
    } else {
        a.n_nt = (Ns + 255) / 256;
        a.bn_mma = ((Ns + a.n_nt - 1) / a.n_nt + 63) / 64 * 64;
        a.n_nt = (Ns + a.bn_mma - 1) / a.bn_mma;
    }
    a.n_items = batches * a.n_mt * a.n_nt; a.n_batches = batches;
    a.b_groups = (a.bn_mma + 63) / 64;
    PolarGemmMaps maps;
    memset(&maps, 0, sizeof maps);
    const __nv_bfloat16* tp[2] = {Thi, Tlo};
    for (int i = 0; i < 2; ++i) {
        if (make_map(&maps.a[i], tp[i], Dt, Ns, batches, Dt, static_cast<uint64_t>(Ns) * Dt, 64)) return cudaErrorInvalidValue;
        if (make_map(&maps.b[i], tp[i], Dt, Ns, batches, Dt, static_cast<uint64_t>(Ns) * Dt, a.bn_mma)) return cudaErrorInvalidValue;
    }
    const int stage_bytes = (a.a_alias_b ? 0 : 2 * 16384) + 2 * a.bn_mma * 128;
    // (the aliased A tile of the last rows reads up to 16 KB past its B tile: into the next tile or the barrier / staging area -
    //  rows past Ns, never stored)
    const int kTail = 1024 /*alignment*/ + 1024 /*barriers*/ + 4 * 8192 /*epilogue staging (unused by the fp32 epilogue; over-read area)*/;
    int stages = (232448 - kTail) / stage_bytes;
    if (stages > 4) stages = 4;
    if (stages < 1) return cudaErrorInvalidValue;
    a.stages = stages;
    const int smem = stages * stage_bytes + kTail;
    const bool tma_out = f32_tma_ok(Ktt, Ns, a.out_f32_stride);
    if (tma_out && make_map_f32(&maps.o[0], Ktt, Ns, Ns, batches, Ns, a.out_f32_stride)) return cudaErrorInvalidValue;
    auto kern = tma_out ? polar_gemm_kernel<false, 6> : polar_gemm_kernel<false, 3>;
    static bool configured[kMaxDevices][2] = {};
    const int dev = current_device();
    if (!configured[dev][tma_out]) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
        if (e != cudaSuccess) return e;
        configured[dev][tma_out] = true;
    }
    const int sm_count = device_sm_count();
    kern<<<a.n_items < sm_count ? a.n_items : sm_count, PG_THREADS, smem, st>>>(maps, a);
    return cudaGetLastError();
}
cudaError_t gemm_token_gram(const __nv_bfloat16* Thi, const __nv_bfloat16* Tlo, int batches, int Ns, int Dt, float* Ktt, cudaStream_t st) {
    // fewer than 16 tokens (e.g. a 3 x 3 teacher grid in the token-space form): the one-tile-per-CTA kernel
    if (Ns < 16) return token_gram_impl<64>(Thi, Tlo, batches, Ns, Dt, Ktt, st);
    return token_gram_persistent(Thi, Tlo, batches, Ns, Dt, Ktt, st);
}

// D[z] = Theta[z] (Ns x Ns, row-major split pair, pitch NsPad) * T[z] (Ns x Dt, row-major split pair): the persistent polar_gemm
// kernel (operand ring and two TMEM accumulators carried across work items, TMA-store epilogue) on row-major operands.
// Work item = (sample, 128-row tile, column tile of <= 256).  The one-tile-per-CTA kernel this replaces (CfgTheta3: one 96 KB
// stage, per-lane 32-byte stores) serialised load, MMA and epilogue: 0.47 ms at cfg2.
static cudaError_t theta_apply_persistent(const __nv_bfloat16* theta, const __nv_bfloat16* theta_lo, int NsPad, const __nv_bfloat16* Thi,
                                          const __nv_bfloat16* Tlo, int batches, int Ns, int Dt, __nv_bfloat16* Dtm, __nv_bfloat16* Dtm_lo,
                                          cudaStream_t st) {
    PolarGemmArgs a;
    memset(&a, 0, sizeof a);
    a.epi = PG_EPI_ROWMAJOR; a.scale_c = 1.f; a.a_rm = 1; a.b_rm = 1;
    a.out_hi = Dtm; a.out_lo = Dtm_lo; a.ld_out = Dt; a.out_stride = static_cast<long long>(Ns) * Dt;
    a.m_rows = Ns; a.n_cols = Dt; a.k_total = Ns;
    a.n_mt = (Ns + 127) / 128;
    if (Dt <= 256) {
        a.n_nt = 1; a.bn_mma = (Dt + 15) / 16 * 16;
    } else {
        a.n_nt = (Dt + 255) / 256;
        a.bn_mma = ((Dt + a.n_nt - 1) / a.n_nt + 63) / 64 * 64;
        a.n_nt = (Dt + a.bn_mma - 1) / a.bn_mma;
    }
    a.n_items = batches * a.n_mt * a.n_nt; a.n_batches = batches;
    a.b_groups = (a.bn_mma + 63) / 64;
    PolarGemmMaps maps;
    memset(&maps, 0, sizeof maps);
    // inner extent Ns (not NsPad): the pad columns are never read, TMA zero-fills them
    if (make_map(&maps.a[0], theta, Ns, Ns, batches, NsPad, static_cast<uint64_t>(Ns) * NsPad, 64)) return cudaErrorInvalidValue;
    if (make_map(&maps.a[1], theta_lo, Ns, Ns, batches, NsPad, static_cast<uint64_t>(Ns) * NsPad, 64)) return cudaErrorInvalidValue;
    if (make_map(&maps.b[0], Thi, Dt, Ns, batches, Dt, static_cast<uint64_t>(Ns) * Dt, 64)) return cudaErrorInvalidValue;
    if (make_map(&maps.b[1], Tlo, Dt, Ns, batches, Dt, static_cast<uint64_t>(Ns) * Dt, 64)) return cudaErrorInvalidValue;
    if (make_map(&maps.o[0], Dtm, Dt, Ns, batches, Dt, static_cast<uint64_t>(Ns) * Dt, 32)) return cudaErrorInvalidValue;
    if (Dtm_lo && make_map(&maps.o[1], Dtm_lo, Dt, Ns, batches, Dt, static_cast<uint64_t>(Ns) * Dt, 32)) return cudaErrorInvalidValue;
    const int stage_bytes = 2 * 16384 + 2 * a.b_groups * 8192;
    const int kTail = 1024 /*alignment*/ + 1024 /*barriers*/ + 4 * 8192 /*epilogue staging*/;
    int stages = (232448 - kTail) / stage_bytes;
    if (stages > 4) stages = 4;
    if (stages < 1) return cudaErrorInvalidValue;
    a.stages = stages;
    const int smem = stages * stage_bytes + kTail;
    auto kern = polar_gemm_kernel<true, 4>;
    static bool configured[kMaxDevices] = {};
    const int dev = current_device();
    if (!configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
        if (e != cudaSuccess) return e;
        configured[dev] = true;
    }
    const int sm_count = device_sm_count();
    kern<<<a.n_items < sm_count ? a.n_items : sm_count, PG_THREADS, smem, st>>>(maps, a);
    return cudaGetLastError();
}

cudaError_t gemm_theta_apply(const __nv_bfloat16* theta, const __nv_bfloat16* theta_lo, int NsPad, const __nv_bfloat16* Thi,
                             const __nv_bfloat16* Tlo, int batches, int Ns, int Dt, __nv_bfloat16* Dtm, __nv_bfloat16* Dtm_lo, cudaStream_t st) {
    // the gradient w.r.t. the mixed teacher leaves as a split pair: rounded to one bf16 it cost 1e-4 .. 6e-4 on the
    // temperature gradients (they are differences of nearly equal per-layer dots of this tensor)
    // (Dtm_lo == nullptr: large tensors, where the rounding averages out, leave as one bf16)
    if (Dt % 8 || NsPad % 8) {
        snprintf(g_gemm_err, sizeof g_gemm_err, "theta_apply: Dt = %d and the Theta pitch %d must be multiples of 8", Dt, NsPad);
        return cudaErrorInvalidValue;
    }
    return theta_apply_persistent(theta, theta_lo, NsPad, Thi, Tlo, batches, Ns, Dt, Dtm, Dtm_lo, st);
}

// Student gradient on the persistent polar_gemm kernel (dense bf16 students, bf16 gradient): work item = (128-row tile of the
// [M][Ds] gradient, column tile), A = the raw student tokens (one exact bf16 buffer: two split terms against Gamma' hi / lo), the
// direct-path gradient and the centring correction enter in the epilogue (SGRAD), the tile leaves through swizzled staging as TMA
// stores.  The one-tile-per-CTA kernel it replaces ran at 1.2 TB/s (ncu, r2k): single 65 KB stage, per-lane row-strided loads
// of gdir and stores of the gradient, load -> MMA -> epilogue in sequence.
static cudaError_t student_grad_persistent(const __nv_bfloat16* S, size_t M, int Ds, const __nv_bfloat16* Ghi, const __nv_bfloat16* Glo,
                                           const float* gdir, const float* corr, const float* scale_ptr, float scale_host,
                                           __nv_bfloat16* out, cudaStream_t st) {
    PolarGemmArgs a;
    memset(&a, 0, sizeof a);
    a.epi = PG_EPI_SGRAD; a.scale_c = 1.f; a.a_rm = 1; a.b_rm = 1; a.a_single = 1;
    a.sg_gdir = gdir; a.sg_corr = corr; a.sg_scale = scale_ptr; a.sg_alpha = scale_host;
    a.out_hi = out; a.out_lo = nullptr; a.ld_out = Ds; a.out_stride = static_cast<long long>(M) * Ds;
    a.m_rows = static_cast<int>(M); a.n_cols = Ds; a.k_total = Ds;
    a.n_mt = static_cast<int>((M + 127) / 128);
    if (Ds <= 256) {
        a.n_nt = 1; a.bn_mma = (Ds + 15) / 16 * 16;
    } else {
        a.n_nt = (Ds + 255) / 256;
        a.bn_mma = ((Ds + a.n_nt - 1) / a.n_nt + 63) / 64 * 64;
        a.n_nt = (Ds + a.bn_mma - 1) / a.bn_mma;
    }
    a.n_items = a.n_mt * a.n_nt; a.n_batches = 1;
    a.b_groups = (a.bn_mma + 63) / 64;
    PolarGemmMaps maps;
    memset(&maps, 0, sizeof maps);
    if (make_map(&maps.a[0], S, Ds, M, 1, Ds, M * Ds, 64)) return cudaErrorInvalidValue;
    if (make_map(&maps.b[0], Ghi, Ds, Ds, 1, Ds, static_cast<uint64_t>(Ds) * Ds, a.bn_mma)) return cudaErrorInvalidValue;
    if (make_map(&maps.b[1], Glo, Ds, Ds, 1, Ds, static_cast<uint64_t>(Ds) * Ds, a.bn_mma)) return cudaErrorInvalidValue;
    if (make_map(&maps.o[0], out, Ds, M, 1, Ds, M * Ds, 32)) return cudaErrorInvalidValue;
    if (make_map_f32(&maps.o[2], gdir, Ds, M, 1, Ds, M * Ds)) return cudaErrorInvalidValue;
    const int stage_bytes = 16384 + 2 * a.bn_mma * 128;
    const int kTail = 1024 /*alignment*/ + 1024 /*barriers*/ + 4 * 8192 /*epilogue staging*/ + 4 * 8192 /*gdir tiles*/;
    int stages = (232448 - kTail) / stage_bytes;
    if (stages > 4) stages = 4;
    if (stages < 1) return cudaErrorInvalidValue;
    a.stages = stages;
    const int smem = stages * stage_bytes + kTail;
    auto kern = polar_gemm_kernel<false, 5>;
    static bool configured[kMaxDevices] = {};
    const int dev = current_device();
    if (!configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
        if (e != cudaSuccess) return e;
        configured[dev] = true;
    }
    const int sm_count = device_sm_count();
    kern<<<a.n_items < sm_count ? a.n_items : sm_count, PG_THREADS, smem, st>>>(maps, a);
    return cudaGetLastError();
}

cudaError_t gemm_student_grad(const __nv_bfloat16* S, size_t M, int Ds, const __nv_bfloat16* Ghi, const __nv_bfloat16* Glo,
                              const float* gdir, const float* corr, const float* scale_ptr, float scale_host, void* out,
                              int out_is_bf16, int gap_period, int gap_valid, cudaStream_t st, const __nv_bfloat16* S_lo) {
    // dense bf16 students with a bf16 gradient (the training configuration): persistent kernel; CLS-stripped views (gapped rows),
    // fp32 gradients and split-bf16 students (three terms) keep the one-tile-per-CTA kernel below
    if (!S_lo && !gap_period && out_is_bf16 && Ds % 8 == 0 && M < (size_t(1) << 31) - 128)
        return student_grad_persistent(S, M, Ds, Ghi, Glo, gdir, corr, scale_ptr, scale_host, static_cast<__nv_bfloat16*>(out), st);
    GemmMaps maps;
    memset(&maps, 0, sizeof maps);
    if (make_map(&maps.a[0], S, Ds, M, 1, Ds, M * Ds, 128)) return cudaErrorInvalidValue;
    if (S_lo && make_map(&maps.a[1], S_lo, Ds, M, 1, Ds, M * Ds, 128)) return cudaErrorInvalidValue;
    if (make_map(&maps.b[0], Ghi, Ds, Ds, 1, Ds, static_cast<uint64_t>(Ds) * Ds, CfgStudentGrad::kBN)) return cudaErrorInvalidValue;
    if (make_map(&maps.b[1], Glo, Ds, Ds, 1, Ds, static_cast<uint64_t>(Ds) * Ds, CfgStudentGrad::kBN)) return cudaErrorInvalidValue;
    GemmArgs a;
    memset(&a, 0, sizeof a);
    a.kb_total = cdiv(Ds, GEMM_BK);
    a.out = out; a.ld_out = Ds; a.rows_valid = static_cast<int>(M); a.cols_valid = Ds;
    a.aux0 = gdir; a.aux1 = corr; a.aux2 = scale_ptr; a.alpha = scale_host; a.beta = out_is_bf16 ? 1.f : 0.f;
    a.gap_period = gap_period; a.gap_valid = gap_valid;
    static_assert(CfgStudentGrad3::kBN == CfgStudentGrad::kBN, "same tiles");
    if (S_lo) return launch<CfgStudentGrad3, EpiStudentGrad>(maps, a, dim3(cdiv(Ds, CfgStudentGrad::kBN), cdiv(M, 128), 1), st);
    return launch<CfgStudentGrad, EpiStudentGrad>(maps, a, dim3(cdiv(Ds, CfgStudentGrad::kBN), cdiv(M, 128), 1), st);
}

// ---------------------------------------------------------------------------------------------------
// polar_gemm: one CTA per problem, run-time tile sizes (polar_gemm.cuh)
// ---------------------------------------------------------------------------------------------------
cudaError_t polar_gemm(bool b_mn, const SplitMat& A, const SplitMat& B, int batches, PolarGemmArgs& a, cudaStream_t st) {
    const int m_rows = A.rows, K = a.k_override > 0 ? a.k_override : A.inner;
    const int n_cols = a.n_override > 0 ? a.n_override : (b_mn ? B.inner : B.rows);
    if (m_rows < 1 || n_cols < 1 || n_cols > (b_mn ? B.inner : B.rows) || K < 1 || K > A.inner || (b_mn ? B.rows : B.inner) < K) {
        snprintf(g_gemm_err, sizeof g_gemm_err, "polar_gemm: inconsistent sizes m=%d n=%d k=%d", m_rows, n_cols, K);
        return cudaErrorInvalidValue;
    }
    a.m_rows = m_rows; a.n_cols = n_cols; a.k_total = K;
    a.n_mt = (m_rows + 127) / 128;
    // column tiles: one tile of up to 256 columns, or equal tiles of a multiple of 64 columns (the auxiliary-tile epilogue
    // keeps a whole tile of the auxiliary matrix per warp in shared memory: 128 columns at most there)
    const int max_tile = a.aux_mode ? 128 : 256;
    if (n_cols <= (a.aux_mode ? 208 : max_tile)) {
        a.n_nt = 1;
        a.bn_mma = (n_cols + 15) / 16 * 16;
    } else {
        a.n_nt = (n_cols + max_tile - 1) / max_tile;
        a.bn_mma = ((n_cols + a.n_nt - 1) / a.n_nt + 63) / 64 * 64;
        a.n_nt = (n_cols + a.bn_mma - 1) / a.bn_mma;
    }
    a.n_items = batches * a.n_mt * a.n_nt;
    a.n_batches = batches;
    if ((a.trace && 4 * a.n_mt * a.n_nt > a.fro_slots) || (a.norm2 && a.fro_slots < 1)) {
        snprintf(g_gemm_err, sizeof g_gemm_err, "polar_gemm: %d partial-trace slots for %d x %d tiles", a.fro_slots, a.n_mt, a.n_nt);
        return cudaErrorInvalidValue;
    }
    a.b_groups = (a.bn_mma + 63) / 64;
    PolarGemmMaps maps;
    memset(&maps, 0, sizeof maps);
    const __nv_bfloat16* ap[2] = {A.hi, A.lo};
    const __nv_bfloat16* bp[2] = {B.hi, B.lo};
    for (int i = 0; i < 2; ++i) {
        if (make_map_tiled(&maps.a[i], ap[i], A.rows, (A.inner + 63) / 64, batches, A.batch_stride, 64)) return cudaErrorInvalidValue;
        // K-major B: one box of bn_mma rows per k-block; MN-major B: 64 (k) x 64 (n) boxes of the [K][n_cols] matrix
        if (make_map_tiled(&maps.b[i], bp[i], B.rows, (B.inner + 63) / 64, batches, B.batch_stride, b_mn ? 64 : a.bn_mma)) return cudaErrorInvalidValue;
    }
    if (a.epi == PG_EPI_SPLIT) {                       // TMA-store maps: 32-row x 64-column boxes of the tiled outputs
        const int ocb = (n_cols + 63) / 64;
        if (make_map_tiled(&maps.o[0], a.out_hi, m_rows, ocb, batches, a.out_stride, 32)) return cudaErrorInvalidValue;
        if (make_map_tiled(&maps.o[1], a.out_lo, m_rows, ocb, batches, a.out_stride, 32)) return cudaErrorInvalidValue;
        if (a.aux_mode) {
            if (make_map_tiled(&maps.o[2], a.aux_hi, m_rows, ocb, batches, a.out_stride, 32)) return cudaErrorInvalidValue;
            if (make_map_tiled(&maps.o[3], a.aux_lo, m_rows, ocb, batches, a.out_stride, 32)) return cudaErrorInvalidValue;
        }
    }
    if (a.epi == PG_EPI_THETA) {                       // row-major [m_rows][ld_out] outputs, 32 x 64 boxes, columns clipped at n_cols
        if (make_map(&maps.o[0], a.out_hi, n_cols, m_rows, batches, a.ld_out, a.out_stride, 32)) return cudaErrorInvalidValue;
        if (make_map(&maps.o[1], a.out_lo, n_cols, m_rows, batches, a.ld_out, a.out_stride, 32)) return cudaErrorInvalidValue;
    }
    if (a.a_alias_b && (b_mn || A.hi != B.hi || m_rows != n_cols)) {
        snprintf(g_gemm_err, sizeof g_gemm_err, "polar_gemm: a_alias_b needs the same K-major matrix on both sides");
        return cudaErrorInvalidValue;
    }
    if (a.a_alias_b && a.n_nt > 1) a.a_alias_b = 0;      // the A tile is only inside the B tile when one tile spans all columns
    const int b_bytes = b_mn ? a.b_groups * 8192 : a.bn_mma * 128;
    const int stage_bytes = (a.a_alias_b ? 0 : 2 * 16384) + 2 * b_bytes;
    const int kTail = 1024 /*alignment*/ + 1024 /*barriers*/ + 4 * 8192 /*epilogue staging*/ + (a.aux_mode ? 4 * 8192 * ((a.bn_mma + 63) / 64) : 0) /*aux tiles: every column block of an item*/ +
                      (a.epi == PG_EPI_THETA ? 4 * 2048 : 0) /*THETA: a and sqrt(a) of the tile's columns per epilogue warp*/;   // (the aliased A tile of the last rows reads up to 8 KB past its B tile: into the barrier / staging area, rows never used)
    int stages = (232448 - kTail) / stage_bytes;
    if (stages > 4) stages = 4;
    if (stages < 1) {
        snprintf(g_gemm_err, sizeof g_gemm_err, "polar_gemm: one stage (%d B) exceeds shared memory", stage_bytes);
        return cudaErrorInvalidValue;
    }
    a.stages = stages;
    const int smem = stages * stage_bytes + kTail;
    // epilogue kind -> kernel instantiation (polar_gemm.cuh); fp32 outputs leave as TMA stores (table index 4 = kind 6) when the
    // row pitch allows it
    int kind = a.epi == PG_EPI_F32 ? 3 : a.epi == PG_EPI_THETA ? 2 : a.aux_mode ? 1 : 0;
    if (kind == 3 && f32_tma_ok(a.out_f32, a.ld_f32, a.out_f32_stride)) {
        if (make_map_f32(&maps.o[0], a.out_f32, n_cols, m_rows, batches, a.ld_f32, a.out_f32_stride)) return cudaErrorInvalidValue;
        kind = 4;
    }
    using Kern = void (*)(const PolarGemmMaps, const PolarGemmArgs);
    static const Kern kerns[2][5] = {
        {polar_gemm_kernel<false, 0>, polar_gemm_kernel<false, 1>, polar_gemm_kernel<false, 2>, polar_gemm_kernel<false, 3>, polar_gemm_kernel<false, 6>},
        {polar_gemm_kernel<true, 0>, polar_gemm_kernel<true, 1>, polar_gemm_kernel<true, 2>, polar_gemm_kernel<true, 3>, polar_gemm_kernel<true, 6>}};
    const Kern kern = kerns[b_mn][kind];
    static bool configured[kMaxDevices][2][5] = {};
    const int dev = current_device();
    if (!configured[dev][b_mn][kind]) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
        if (e != cudaSuccess) return e;
        configured[dev][b_mn][kind] = true;
    }
    const int sm_count = device_sm_count();
    const int grid = a.n_items < sm_count ? a.n_items : sm_count;
    kern<<<grid, PG_THREADS, smem, st>>>(maps, a);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------
// polar_fused_abm: Bm = ca I + cb (rA) + cc (rA)^2 with A = T W^T kept on chip (polar_fused.cuh); D_s <= 192
// ---------------------------------------------------------------------------------------------------
bool polar_fused_supported(int n, int k) { return n <= 192 && k <= 256 && n >= 16; }
cudaError_t polar_fused_abm(const SplitMat& T, const SplitMat& W, const SplitMat& Bm, int batches, PolarFusedArgs& a, cudaStream_t st) {
    const int n = T.rows, K = T.inner;
    if (!polar_fused_supported(n, K) || W.rows != n || W.inner != K || Bm.rows != n || Bm.inner != n) {
        snprintf(g_gemm_err, sizeof g_gemm_err, "polar_fused_abm: unsupported sizes n=%d k=%d", n, K);
        return cudaErrorInvalidValue;
    }
    a.n = n; a.k_total = K; a.bn = (n + 15) / 16 * 16; a.rows_ld = (n + 63) / 64 * 64; a.n_mt = (n + 127) / 128; a.n_problems = batches;
    PolarFusedMaps maps;
    memset(&maps, 0, sizeof maps);
    const __nv_bfloat16* tp[2] = {T.hi, T.lo};
    const __nv_bfloat16* wp[2] = {W.hi, W.lo};
    __nv_bfloat16* op[2] = {Bm.hi, Bm.lo};
    for (int i = 0; i < 2; ++i) {
        if (make_map_tiled(&maps.t[i], tp[i], T.rows, (T.inner + 63) / 64, batches, T.batch_stride, 64)) return cudaErrorInvalidValue;
        if (make_map_tiled(&maps.w[i], wp[i], W.rows, (W.inner + 63) / 64, batches, W.batch_stride, a.bn)) return cudaErrorInvalidValue;
        if (make_map_tiled(&maps.o[i], op[i], Bm.rows, (Bm.inner + 63) / 64, batches, Bm.batch_stride, 32, 32)) return cudaErrorInvalidValue;
    }
    const int stage_bytes = 2 * a.rows_ld * 128 + 2 * a.bn * 128;
    const int ring_bytes = PF_STAGES * stage_bytes;
    const int copy_bytes = 2 * ((n + 63) / 64) * a.rows_ld * 128;
    if (copy_bytes + 8192 > ring_bytes) {                      // (tile 1 of the last block reads up to 64 rows past the copy)
        snprintf(g_gemm_err, sizeof g_gemm_err, "polar_fused_abm: operand copy (%d B) does not fit the ring (%d B)", copy_bytes, ring_bytes);
        return cudaErrorInvalidValue;
    }
    const int smem = ring_bytes + 1024 /*alignment*/ + 1024 /*barriers*/ + 8 * 4096 /*staging*/;
    if (smem > 232448) {
        snprintf(g_gemm_err, sizeof g_gemm_err, "polar_fused_abm: %d B of shared memory needed", smem);
        return cudaErrorInvalidValue;
    }
    static bool configured[kMaxDevices] = {false};
    const int dev = current_device();
    if (!configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(polar_fused_abm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
        if (e != cudaSuccess) return e;
        configured[dev] = true;
    }
    const int sm_count = device_sm_count();
    const int grid = batches < sm_count ? batches : sm_count;
    polar_fused_abm_kernel<<<grid, PF_THREADS, smem, st>>>(maps, a);
    return cudaGetLastError();
}

// variant 0: C[M][N] = A[M][K] B[N][K]^T          (both K-major)
// variant 1: C[M][N] = A[K][M]^T B[K][N]          (both MN-major; split-K + atomics; C pre-zeroed)
// variant 2: C[M][N] = A[M][K] B[K][N]            (A K-major, B MN-major)
// variant 3: C[M][M] = A A^T + A B^T + B A^T      (token_gram path: A = hi [M][K], B = lo [M][K])
cudaError_t gemm_selftest(int variant, const __nv_bfloat16* A, const __nv_bfloat16* B, float* C, int M, int N, int K,
                          cudaStream_t st) {
    GemmMaps maps;
    memset(&maps, 0, sizeof maps);
    GemmArgs a;
    memset(&a, 0, sizeof a);
    a.out = C; a.ld_out = N; a.rows_valid = M; a.cols_valid = N; a.alpha = 1.f;
    if (variant == 0) {
        if (make_map(&maps.a[0], A, K, M, 1, K, static_cast<uint64_t>(M) * K, 128)) return cudaErrorInvalidValue;
        if (make_map(&maps.b[0], B, K, N, 1, K, static_cast<uint64_t>(N) * K, CfgTestTN::kBN)) return cudaErrorInvalidValue;
        a.kb_total = cdiv(K, GEMM_BK);
        return launch<CfgTestTN, EpiStoreF32>(maps, a, dim3(cdiv(N, CfgTestTN::kBN), cdiv(M, 128), 1), st);
    }
    if (variant == 1) {
        if (make_map(&maps.a[0], A, M, K, 1, M, static_cast<uint64_t>(M) * K, 64)) return cudaErrorInvalidValue;
        if (make_map(&maps.b[0], B, N, K, 1, N, static_cast<uint64_t>(N) * K, 64)) return cudaErrorInvalidValue;
        a.kb_total = cdiv(K, GEMM_BK);
        a.kb_per_split = 4;
        a.n_splits = cdiv(a.kb_total, a.kb_per_split);
        a.a_batched = 1; a.b_batched = 1;
        return launch<CfgGram, EpiAtomicAddF32>(maps, a, dim3(cdiv(N, CfgGram::kBN), cdiv(M, CfgGram::kMT * 128), a.n_splits), st);
    }
    if (variant == 2) {
        if (make_map(&maps.a[0], A, K, M, 1, K, static_cast<uint64_t>(M) * K, 128)) return cudaErrorInvalidValue;
        if (make_map(&maps.b[0], B, N, K, 1, N, static_cast<uint64_t>(N) * K, 64)) return cudaErrorInvalidValue;
        a.kb_total = cdiv(K, GEMM_BK);
        return launch<CfgTheta, EpiStoreF32>(maps, a, dim3(cdiv(N, CfgTheta::kBN), cdiv(M, CfgTheta::kMT * 128), 1), st);
    }
    if (variant == 3) {
        return gemm_token_gram(A, B, 1, M, K, C, st);
    }
    return cudaErrorInvalidValue;
}

}  // namespace basd
