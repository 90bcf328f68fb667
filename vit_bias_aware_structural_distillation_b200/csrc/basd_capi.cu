// C-ABI entry points (include/basd_b200.h): workspace layout and kernel orchestration of the four phases.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "../../include/basd_b200.h"
#include "spectral.h"

using namespace basd;

static thread_local char g_err[512] = "";
static int fail(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return 1;
}
#define CK(expr)                                                                                             \
    do {                                                                                                     \
        cudaError_t _e = (expr);                                                                             \
        if (_e != cudaSuccess)                                                                               \
            return fail("%s:%d %s -> %s; %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e), gemm_last_error()); \
    } while (0)

extern "C" const char* basd_last_error(void) { return g_err; }

// ---------------------------------------------------------------------------------------------- live kernel timing
// Optional CUDA-event brackets around each kernel group, recorded on the launching stream inside the caller's timed
// region (bench.py's roofline numbers come from here, not from a profiler).  Also counts kernel launches.
// The launch counter is atomic; the event brackets are a single-caller measurement facility (basd_timing_enable is off
// by default and documented as not re-entrant in include/basd_b200.h) - the compute entry points themselves keep no
// mutable process state.
namespace {
constexpr int kTimeSlots = 18;
constexpr int kMaxPairs = 2048;
const char* kSlotNames[kTimeSlots] = {"importance_rows", "split_pack", "project", "gram", "colsum", "pooled_eig", "angles",
                                      "importance_mix", "mix_teacher", "token_gram", "polar_prep", "loss_reduce", "theta_apply",
                                      "wgrad_dots", "selector_bwd", "student_grad", "polar_gemm", "polar_finish"};
struct TimeSlot { cudaEvent_t ev[kMaxPairs][2]; int created = 0; int used = 0; };
TimeSlot g_slots[kTimeSlots];
bool g_timing = false;
std::atomic<long long> g_launches{0};
struct Scope {
    int slot; cudaStream_t st; bool on;
    Scope(int slot_, cudaStream_t st_, int n_launches) : slot(slot_), st(st_), on(false) {
        g_launches += n_launches;
        TimeSlot& t = g_slots[slot];
        if (!g_timing || t.used >= kMaxPairs) return;
        if (t.used >= t.created) { cudaEventCreate(&t.ev[t.created][0]); cudaEventCreate(&t.ev[t.created][1]); ++t.created; }
        cudaEventRecord(t.ev[t.used][0], st);
        on = true;
    }
    ~Scope() { if (on) { TimeSlot& t = g_slots[slot]; cudaEventRecord(t.ev[t.used][1], st); ++t.used; } }
};
}  // namespace
extern "C" void basd_timing_enable(int on) { g_timing = on != 0; }
extern "C" void basd_timing_reset(void) { for (auto& t : g_slots) t.used = 0; g_launches = 0; }
extern "C" long long basd_launch_count(void) { return g_launches.load(); }
extern "C" int basd_timing_slots(void) { return kTimeSlots; }
extern "C" const char* basd_timing_name(int slot) { return (slot >= 0 && slot < kTimeSlots) ? kSlotNames[slot] : ""; }
// total milliseconds and number of timed brackets of a slot (synchronises on the recorded events)
extern "C" int basd_timing_read(int slot, float* ms_total, int* brackets) {
    if (slot < 0 || slot >= kTimeSlots || !ms_total || !brackets) return fail("bad timing slot");
    TimeSlot& t = g_slots[slot];
    float tot = 0.f;
    for (int i = 0; i < t.used; ++i) {
        float ms = 0.f;
        cudaEventSynchronize(t.ev[i][1]);
        if (cudaEventElapsedTime(&ms, t.ev[i][0], t.ev[i][1]) == cudaSuccess) tot += ms;
    }
    *ms_total = tot; *brackets = t.used;
    return 0;
}
#define TIMED(slot, n, stmt) do { Scope _sc(slot, st, n); stmt; } while (0)
// brackets usable from the other translation units (spectral.h: TimingScope)
namespace basd {
TimingScope::TimingScope(int slot, cudaStream_t st, int n_launches) : impl(new Scope(slot, st, n_launches)) {}
TimingScope::~TimingScope() { delete static_cast<Scope*>(impl); }
}  // namespace basd
extern "C" const char* basd_version(void) { return "basd_b200 0.1 (sm_100a)"; }
extern "C" int basd_polar_steps(void) { return basd::polar_steps(); }
namespace basd { int polar_launches_per_step(int Ds, int Ns); }
extern "C" int basd_polar_launches_per_step(int Ds, int Ns) { return basd::polar_launches_per_step(Ds, Ns); }

namespace {

// Which space the Procrustes polar iteration runs in (polar.cu):
//   kPathFeature : student features (D_s x N_s iterate); needs rank(C) = D_s, i.e. D_s <= min(N_s, N_t) - 1
//   kPathTeacherTokens : teacher tokens (N_t x D_s iterate), D_s > min(N_s, N_t) - 1 and N_t <= N_s
enum { kPathFeature = 0, kPathTeacherTokens = 1 };
int polar_path(const basd_shape& s) {
    const int rank_t = (s.Nt < s.Ns ? s.Nt : s.Ns) - 1;
    return s.Ds <= rank_t ? kPathFeature : kPathTeacherTokens;
}

struct Layout {
    size_t rows, pt_hi, pt_lo, tpk, spk, z, stats, ranks, sweeps, evals, evecs_km, evecs_cm, d2, w, cosv, gamma, ang_scr, a, ssum,
        tbar_hi, tbar_lo, ktt, gdir, theta, gwt, loss_b, dbg, geo_i, gw, gam_hi, gam_lo, corr,
        pw, pw2, pt, pa, pb, pkt, psw, gsw, pvec, pscal, pfro, pres, theta_lo, dtm, eig_scr, gram_part, colsum_part, gw_part,
        vfg, vfgt, vginvc, vginvt, vx0, vx1, vx2, vh, vm2, vginv, vthraw, vftf, total;
    int NsPad, Np, path, Nk, Dsp, dtm_split;    // Nk: token rows of the mixed teacher / Theta (Ns, or Nt in the teacher-token form)
};

size_t align_up(size_t x) { return (x + 1023) & ~static_cast<size_t>(1023); }

Layout make_layout(const basd_shape& s) {
    Layout L;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes); return o; };
    const size_t B = s.B, Ns = s.Ns, Nt = s.Nt, Ds = s.Ds, Dt = s.Dt, Lt = s.Lt, P = s.P;
    L.path = polar_path(s);
    const bool vt = L.path == kPathTeacherTokens;
    // token-space form: the mixed teacher stays on its own grid when that is the coarser one (the resampling is folded into F);
    // a FINER teacher grid (N_t > N_s) is resampled to the student's first - rank(C) = N_s - 1 either way
    const size_t Nk = vt ? (Nt < Ns ? Nt : Ns) : Ns;
    L.Nk = static_cast<int>(Nk);
    L.NsPad = static_cast<int>((Nk + 7) / 8 * 8);
    L.Dsp = static_cast<int>((Ds + 15) / 16 * 16 + 8);
    L.rows = take(4 * Lt * B * Nt);
    L.pt_hi = take(2 * Ds * Dt);
    L.pt_lo = take(2 * Ds * Dt);
    // fp32 tokens are packed to dense bf16 [layer or point][B][N][D]; split-bf16 pairs as a hi block then a lo block
    const size_t pack = s.act_dtype == BASD_DTYPE_F32 ? 1 : s.act_dtype == BASD_DTYPE_F32_SPLIT ? 2 : 0;
    L.tpk = take(pack * 2 * Lt * B * Nt * Dt);
    L.spk = take(pack * 2 * P * B * Ns * Ds);
    L.z = take(2 * 2 * Lt * B * (Nt + 1) * Ds);    // projected teacher tokens, split pair: hi block then lo block (rows of a CLS-stripped view: B (Nt + 1) - 1)
    L.stats = take(4 * (Lt + P) * (Ds * Ds + Ds));
    L.ranks = take(4 * Lt);
    L.sweeps = take(4 * (2 * Lt + P));
    L.evals = take(4 * (Lt + P) * Ds);
    L.evecs_km = take(4 * (Lt + P) * Ds * Ds);
    L.evecs_cm = take(4 * (Lt + P) * Ds * Ds);
    L.eig_scr = take(4 * pooled_eig_scratch_floats(s.Ds, 2 * s.Lt + s.P));   // D_s > 224: eigenproblem matrices in global memory
    // per-CTA partial results of the split-K Grams, column sums and weight-gradient dots (each summed in a fixed order)
    {
        // (sized for the CLS-stripped-view variants too: B (Nt + 1) projected rows; 64-row blocks per sample for the student)
        const size_t gp_t = gemm_gram_part_floats(B * (Nt + 1), s.Ds, s.Lt), gp_s = gemm_gram_part_floats(B * ((Ns + 63) / 64 * 64), s.Ds, s.P);
        L.gram_part = take(4 * (gp_t > gp_s ? gp_t : gp_s));
        const size_t cp_a = colsum_part_floats(s.Lt + s.P, B * Nt, s.Ds), cp_t = colsum_part_floats(s.Lt, B * (Nt + 1), s.Ds),
                     cp_s = colsum_part_floats(s.P, B * Ns, s.Ds);
        const size_t cp = cp_a > cp_t ? (cp_a > cp_s ? cp_a : cp_s) : (cp_t > cp_s ? cp_t : cp_s);
        L.colsum_part = take(4 * cp);
        L.gw_part = take(4 * wgrad_part_floats(s.P, s.Lt));
    }
    L.d2 = take(4 * P * Lt);
    L.w = take(4 * P * Lt);
    L.cosv = take(4 * P * Lt * Ds);
    L.gamma = take(4 * P * Lt * Ds * Ds);
    L.ang_scr = take(4 * P * Lt * 8 * Ds * Ds);
    L.a = take(4 * P * B * Ns);
    L.ssum = take(4 * P * B);
    L.tbar_hi = take(2 * P * B * Nk * Dt);
    L.tbar_lo = take(2 * P * B * Nk * Dt);
    L.ktt = take(4 * P * B * Nk * Nk);
    // Newton-Schulz polar iteration (polar.cu): split-bf16 matrices per (point, sample) problem, hi then lo
    L.Np = static_cast<int>((Ns + 63) / 64 * 64);      // column-block tiled storage: columns padded to 64
    const size_t nprob = P * B, Np = L.Np;
    const size_t Dp = (Ds + 63) / 64 * 64;
    const size_t Mp = (Nk + 63) / 64 * 64, Xp = (static_cast<size_t>(L.Dsp) + 63) / 64 * 64;
    L.pw = take(vt ? 0 : 2 * 2 * nprob * Ds * Np);
    L.pw2 = take(vt ? 0 : 2 * 2 * nprob * Ds * Np);
    L.pt = take(vt ? 0 : 2 * 2 * nprob * Ds * Np);
    L.pa = take(vt ? 2 * 2 * nprob * Nk * Mp : 2 * 2 * nprob * Ds * Dp);       // A  (core x core)
    L.pb = take(vt ? 2 * 2 * nprob * Nk * Mp : 2 * 2 * nprob * Ds * Dp);       // Bm
    L.pkt = take(vt ? 0 : 2 * 2 * nprob * Ns * Np);
    L.psw = take(2 * 2 * nprob * Ns * Dp);
    L.vfg = take(vt ? 2 * 2 * nprob * Ns * Mp : 0);
    L.vfgt = take(vt ? 2 * 2 * nprob * Nk * Np : 0);
    L.vginvc = take(vt ? 2 * 2 * nprob * Nk * Mp : 0);
    L.vginvt = take(vt ? 2 * 2 * nprob * Nk * Mp : 0);
    L.vx0 = take(vt ? 2 * 2 * nprob * Nk * Xp : 0);
    L.vx1 = take(vt ? 2 * 2 * nprob * Nk * Xp : 0);
    L.vx2 = take(vt ? 2 * 2 * nprob * Nk * Xp : 0);
    L.vh = take(vt ? 2 * 2 * nprob * Nk * Mp : 0);
    L.vm2 = take(vt ? 2 * 2 * nprob * Nk * Mp : 0);
    L.vginv = take(vt ? 4 * nprob * Nk * Nt : 0);
    L.vthraw = take(vt ? 4 * nprob * Nk * Nt : 0);
    L.vftf = take(vt ? 4 * nprob * Nk * Nt : 0);
    L.gsw = take(4 * nprob * Ns * Ds);
    L.pvec = take(4 * nprob * 4 * Ns);
    L.pscal = take(4 * nprob * 4);
    L.pfro = take(4 * nprob * polar_fro_slots(vt ? L.Nk : s.Ds));
    L.pres = take(4 * nprob * polar_fro_slots(vt ? L.Nk : s.Ds));
    L.gdir = take(4 * P * B * Ns * Ds);
    L.theta = take(2 * P * B * Nk * L.NsPad);
    L.theta_lo = take(2 * P * B * Nk * L.NsPad);
    // Gradient w.r.t. the mixed teacher: one bf16 at the BASELINE sizes; a split pair (hi block then lo block) when the
    // tensor is small - its rounding error reaches the temperature gradients as noise ~ 2^-9 / sqrt(elements) amplified by the
    // cancellation between layers: 5e-4 at 2.5e4 elements, 1e-5 at the 3.8e7 of cfg2
    L.dtm_split = (P * B * Nk * Dt) < (size_t(1) << 24) ? 1 : 0;
    L.dtm = take((L.dtm_split ? 2 : 1) * 2 * P * B * Nk * Dt);
    L.gwt = take(4 * P * B * Ns);
    L.loss_b = take(4 * P * B);
    L.dbg = take(4 * P * B * 5);
    L.geo_i = take(4 * (P + 2));                          // per-point means, their mean, largest polar residual
    L.gw = take(4 * P * Lt);
    L.gam_hi = take(2 * P * Ds * Ds);
    L.gam_lo = take(2 * P * Ds * Ds);
    L.corr = take(4 * P * Ds);
    L.total = off;
    return L;
}

int check_shape(const basd_shape& s) {
    if (s.B < 1 || s.Ns < 2 || s.Nt < 1 || s.Lt < 1 || s.P < 1) return fail("invalid shape");
    if (s.world_size < 1) return fail("world_size must be >= 1");
    if (s.act_dtype < BASD_DTYPE_F32 || s.act_dtype > BASD_DTYPE_F32_SPLIT)
        return fail("basd_shape.act_dtype must be BASD_DTYPE_F32 (0), BASD_DTYPE_BF16 (1) or BASD_DTYPE_F32_SPLIT (2), got %d", s.act_dtype);
    if (s.attn_dtype != BASD_DTYPE_F32 && s.attn_dtype != BASD_DTYPE_BF16)
        return fail("basd_shape.attn_dtype must be BASD_DTYPE_F32 (0) or BASD_DTYPE_BF16 (1), got %d", s.attn_dtype);
    if (s.has_cls < 0 || s.has_cls > BASD_ATTN_QUERY_MEAN) return fail("basd_shape.has_cls must be 0, 1 or BASD_ATTN_QUERY_MEAN (2), got %d", s.has_cls);
    if (s.mode < BASD_MODE_LOSS || s.mode > BASD_MODE_SELECTOR) return fail("unknown basd_shape.mode %d", s.mode);
    if (s.mode == BASD_MODE_PAIR && (s.Lt != 1 || s.P != 1)) return fail("BASD_MODE_PAIR takes one student and one teacher tensor (Lt = P = 1)");
    if (s.P > BASD_MAX_POINTS || s.Lt > BASD_MAX_LAYERS) return fail("P <= %d and Lt <= %d required", BASD_MAX_POINTS, BASD_MAX_LAYERS);
    if (s.Ds % 8 || s.Dt % 8) return fail("Ds and Dt must be multiples of 8 (16-byte rows), got %d, %d", s.Ds, s.Dt);
    if (s.Ds > 1024) return fail("Ds=%d > 1024 is not supported", s.Ds);
    if (s.polar_steps != 0 && (s.polar_steps < kPolarStepsMin || s.polar_steps > kPolarStepsMax))
        return fail("polar_steps must be 0 (default %d) or %d..%d, got %d", kPolarStepsDefault, kPolarStepsMin, kPolarStepsMax, s.polar_steps);
    if (polar_path(s) == kPathTeacherTokens) {
        // rank(C) = min(Ns, Nt) - 1 < Ds: the polar iteration runs in token space, on the coarser of the two token grids
        const int nk = s.Nt < s.Ns ? s.Nt : s.Ns;
        if (nk > kVtMaxTokens)
            return fail("Ds=%d > min(Ns, Nt) - 1 with min(Ns, Nt) = %d > %d: the token-space Cholesky factor no longer fits shared memory", s.Ds, nk, kVtMaxTokens);
        if (s.Nt < 2) return fail("Nt >= 2 required");
    }
    return 0;
}

bool dense3(const int64_t* st, int N, int D) { return st[2] == 1 && st[1] == D && st[0] == static_cast<int64_t>(N) * D; }
// the CLS-stripped view out[:, 1:, :] of a dense [B][N+1][D] tensor (trainer.py:29, teacher.py:157): consumed in place
bool cls_view3(const int64_t* st, int N, int D) { return st[2] == 1 && st[1] == D && st[0] == static_cast<int64_t>(N + 1) * D; }

struct Resolved {
    const __nv_bfloat16* teacher[BASD_MAX_LAYERS];
    const __nv_bfloat16* student[BASD_MAX_POINTS];
    const __nv_bfloat16* teacher_lo[BASD_MAX_LAYERS];     // split-bf16 tokens (BASD_DTYPE_F32_SPLIT): lo halves; null otherwise
    const __nv_bfloat16* student_lo[BASD_MAX_POINTS];
    long long teacher_bs, student_bs;       // batch strides in elements
    int teacher_gap, student_gap;           // 1: rows of the tensor read as a flat matrix carry one foreign row between samples
};

// After phase 1 the bf16, dense versions of the tokens are either the inputs themselves or the packed copies (hi and lo
// halves of split pairs).
bool packs(const basd_shape& s) { return s.act_dtype == BASD_DTYPE_F32 || s.act_dtype == BASD_DTYPE_F32_SPLIT; }
int resolve(const basd_shape& s, const basd_inputs& in, uint8_t* ws, const Layout& L, Resolved* r) {
    const bool pack = packs(s), split = s.act_dtype == BASD_DTYPE_F32_SPLIT;
    const size_t t_block = static_cast<size_t>(s.Lt) * s.B * s.Nt * s.Dt, s_block = static_cast<size_t>(s.P) * s.B * s.Ns * s.Ds;
    memset(r->teacher_lo, 0, sizeof r->teacher_lo);
    memset(r->student_lo, 0, sizeof r->student_lo);
    r->teacher_bs = static_cast<long long>(s.Nt) * s.Dt; r->student_bs = static_cast<long long>(s.Ns) * s.Ds;
    r->teacher_gap = 0; r->student_gap = 0;
    if (!pack) {
        // bf16 tokens are consumed in place by TMA: dense [B,N,D], or the CLS-stripped view of a dense [B,N+1,D] tensor
        if (cls_view3(in.teacher_strides, s.Nt, s.Dt)) { r->teacher_gap = 1; r->teacher_bs = in.teacher_strides[0]; }
        else if (!dense3(in.teacher_strides, s.Nt, s.Dt))
            return fail("bf16 teacher tokens must be dense [B,N,D] or a [:,1:,:] view of a dense [B,N+1,D] tensor (strides %lld,%lld,%lld)",
                        (long long)in.teacher_strides[0], (long long)in.teacher_strides[1], (long long)in.teacher_strides[2]);
        if (cls_view3(in.student_strides, s.Ns, s.Ds)) { r->student_gap = 1; r->student_bs = in.student_strides[0]; }
        else if (!dense3(in.student_strides, s.Ns, s.Ds))
            return fail("bf16 student tokens must be dense [B,N,D] or a [:,1:,:] view of a dense [B,N+1,D] tensor (strides %lld,%lld,%lld)",
                        (long long)in.student_strides[0], (long long)in.student_strides[1], (long long)in.student_strides[2]);
    }
    for (int j = 0; j < s.Lt; ++j) {
        if (!in.teacher[j] || (!in.attn[j] && s.mode != BASD_MODE_SELECTOR)) return fail("null teacher/attention pointer at layer %d", j);
        r->teacher[j] = pack ? reinterpret_cast<const __nv_bfloat16*>(ws + L.tpk) + static_cast<size_t>(j) * s.B * s.Nt * s.Dt
                             : reinterpret_cast<const __nv_bfloat16*>(in.teacher[j]);
        if (reinterpret_cast<uintptr_t>(r->teacher[j]) & 15) return fail("teacher tensor %d not 16-byte aligned", j);
        if (split) r->teacher_lo[j] = r->teacher[j] + t_block;
    }
    for (int i = 0; i < s.P; ++i) {
        if (!in.student[i]) return fail("null student pointer at point %d", i);
        r->student[i] = pack ? reinterpret_cast<const __nv_bfloat16*>(ws + L.spk) + static_cast<size_t>(i) * s.B * s.Ns * s.Ds
                             : reinterpret_cast<const __nv_bfloat16*>(in.student[i]);
        if (reinterpret_cast<uintptr_t>(r->student[i]) & 15) return fail("student tensor %d not 16-byte aligned", i);
        if (split) r->student_lo[i] = r->student[i] + s_block;
    }
    return 0;
}

}  // namespace

extern "C" int basd_workspace_bytes(const basd_shape* shape, size_t* bytes) {
    if (!shape || !bytes) return fail("null argument");
    if (check_shape(*shape)) return 1;
    *bytes = make_layout(*shape).total;
    return 0;
}

extern "C" int basd_view(const basd_shape* shape, void* workspace, const char* name, void** ptr, size_t* count) {
    if (!shape || !workspace || !name || !ptr || !count) return fail("null argument");
    const basd_shape& s = *shape;
    const Layout L = make_layout(s);
    uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
    const size_t B = s.B, Ns = s.Ns, Nt = s.Nt, Ds = s.Ds, Lt = s.Lt, P = s.P;
    struct E { const char* n; size_t off; size_t cnt; } table[] = {
        {"stats", L.stats, (Lt + P) * (Ds * Ds + Ds)}, {"gw", L.gw, P * Lt}, {"ranks", L.ranks, Lt}, {"w", L.w, P * Lt},
        {"d2", L.d2, P * Lt}, {"geo_i", L.geo_i, P + 1}, {"polar_resid", L.geo_i + 4 * (P + 1), 1}, {"loss_b", L.loss_b, P * B}, {"rows", L.rows, Lt * B * Nt},
        {"a", L.a, P * B * Ns}, {"evals", L.evals, (Lt + P) * Ds}, {"cos", L.cosv, P * Lt * Ds}, {"dbg", L.dbg, P * B * 5},
        {"gdir", L.gdir, P * B * Ns * Ds}, {"ktt", L.ktt, P * B * L.Nk * L.Nk}, {"sweeps", L.sweeps, 2 * Lt + P},
        {"gamma", L.gamma, P * Lt * Ds * Ds}, {"gwt", L.gwt, P * B * Ns}, {"evecs", L.evecs_km, (Lt + P) * Ds * Ds},
        {"corr", L.corr, P * Ds}, {"ssum", L.ssum, P * B},
        // polar iteration state (bf16 pairs: count is in bf16 elements, hi block then lo block)
        {"polar_w", (polar_steps() % 2) ? L.pw2 : L.pw, 2 * P * B * Ds * L.Np}, {"polar_kt", L.pkt, 2 * P * B * Ns * L.Np},
        {"polar_sw", L.psw, 2 * P * B * Ns * ((Ds + 63) / 64 * 64)}, {"polar_a", L.pa, 2 * P * B * Ds * ((Ds + 63) / 64 * 64)}, {"polar_gsw", L.gsw, P * B * Ns * Ds}, {"polar_fro2", L.pfro, P * B * static_cast<size_t>(polar_fro_slots(L.path == kPathTeacherTokens ? L.Nk : s.Ds))},
        {"theta", L.theta, P * B * L.Nk * L.NsPad},
    };
    for (const E& e : table)
        if (!strcmp(e.n, name)) { *ptr = ws + e.off; *count = e.cnt; return 0; }
    return fail("unknown view '%s'", name);
}

extern "C" int basd_forward_stats(const basd_shape* shape, const basd_inputs* in_, void* workspace, void* stream) {
    if (!shape || !in_ || !workspace) return fail("null argument");
    const basd_shape& s = *shape;
    const basd_inputs& in = *in_;
    if (check_shape(s)) return 1;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
    const Layout L = make_layout(s);
    const size_t Mt = static_cast<size_t>(s.B) * s.Nt, Ms = static_cast<size_t>(s.B) * s.Ns;
    const size_t stat_stride = static_cast<size_t>(s.Ds) * s.Ds + s.Ds;
    float* stats = reinterpret_cast<float*>(ws + L.stats);

    const bool selector = s.mode != BASD_MODE_PAIR;            // the pooled statistics feed the layer selector only
    if (selector && (!in.proj_s || !in.proj_t || !in.log_temperatures)) return fail("null proj_s / proj_t / log_temperatures");
    if (s.mode != BASD_MODE_SELECTOR) {
        PtrTable attn;
        memset(&attn, 0, sizeof attn);
        for (int j = 0; j < s.Lt; ++j) attn.p[j] = in.attn[j];
        long long as[4] = {in.attn_strides[0], in.attn_strides[1], in.attn_strides[2], in.attn_strides[3]};
        TIMED(0, 1, CK(launch_importance_rows(attn, s.attn_dtype == BASD_DTYPE_BF16, s.Lt, s.B, s.H, s.Nt, s.has_cls, as,
                                  reinterpret_cast<float*>(ws + L.rows), st)));
    }
    __nv_bfloat16* pt_hi = reinterpret_cast<__nv_bfloat16*>(ws + L.pt_hi);
    __nv_bfloat16* pt_lo = reinterpret_cast<__nv_bfloat16*>(ws + L.pt_lo);
    {
        Scope sc(1, st, 1 + (packs(s) ? s.Lt + s.P : 0));
        if (selector) CK(launch_split_bf16(in.proj_t, pt_hi, pt_lo, static_cast<size_t>(s.Ds) * s.Dt, st));
        if (packs(s)) {
            // fp32 tokens: rounded to bf16, or (BASD_DTYPE_F32_SPLIT) kept as split pairs, lo halves one block behind the hi halves
            const bool split = s.act_dtype == BASD_DTYPE_F32_SPLIT;
            __nv_bfloat16* tpk = reinterpret_cast<__nv_bfloat16*>(ws + L.tpk);
            __nv_bfloat16* spk = reinterpret_cast<__nv_bfloat16*>(ws + L.spk);
            const size_t t_block = static_cast<size_t>(s.Lt) * Mt * s.Dt, s_block = static_cast<size_t>(s.P) * Ms * s.Ds;
            for (int j = 0; j < s.Lt; ++j)
                CK(launch_pack_bf16(in.teacher[j], 0, in.teacher_strides[0], in.teacher_strides[1], in.teacher_strides[2], s.B, s.Nt, s.Dt,
                                    tpk + static_cast<size_t>(j) * Mt * s.Dt, split ? tpk + t_block + static_cast<size_t>(j) * Mt * s.Dt : nullptr, st));
            for (int i = 0; i < s.P; ++i)
                CK(launch_pack_bf16(in.student[i], 0, in.student_strides[0], in.student_strides[1], in.student_strides[2], s.B, s.Ns, s.Ds,
                                    spk + static_cast<size_t>(i) * Ms * s.Ds, split ? spk + s_block + static_cast<size_t>(i) * Ms * s.Ds : nullptr, st));
        }
    }
    Resolved r;
    if (resolve(s, in, ws, L, &r)) return 1;
    if (!selector) return 0;
    // A CLS-stripped teacher view is projected as the dense matrix of B (Nt + 1) - 1 rows it is in memory; the rows that
    // belong to no sample leave the projection as zeros, so the Gram and the column sums below are those of the B Nt tokens.
    const size_t Mt_dense = Mt;
    const size_t Mt_rows = r.teacher_gap ? static_cast<size_t>(s.B) * (s.Nt + 1) - 1 : Mt;
    __nv_bfloat16* z = reinterpret_cast<__nv_bfloat16*>(ws + L.z);
    __nv_bfloat16* zlo = z + static_cast<size_t>(s.Lt) * Mt_rows * s.Ds;
    {
        Scope sc(2, st, (s.Lt + 15) / 16);
        const void* layers[kMaxLayers];
        for (int j = 0; j < s.Lt; ++j) layers[j] = r.teacher[j];
        CK(gemm_project(layers, s.Lt, Mt_rows, s.Dt, pt_hi, pt_lo, s.Ds, z, zlo, r.teacher_gap ? s.Nt + 1 : 0, s.Nt, st, r.teacher_lo[0]));
    }
    {
        // Grams AND column sums in one pass over the operands (the ones-operand MMA of umma_gemm.cuh): Ds % 4 == 0 is implied by Ds % 8
        float* gram_part = reinterpret_cast<float*>(ws + L.gram_part);
        const bool fused = gemm_gram_colsum_fused(s.Ds, true);
        {
            Scope sc(3, st, 6);
            CK(gemm_gram_batched(z, zlo, Mt_rows, s.Ds, s.Lt, stats, static_cast<long long>(stat_stride), gram_part, st, fused));
            if (r.student_lo[0]) {              // split-bf16 students (packed: one [P][Ms][Ds] block per half): three-term Grams
                CK(gemm_gram_batched(r.student[0], r.student_lo[0], Ms, s.Ds, s.P, stats + s.Lt * stat_stride, static_cast<long long>(stat_stride),
                                     gram_part, st, fused));
            } else {
                const void* pts[kMaxPoints];
                for (int i = 0; i < s.P; ++i) pts[i] = r.student[i];
                CK(gemm_gram_table(pts, s.P, Ms, s.Ds, stats + s.Lt * stat_stride, static_cast<long long>(stat_stride), gram_part,
                                   r.student_gap ? s.Ns : 0, r.student_bs, st, fused));
            }
        }
        if (!fused) {                           // D_s > 192 (two-tile Grams): separate column-sum kernels
            const bool one_launch = Mt_rows == Ms && !r.student_gap;
            Scope sc2(4, st, one_launch ? 2 : 4);
            ColsumJobs jt, js;
            memset(&jt, 0, sizeof jt); memset(&js, 0, sizeof js);
            for (int j = 0; j < s.Lt; ++j) {
                jt.hi[j] = z + static_cast<size_t>(j) * Mt_rows * s.Ds; jt.lo[j] = zlo + static_cast<size_t>(j) * Mt_rows * s.Ds;
                jt.out[j] = stats + j * stat_stride + static_cast<size_t>(s.Ds) * s.Ds;
            }
            for (int i = 0; i < s.P; ++i) {
                js.hi[i] = r.student[i]; js.lo[i] = r.student_lo[i];
                js.out[i] = stats + (s.Lt + i) * stat_stride + static_cast<size_t>(s.Ds) * s.Ds;
            }
            if (one_launch) {                   // same row count, same addressing: one launch covers teacher and student jobs
                for (int i = 0; i < s.P; ++i) { jt.hi[s.Lt + i] = js.hi[i]; jt.lo[s.Lt + i] = js.lo[i]; jt.out[s.Lt + i] = js.out[i]; }
                CK(launch_colsum(jt, s.Lt + s.P, Mt_rows, s.Ds, reinterpret_cast<float*>(ws + L.colsum_part), st));
            } else {
                CK(launch_colsum(jt, s.Lt, Mt_rows, s.Ds, reinterpret_cast<float*>(ws + L.colsum_part), st));
                CK(launch_colsum(js, s.P, Ms, s.Ds, reinterpret_cast<float*>(ws + L.colsum_part), st, r.student_gap ? s.Ns : 0, r.student_bs));
            }
        }
        (void)Mt_dense;
    }
    return 0;
}

extern "C" int basd_forward_solve(const basd_shape* shape, const basd_inputs* in_, void* workspace, float* geo_loss, void* stream) {
    if (!shape || !in_ || !workspace || !geo_loss) return fail("null argument");
    const basd_shape& s = *shape;
    const basd_inputs& in = *in_;
    if (check_shape(s)) return 1;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
    const Layout L = make_layout(s);
    Resolved r;
    if (resolve(s, in, ws, L, &r)) return 1;
    const float Mt = static_cast<float>(s.B) * s.Nt * s.world_size, Ms = static_cast<float>(s.B) * s.Ns * s.world_size;
    float* stats = reinterpret_cast<float*>(ws + L.stats);
    int* ranks = reinterpret_cast<int*>(ws + L.ranks);
    float* evals = reinterpret_cast<float*>(ws + L.evals);
    float* evk = reinterpret_cast<float*>(ws + L.evecs_km);
    float* evc = reinterpret_cast<float*>(ws + L.evecs_cm);
    float* d2 = reinterpret_cast<float*>(ws + L.d2);
    float* w = reinterpret_cast<float*>(ws + L.w);

    if (s.mode == BASD_MODE_PAIR) {
        // one teacher layer, one student point, no selector: mixing weight 1, rank and distance reported as 0
        CK(launch_fill_f32(w, 1.f, 1, st));
        CK(cudaMemsetAsync(ranks, 0, sizeof(int) * s.Lt, st));
        CK(cudaMemsetAsync(d2, 0, sizeof(float) * s.P * s.Lt, st));
    } else {
        TIMED(5, 1, CK(launch_pooled_eig(stats, s.Ds, s.Lt, s.P, Mt, Ms, ranks, evals, evk, evc, reinterpret_cast<int*>(ws + L.sweeps),
                                      reinterpret_cast<float*>(ws + L.eig_scr), st)));
        TIMED(6, 2, CK(launch_angles(s.Ds, s.Lt, s.P, ranks, evals, evk, evc, in.proj_s, reinterpret_cast<float*>(ws + L.ang_scr), d2,
                         reinterpret_cast<float*>(ws + L.gamma), reinterpret_cast<float*>(ws + L.cosv), in.log_temperatures, w, st)));
    }
    if (s.mode == BASD_MODE_SELECTOR) {
        CK(cudaMemsetAsync(geo_loss, 0, sizeof(float), st));
        CK(cudaMemsetAsync(ws + L.geo_i, 0, sizeof(float) * (s.P + 2), st));
        return 0;
    }
    float* a = reinterpret_cast<float*>(ws + L.a);
    float* ssum = reinterpret_cast<float*>(ws + L.ssum);
    TIMED(7, 1, CK(launch_importance_mix(reinterpret_cast<float*>(ws + L.rows), w, s.Lt, s.P, s.B, s.Nt, s.Ns, a, ssum, st)));
    PtrTable tt;
    memset(&tt, 0, sizeof tt);
    for (int j = 0; j < s.Lt; ++j) tt.p[j] = r.teacher[j];
    __nv_bfloat16* thi = reinterpret_cast<__nv_bfloat16*>(ws + L.tbar_hi);
    __nv_bfloat16* tlo = reinterpret_cast<__nv_bfloat16*>(ws + L.tbar_lo);
    // teacher-token form: the mixed teacher stays on its own token grid (the resampling is folded into F, polar.cu)
    const bool vt = L.path == kPathTeacherTokens;
    PtrTable tt_lo;
    memset(&tt_lo, 0, sizeof tt_lo);
    for (int j = 0; j < s.Lt; ++j) tt_lo.p[j] = r.teacher_lo[j];
    TIMED(8, 1, CK(launch_mix_teacher(tt, w, s.Lt, s.P, s.B, s.Nt, L.Nk, s.Dt, thi, tlo, st, r.teacher_bs, r.teacher_lo[0] ? &tt_lo : nullptr)));
    float* ktt = reinterpret_cast<float*>(ws + L.ktt);
    TIMED(9, 1, CK(gemm_token_gram(thi, tlo, s.P * s.B, L.Nk, s.Dt, ktt, st)));

    PolarArgs pa;
    memset(&pa, 0, sizeof pa);
    pa.Ns = s.Ns; pa.Ds = s.Ds; pa.B = s.B; pa.P = s.P; pa.NsPad = L.NsPad; pa.n_problems = s.P * s.B;
    for (int i = 0; i < s.P; ++i) { pa.student[i] = r.student[i]; pa.student_lo[i] = r.student_lo[i]; }
    pa.student_bs = r.student_bs;
    pa.Ktt = ktt; pa.a = a; pa.ssum = ssum;
    {
        const long long nprob = pa.n_problems;
        auto split = [&](size_t off, int rows, int inner) {      // tiled: [problem][col block][row][64], hi block then lo block
            SplitMat m;
            m.rows = rows; m.inner = inner; m.batch_stride = static_cast<long long>((inner + 63) / 64) * rows * 64;
            m.hi = reinterpret_cast<__nv_bfloat16*>(ws + off);
            m.lo = m.hi + nprob * m.batch_stride;
            return m;
        };
        pa.SW = split(L.psw, s.Ns, s.Ds);
        if (!vt) {
            pa.W = split(L.pw, s.Ds, s.Ns);
            pa.W2 = split(L.pw2, s.Ds, s.Ns);
            pa.T = split(L.pt, s.Ds, s.Ns);
            pa.A = split(L.pa, s.Ds, s.Ds);
            pa.Bm = split(L.pb, s.Ds, s.Ds);
            pa.Kt = split(L.pkt, s.Ns, s.Ns);
        } else {
            pa.vt = 1; pa.Nt = L.Nk; pa.NtPad = L.NsPad; pa.Dsp = L.Dsp;
            pa.A = split(L.pa, L.Nk, L.Nk);
            pa.Bm = split(L.pb, L.Nk, L.Nk);
            pa.FG = split(L.vfg, s.Ns, L.Nk);
            pa.FGt = split(L.vfgt, L.Nk, s.Ns);
            pa.GinvC = split(L.vginvc, L.Nk, L.Nk);
            pa.GinvT = split(L.vginvt, L.Nk, L.Nk);
            pa.X0 = split(L.vx0, L.Nk, L.Dsp);
            pa.X1 = split(L.vx1, L.Nk, L.Dsp);
            pa.X2 = split(L.vx2, L.Nk, L.Dsp);
            pa.Hm = split(L.vh, L.Nk, L.Nk);
            pa.M2 = split(L.vm2, L.Nk, L.Nk);
            pa.ginv = reinterpret_cast<float*>(ws + L.vginv);
            pa.thraw = reinterpret_cast<float*>(ws + L.vthraw);
            pa.ftf = reinterpret_cast<float*>(ws + L.vftf);
        }
    }
    pa.Gsw = reinterpret_cast<float*>(ws + L.gsw);
    pa.vec = reinterpret_cast<float*>(ws + L.pvec);
    pa.scal = reinterpret_cast<float*>(ws + L.pscal);
    pa.fro2 = reinterpret_cast<float*>(ws + L.pfro);
    pa.fro_slots = polar_fro_slots(vt ? L.Nk : s.Ds);
    pa.resid = reinterpret_cast<float*>(ws + L.pres);
    pa.steps = s.polar_steps ? s.polar_steps : kPolarStepsDefault;
    pa.gdir = reinterpret_cast<float*>(ws + L.gdir);
    pa.theta = reinterpret_cast<__nv_bfloat16*>(ws + L.theta);
    pa.theta_lo = reinterpret_cast<__nv_bfloat16*>(ws + L.theta_lo);
    pa.gwt = reinterpret_cast<float*>(ws + L.gwt);
    pa.loss_b = reinterpret_cast<float*>(ws + L.loss_b);
    pa.dbg = reinterpret_cast<float*>(ws + L.dbg);
    if (vt) CK(launch_polar_procrustes_vt(pa, st));
    else CK(launch_polar_procrustes(pa, st));  // timing slots 10 / 16 / 17 are bracketed inside
    float* geo_i = reinterpret_cast<float*>(ws + L.geo_i);
    TIMED(11, 1, CK(launch_loss_reduce(pa.loss_b, pa.dbg, s.P, s.B, geo_i, geo_i + s.P, geo_i + s.P + 1, st)));
    CK(cudaMemcpyAsync(geo_loss, geo_i + s.P, sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
}

extern "C" int basd_backward_dots(const basd_shape* shape, const basd_inputs* in_, void* workspace, void* stream) {
    if (!shape || !in_ || !workspace) return fail("null argument");
    const basd_shape& s = *shape;
    if (check_shape(s)) return 1;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
    const Layout L = make_layout(s);
    if (s.mode != BASD_MODE_LOSS) return 0;      // PAIR: no mixing weights to differentiate; SELECTOR: d total / d w comes from the caller
    Resolved r;
    if (resolve(s, *in_, ws, L, &r)) return 1;
    PtrTable tt, tt_lo;
    memset(&tt, 0, sizeof tt);
    memset(&tt_lo, 0, sizeof tt_lo);
    for (int j = 0; j < s.Lt; ++j) { tt.p[j] = r.teacher[j]; tt_lo.p[j] = r.teacher_lo[j]; }
    __nv_bfloat16* thi = reinterpret_cast<__nv_bfloat16*>(ws + L.tbar_hi);
    __nv_bfloat16* tlo = reinterpret_cast<__nv_bfloat16*>(ws + L.tbar_lo);
    __nv_bfloat16* dtm = reinterpret_cast<__nv_bfloat16*>(ws + L.dtm);
    __nv_bfloat16* dtm_lo = L.dtm_split ? dtm + static_cast<size_t>(s.P) * s.B * L.Nk * s.Dt : nullptr;
    // (teacher-token form: Theta, the mixed teacher and its gradient live on the teacher's own token grid, L.Nk = Nt rows)
    TIMED(12, 1, CK(gemm_theta_apply(reinterpret_cast<__nv_bfloat16*>(ws + L.theta), reinterpret_cast<__nv_bfloat16*>(ws + L.theta_lo), L.NsPad,
                                     thi, tlo, s.P * s.B, L.Nk, s.Dt, dtm, dtm_lo, st)));
    float* gw = reinterpret_cast<float*>(ws + L.gw);
    TIMED(13, 3, CK(launch_wgrad_dots(tt, dtm, dtm_lo, reinterpret_cast<float*>(ws + L.gwt), reinterpret_cast<float*>(ws + L.rows), s.Lt, s.P, s.B, s.Nt,
                         s.Ns, s.Dt, gw, reinterpret_cast<float*>(ws + L.gw_part), st, L.path == kPathTeacherTokens && L.Nk == s.Nt && s.Nt != s.Ns, r.teacher_bs,
                         r.teacher_lo[0] ? &tt_lo : nullptr)));
    return 0;
}

extern "C" int basd_backward_finish(const basd_shape* shape, const basd_inputs* in_, void* workspace, const float* grad_geo,
                                    void* const* grad_student, int grad_dtype, float* grad_log_temperatures, void* stream) {
    if (!shape || !in_ || !workspace || !grad_geo || !grad_student || !grad_log_temperatures) return fail("null argument");
    const basd_shape& s = *shape;
    const basd_inputs& in = *in_;
    if (check_shape(s)) return 1;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
    const Layout L = make_layout(s);
    Resolved r;
    if (resolve(s, in, ws, L, &r)) return 1;
    const float Ms = static_cast<float>(s.B) * s.Ns * s.world_size;
    // LOSS / PAIR: geo = mean over P points and B samples of the per-sample loss; SELECTOR: "gw" already is d total / d w
    const float scale = s.mode == BASD_MODE_SELECTOR ? 1.f : 1.f / (static_cast<float>(s.P) * s.B);
    __nv_bfloat16* ghi = reinterpret_cast<__nv_bfloat16*>(ws + L.gam_hi);
    __nv_bfloat16* glo = reinterpret_cast<__nv_bfloat16*>(ws + L.gam_lo);
    float* corr = reinterpret_cast<float*>(ws + L.corr);
    const size_t MsL = static_cast<size_t>(s.B) * s.Ns;
    if (s.mode == BASD_MODE_PAIR) {               // no selector path: Gamma' = 0, the gradient is the direct Procrustes term
        CK(cudaMemsetAsync(ghi, 0, 2 * static_cast<size_t>(s.P) * s.Ds * s.Ds, st));
        CK(cudaMemsetAsync(glo, 0, 2 * static_cast<size_t>(s.P) * s.Ds * s.Ds, st));
        CK(cudaMemsetAsync(corr, 0, 4 * static_cast<size_t>(s.P) * s.Ds, st));
        CK(cudaMemsetAsync(grad_log_temperatures, 0, 4 * static_cast<size_t>(s.P), st));
    } else {
        if (s.mode == BASD_MODE_SELECTOR)         // no Procrustes term: the direct-path gradient is zero
            CK(cudaMemsetAsync(ws + L.gdir, 0, 4 * static_cast<size_t>(s.P) * MsL * s.Ds, st));
        TIMED(14, 2, CK(launch_selector_bwd(s.Ds, s.Lt, s.P, reinterpret_cast<float*>(ws + L.gw), grad_geo, scale, reinterpret_cast<float*>(ws + L.w),
                               reinterpret_cast<float*>(ws + L.d2), in.log_temperatures, reinterpret_cast<float*>(ws + L.gamma),
                               reinterpret_cast<float*>(ws + L.stats), Ms, ghi, glo, corr, grad_log_temperatures, st)));
    }
    // (a CLS-stripped student view enters the product as the dense matrix of B (Ns + 1) - 1 rows it is in memory; the
    //  epilogue skips the rows between samples and writes the dense [B][Ns][Ds] gradient)
    const size_t Ms_rows = r.student_gap ? static_cast<size_t>(s.B) * (s.Ns + 1) - 1 : MsL;
    Scope sg(15, st, s.P);
    for (int i = 0; i < s.P; ++i) {
        if (!grad_student[i]) return fail("null grad_student[%d]", i);
        CK(gemm_student_grad(r.student[i], Ms_rows, s.Ds, ghi + static_cast<size_t>(i) * s.Ds * s.Ds, glo + static_cast<size_t>(i) * s.Ds * s.Ds,
                             reinterpret_cast<float*>(ws + L.gdir) + static_cast<size_t>(i) * MsL * s.Ds, corr + static_cast<size_t>(i) * s.Ds,
                             grad_geo, scale, grad_student[i], grad_dtype == BASD_DTYPE_BF16, r.student_gap ? s.Ns + 1 : 0, s.Ns, st, r.student_lo[i]));
    }
    return 0;
}

// ------------------------------------------------------------------------------------------- marchenko_pastur_rank
extern "C" int basd_mp_rank_workspace_bytes(int64_t M, int D, size_t* bytes) {
    if (!bytes || M < 1 || D < 8) return fail("invalid argument");
    *bytes = 2 * align_up(2 * static_cast<size_t>(M) * D) + align_up(4 * 2 * (static_cast<size_t>(D) * D + D)) + align_up(4 * 2 * D) +
             2 * align_up(4 * 2 * static_cast<size_t>(D) * D) + align_up(4 * pooled_eig_scratch_floats(D, 2)) +
             align_up(4 * gemm_gram_part_floats(static_cast<size_t>(M), D, 1)) + 4096;
    return 0;
}

extern "C" int basd_mp_rank(const void* features, int64_t M, int D, int dtype, int64_t row_stride, int* rank_out, void* workspace,
                            void* stream) {
    if (!features || !rank_out || !workspace) return fail("null argument");
    if (D % 8 || D > 4096) return fail("basd_mp_rank: D must be a multiple of 8 and <= 4096 (got %d)", D);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
    size_t off = 0;
    __nv_bfloat16* zb = reinterpret_cast<__nv_bfloat16*>(ws + off); off += align_up(2 * static_cast<size_t>(M) * D);
    __nv_bfloat16* zl = reinterpret_cast<__nv_bfloat16*>(ws + off); off += align_up(2 * static_cast<size_t>(M) * D);
    float* stats = reinterpret_cast<float*>(ws + off); off += align_up(4 * 2 * (static_cast<size_t>(D) * D + D));
    float* evals = reinterpret_cast<float*>(ws + off); off += align_up(4 * 2 * D);
    float* evk = reinterpret_cast<float*>(ws + off); off += align_up(4 * 2 * static_cast<size_t>(D) * D);
    float* evc = reinterpret_cast<float*>(ws + off); off += align_up(4 * 2 * static_cast<size_t>(D) * D);
    float* eig_scr = reinterpret_cast<float*>(ws + off); off += align_up(4 * pooled_eig_scratch_floats(D, 2));   // the launch runs the MP problem and the centred one
    float* gram_part = reinterpret_cast<float*>(ws + off); off += align_up(4 * gemm_gram_part_floats(static_cast<size_t>(M), D, 1));
    int* ranks = reinterpret_cast<int*>(ws + off);
    const bool exact = dtype == BASD_DTYPE_BF16;             // fp32 features keep fp32-class precision as a split pair
    CK(launch_pack_bf16(features, exact, 0, row_stride, 1, 1, static_cast<int>(M), D, zb, exact ? nullptr : zl, st));
    CK(cudaMemsetAsync(stats, 0, 4 * 2 * (static_cast<size_t>(D) * D + D), st));
    CK(gemm_gram(zb, exact ? nullptr : zl, static_cast<size_t>(M), D, stats, gram_part, st));
    CK(launch_pooled_eig(stats, D, 1, 0, static_cast<float>(M), 1.f, ranks, evals, evk, evc, nullptr, eig_scr, st, kEigMpOnly));
    CK(cudaMemcpyAsync(rank_out, ranks, sizeof(int), cudaMemcpyDeviceToDevice, st));
    return 0;
}

// ------------------------------------------------------------------------------------------- CLS attention rows
extern "C" int basd_cls_attention_rows(const void* q, const void* k, int dtype, int B, int H, int S, int dh, const int64_t* q_strides,
                                       const int64_t* k_strides, float scale, float* out, void* stream) {
    if (!q || !k || !out || !q_strides || !k_strides) return fail("null argument");
    if (B < 1 || H < 1 || S < 2 || dh < 1) return fail("invalid attention shape");
    if (q_strides[3] != 1 || k_strides[3] != 1) return fail("basd_cls_attention_rows: the head-dim stride of q and k must be 1");
    const long long qs[2] = {q_strides[0], q_strides[1]};
    const long long ks[3] = {k_strides[0], k_strides[1], k_strides[2]};
    CK(launch_cls_attention_rows(q, k, dtype == BASD_DTYPE_BF16, B, H, S, dh, qs, ks, scale, out, reinterpret_cast<cudaStream_t>(stream)));
    return 0;
}

// ------------------------------------------------------------------------------------------- query-mean attention rows
extern "C" int basd_query_mean_attention(const void* q, const void* k, int dtype, int B, int H, int S, int dh, const int64_t* q_strides,
                                         const int64_t* k_strides, float scale, float* out, void* stream) {
    if (!q || !k || !out || !q_strides || !k_strides) return fail("null argument");
    if (dtype != BASD_DTYPE_F32 && dtype != BASD_DTYPE_BF16) return fail("basd_query_mean_attention: unknown dtype %d", dtype);
    if (B < 1 || H < 1 || static_cast<long long>(B) * H > 0x7fffffffLL) return fail("basd_query_mean_attention: invalid B=%d, H=%d", B, H);
    if (S < 1 || S > kQueryMeanMaxTokens) return fail("basd_query_mean_attention: S=%d outside 1..%d", S, kQueryMeanMaxTokens);
    if (dh < 8 || dh > kQueryMeanMaxHeadDim || dh % 8)
        return fail("basd_query_mean_attention: dh=%d must be a multiple of 8 in 8..%d", dh, kQueryMeanMaxHeadDim);
    if (q_strides[3] != 1 || k_strides[3] != 1) return fail("basd_query_mean_attention: the head-dim stride of q and k must be 1");
    // The stride of a size-1 dimension is arbitrary (frameworks report anything there): replace it by the packed one.
    long long qs[3], ks[3];
    const int64_t* in[2] = {q_strides, k_strides};
    long long* o[2] = {qs, ks};
    for (int i = 0; i < 2; ++i) {
        o[i][2] = S == 1 ? dh : in[i][2];
        o[i][1] = H == 1 ? static_cast<long long>(S) * o[i][2] : in[i][1];
        o[i][0] = B == 1 ? static_cast<long long>(H) * o[i][1] : in[i][0];
    }
    // bf16 operands are read by TMA (16-byte aligned base and strides); fp32 rows as 16-byte vectors
    const long long align = dtype == BASD_DTYPE_BF16 ? 8 : 4;
    for (int i = 0; i < 2; ++i) {
        const void* p = i ? k : q;
        if ((reinterpret_cast<uintptr_t>(p) & 15) || o[i][0] < 1 || o[i][1] < 1 || o[i][2] < 1 || o[i][0] % align || o[i][1] % align || o[i][2] % align)
            return fail("basd_query_mean_attention: %s needs a 16-byte aligned base and positive (b,h,s) strides that are multiples of %lld elements "
                        "(got %p, %lld,%lld,%lld)", i ? "k" : "q", align, p, o[i][0], o[i][1], o[i][2]);
    }
    CK(launch_query_mean_attention(q, k, dtype == BASD_DTYPE_BF16, B, H, S, dh, qs, ks, scale, out, reinterpret_cast<cudaStream_t>(stream)));
    return 0;
}

// ------------------------------------------------------------------------------------------- _align_token_count
extern "C" int basd_align_tokens(const void* tokens, int dtype, const int64_t* strides, int B, int Nin, int Nout, int D, void* out, void* stream) {
    if (!tokens || !strides || !out) return fail("null argument");
    if (B < 1 || Nin < 1 || Nout < 1 || D < 1) return fail("invalid token shape");
    CK(launch_align_tokens(tokens, dtype == BASD_DTYPE_BF16, strides[0], strides[1], strides[2], B, Nin, Nout, D, out,
                           reinterpret_cast<cudaStream_t>(stream)));
    return 0;
}
extern "C" int basd_align_tokens_bwd(const void* grad_out, int dtype, int B, int Nin, int Nout, int D, void* grad_in, void* stream) {
    if (!grad_out || !grad_in) return fail("null argument");
    if (B < 1 || Nin < 1 || Nout < 1 || D < 1) return fail("invalid token shape");
    CK(launch_align_tokens_bwd(grad_out, dtype == BASD_DTYPE_BF16, B, Nin, Nout, D, grad_in, reinterpret_cast<cudaStream_t>(stream)));
    return 0;
}

// ------------------------------------------------------------------------------------------- UW-SO weighting (combined.py:78-85)
__global__ void uwso_combine_kernel(const float* __restrict__ ce, const float* __restrict__ geo, const float* __restrict__ det_ce,
                                    const float* __restrict__ det_geo, float eps, float* __restrict__ out3) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    // the reference's own operation order: inv_i = 1 / clamp(d_i, min = eps); w = inv / sum(inv); total = w_0 L_0 + w_1 L_1
    // (clamp keeps a NaN term NaN like torch.clamp does - SURVEY.md C.1: an MP rank of 0 makes the reference's loss NaN; no FMA
    //  contraction: the total is bit-identical to the reference's separate multiplies and add)
    const float d0 = *det_ce, d1 = *det_geo;
    const float i0 = 1.0f / (d0 < eps ? eps : d0), i1 = 1.0f / (d1 < eps ? eps : d1);
    const float sum = __fadd_rn(i0, i1);
    const float w0 = i0 / sum, w1 = i1 / sum;
    out3[0] = __fadd_rn(__fmul_rn(w0, *ce), __fmul_rn(w1, *geo));
    out3[1] = w0;
    out3[2] = w1;
}
extern "C" int basd_uwso_combine(const float* ce, const float* geo, const float* det_ce, const float* det_geo, float eps, float* out3,
                                 void* stream) {
    if (!ce || !geo || !det_ce || !det_geo || !out3) return fail("null argument");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    TIMED(11, 1, (uwso_combine_kernel<<<1, 32, 0, st>>>(ce, geo, det_ce, det_geo, eps, out3)));
    CK(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------- host attention rows
// Of a teacher attention map [B,H,S,S] in HOST memory the loss reads the CLS query row only (relational.py:24).  One pitched
// DMA per layer (width = one row, pitch = one map) moves exactly those rows to a dense device [B,H,1,S] tensor - no host-side
// gather, no staging buffer; asynchronous when the host tensor is pinned.
extern "C" int basd_copy_cls_rows_h2d(const void* host_attn, int elem_bytes, int B, int H, int S, const int64_t* strides, void* dev_rows,
                                      void* stream) {
    if (!host_attn || !dev_rows || !strides) return fail("null argument");
    if (B < 1 || H < 1 || S < 1 || (elem_bytes != 2 && elem_bytes != 4)) return fail("invalid attention shape");
    if (strides[3] != 1) return fail("basd_copy_cls_rows_h2d: the key stride must be 1");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const size_t width = static_cast<size_t>(S) * elem_bytes;
    const char* src = reinterpret_cast<const char*>(host_attn);
    char* dst = reinterpret_cast<char*>(dev_rows);
    if (strides[0] == static_cast<int64_t>(H) * strides[1]) {          // (b, h) rows equally spaced: one copy
        CK(cudaMemcpy2DAsync(dst, width, src, static_cast<size_t>(strides[1]) * elem_bytes, width, static_cast<size_t>(B) * H,
                             cudaMemcpyHostToDevice, st));
    } else {
        for (int b = 0; b < B; ++b)
            CK(cudaMemcpy2DAsync(dst + static_cast<size_t>(b) * H * width, width, src + static_cast<size_t>(b) * strides[0] * elem_bytes,
                                 static_cast<size_t>(strides[1]) * elem_bytes, width, H, cudaMemcpyHostToDevice, st));
    }
    return 0;
}

// ------------------------------------------------------------------------------------------- test hooks
extern "C" int basd_selftest_gemm(int variant, const void* A, const void* B, float* C, int M, int N, int K, void* stream) {
    CK(gemm_selftest(variant, reinterpret_cast<const __nv_bfloat16*>(A), reinterpret_cast<const __nv_bfloat16*>(B), C, M, N, K,
                     reinterpret_cast<cudaStream_t>(stream)));
    return 0;
}

// eigen-decomposition of a symmetric PSD matrix G [n][n]: evals [n] descending, evecs [n][n] (row e = e-th eigenvector).
// workspace: 4 * (n*n + n) + 4 * n * n bytes (+ alignment slack 4096), plus 4 * n * (n + 3) bytes when n > 224.
extern "C" int basd_selftest_eig(const float* G, int n, float* evals, float* evecs, int* sweeps, void* workspace, void* stream) {
    if (!G || !evals || !evecs || !workspace) return fail("null argument");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
    float* stats = reinterpret_cast<float*>(ws);
    float* evc = reinterpret_cast<float*>(ws + align_up(4 * (static_cast<size_t>(n) * n + n)));
    float* eig_scr = reinterpret_cast<float*>(ws + align_up(4 * (static_cast<size_t>(n) * n + n)) + align_up(4 * static_cast<size_t>(n) * n));
    CK(cudaMemsetAsync(stats, 0, 4 * (static_cast<size_t>(n) * n + n), st));
    CK(cudaMemcpyAsync(stats, G, 4 * static_cast<size_t>(n) * n, cudaMemcpyDeviceToDevice, st));
    CK(launch_pooled_eig(stats, n, 0, 1, 1.f, 1.f, nullptr, evals, evecs, evc, sweeps, eig_scr, st));
    return 0;
}
