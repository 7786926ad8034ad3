// genrec_b200 - C ABI (include/genrec_b200.h): argument checking, buffer carving and kernel orchestration.
// Nothing here allocates or synchronises; every kernel goes onto the caller's stream.
#include "../../include/genrec_b200.h"

#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <utility>

#include "attn_hstu.cuh"
#include "attn_sasrec.cuh"
#include "attn_t5.cuh"
#include "attn_tc.cuh"
#include "beam.cuh"
#include "common.cuh"
#include "dp_adam.cuh"
#include "exact_f32.cuh"
#include "rowwise.cuh"
#include "rq_argmin.cuh"
#include "tc_gemm.cuh"
#include "tc_ce.cuh"
#include "tc_tn_group.cuh"
#include <cstdlib>

using namespace grb;

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define GRB_CUDA(expr)                                                                                  \
    do {                                                                                                \
        cudaError_t _e = (expr);                                                                        \
        if (_e != cudaSuccess) return fail(GRB_ECUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
    } while (0)
#define GRB_REQUIRE(cond, ...)                            \
    do {                                                  \
        if (!(cond)) return fail(GRB_EINVAL, __VA_ARGS__); \
    } while (0)
#define GRB_TRY(expr)          \
    do {                       \
        int _r = (expr);       \
        if (_r != 0) return _r; \
    } while (0)

inline size_t align_up(size_t v, size_t a = 256) { return (v + a - 1) / a * a; }
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

int current_device() {
    int dev = 0;
    cudaGetDevice(&dev);
    return dev;
}
int sm_count() {     // per device ordinal: a process may drive several GPUs
    static int n[64] = {0};
    const int dev = current_device() & 63;
    if (n[dev] == 0) {
        int v = 0;
        cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
        n[dev] = v > 0 ? v : 148;
    }
    return n[dev];
}
// GRB_CE = store : G' stored, dE by the TN GEMM (round-1 schedule; always at D = 256)
//          exact : no [T, C] tensor, two class sweeps (the exponent shift is the exact row maximum)
//          (default) : no [T, C] tensor, ONE class sweep (shift = max(probe-tile maximum, target logit), see tc_ce.cuh)
int ce_mode_env() {
    static const int v = [] {
        const char* e = getenv("GRB_CE");
        if (e && !strcmp(e, "store")) return (int)CE_STORE_G;
        if (e && (!strcmp(e, "exact") || !strcmp(e, "keep"))) return (int)CE_KEEP_G;
        return (int)CE_ONE_SWEEP;
    }();
    return v;
}
bool ce_store_forced() { return ce_mode_env() == CE_STORE_G; }
int row_grid(int T) {
    int need = (T + ROW_THREADS / 32 - 1) / (ROW_THREADS / 32);
    int cap = sm_count() * 8;
    return need < cap ? (need < 1 ? 1 : need) : cap;
}


// ---- GEMM wrappers over the tcgen05/TMA kernel.  Operand majors: *_MN = 0 -> K contiguous, 1 -> M/N contiguous (see tc_gemm.cuh).
int tn_splits(int M, int N, int K) {
    int tiles = ((M + TC_BM - 1) / TC_BM) * ((N + TC_BN - 1) / TC_BN);
    int want = (sm_count() + tiles - 1) / tiles;
    int kb = (K + TC_BK - 1) / TC_BK;
    int maxs = kb / 2 > 0 ? kb / 2 : 1;
    return want < 1 ? 1 : (want > maxs ? maxs : want);
}
// z = x W^T + b ; act: 0 none, 1 silu, 2 relu   (NT)
cudaError_t gemm_bias_act(int act, const bf16* x, const bf16* w, const float* bias, bf16* z, bf16* a, int M, int N, int K, const Dropout& drop,
                          cudaStream_t st) {
    if (act == 0) return launch_tc_gemm<0, 0>(x, w, M, N, K, K, K, 1, TcEpiBiasAct<0>{bias, N, drop}, z, nullptr, N, sm_count(), st);
    if (act == 1) return launch_tc_gemm<0, 0>(x, w, M, N, K, K, K, 1, TcEpiBiasAct<1>{bias, N, drop}, z, a, N, sm_count(), st);
    return launch_tc_gemm<0, 0>(x, w, M, N, K, K, K, 1, TcEpiBiasAct<2>{bias, N, drop}, z, a, N, sm_count(), st);
}
// y = res + drop(x W^T + b) (* row_scale)   (NT)
cudaError_t gemm_bias_res(const bf16* x, const bf16* w, const float* bias, const float* res, const float* row_scale, float* y, int M, int N,
                          int K, const Dropout& drop, cudaStream_t st) {
    return launch_tc_gemm<0, 0>(x, w, M, N, K, K, K, 1, TcEpiBiasResidual{bias, res, row_scale, N, drop}, y, nullptr, N, sm_count(), st);
}
// g[M,N] = dropmask(dy[M,K] W[K,N]) * act'(z)   (NN) ; act 1 silu, 2 relu
cudaError_t gemm_dact(int act, const bf16* dy, const bf16* w, const bf16* z, bf16* g, int M, int N, int K, const Dropout& drop, cudaStream_t st) {
    if (act == 1) return launch_tc_gemm<0, 1>(dy, w, M, N, K, K, N, 1, TcEpiDAct<1>{z, N, drop}, g, nullptr, N, sm_count(), st);
    return launch_tc_gemm<0, 1>(dy, w, M, N, K, K, N, 1, TcEpiDAct<2>{z, N, drop}, g, nullptr, N, sm_count(), st);
}
// out[M,N] fp32 = scale * A[M,K] B[K,N] (+ res)   (NN)
cudaError_t gemm_nn_f32(const bf16* A, const bf16* B, float* out, const float* res, float scale, int M, int N, int K, int lda, int ldb,
                        cudaStream_t st) {
    return launch_tc_gemm<0, 1>(A, B, M, N, K, lda, ldb, 1, TcEpiF32{res, N, scale}, out, nullptr, N, sm_count(), st);
}
// out[M,N] fp32 += A^T B with A stored [K,M], B stored [K,N]   (TN, split-K, atomics)
cudaError_t gemm_tn_atomic(const bf16* A, const bf16* B, float* out, int M, int N, int K, int lda, int ldb, cudaStream_t st) {
    return launch_tc_gemm<1, 1>(A, B, M, N, K, lda, ldb, tn_splits(M, N, K), TcEpiAtomicF32{out, N, 1.f}, nullptr, nullptr, 0, sm_count(), st);
}
// out[M,N] fp32 (leading dim N, any parity) = A B^T   (NT)
cudaError_t gemm_nt_f32_plain(const bf16* A, const bf16* B, float* out, int M, int N, int K, cudaStream_t st) {
    return launch_tc_gemm<0, 0>(A, B, M, N, K, K, K, 1, TcEpiF32Plain{out, N}, nullptr, nullptr, 0, sm_count(), st);
}

// ---- carved layouts ------------------------------------------------------------------------------------------
struct LayerSaved {
    bf16 *xb, *zp, *P, *O, *xn, *z1, *hact;
    float *st1, *x1, *st2;
    size_t bytes;
};
LayerSaved carve_saved(void* base, size_t T, size_t D) {
    LayerSaved s;
    size_t off = 0;
    char* b = static_cast<char*>(base);
    auto take = [&](size_t n) { char* p = b ? b + off : nullptr; off += align_up(n); return p; };
    s.xb = (bf16*)take(T * D * 2);
    s.zp = (bf16*)take(T * 4 * D * 2);
    s.P = (bf16*)take(T * 4 * D * 2);
    s.O = (bf16*)take(T * D * 2);
    s.st1 = (float*)take(T * 2 * 4);
    s.x1 = (float*)take(T * D * 4);
    s.xn = (bf16*)take(T * D * 2);
    s.st2 = (float*)take(T * 2 * 4);
    s.z1 = (bf16*)take(T * 4 * D * 2);
    s.hact = (bf16*)take(T * 4 * D * 2);
    s.bytes = off;
    return s;
}
struct LayerWork {
    bf16 *dyb, *dz1, *dO, *dzp;
    float *dxn, *dx1, *dq_acc;
    size_t bytes;
};
LayerWork carve_work(void* base, size_t T, size_t D) {
    LayerWork w;
    size_t off = 0;
    char* b = static_cast<char*>(base);
    auto take = [&](size_t n) { char* p = b ? b + off : nullptr; off += align_up(n); return p; };
    w.dyb = (bf16*)take(T * D * 2);
    w.dz1 = (bf16*)take(T * 4 * D * 2);
    w.dxn = (float*)take(T * D * 4);
    w.dx1 = (float*)take(T * D * 4);
    w.dO = (bf16*)take(T * D * 2);
    w.dzp = (bf16*)take(T * 4 * D * 2);
    w.dq_acc = (float*)take(T * D * 4);
    w.bytes = off;
    return w;
}

int check_dims(const grb_hstu_dims* d) {
    GRB_REQUIRE(d != nullptr, "dims is null");
    GRB_REQUIRE(d->B > 0 && d->L > 0 && d->H > 0, "B, L, H must be positive (B=%d L=%d H=%d)", d->B, d->L, d->H);
    GRB_REQUIRE(d->D == 64 || d->D == 128 || d->D == 256, "embed_dim %d unsupported (64, 128, 256)", d->D);
    GRB_REQUIRE(d->D % d->H == 0, "embed_dim %% num_heads != 0");
    int dh = d->D / d->H;
    GRB_REQUIRE(dh == 32 || dh == 64, "head_dim %d unsupported (32, 64)", dh);
    GRB_REQUIRE(d->npos >= 1 && d->npos <= ATT_MAX_BUCKETS, "num_position_buckets %d out of range [1,64]", d->npos);
    GRB_REQUIRE(d->ntime >= 0 && d->ntime <= ATT_MAX_BUCKETS, "num_time_buckets %d out of range [0,64]", d->ntime);
    GRB_REQUIRE(d->L <= 16384, "seq_len %d too long", d->L);
    GRB_REQUIRE(d->dropout_p >= 0.f && d->dropout_p < 1.f, "dropout_p out of range");
    return 0;
}

// opt in to > 48 KB dynamic shared memory once per (kernel, high-water mark): no runtime call on the steady-state path,
// in particular none while a CUDA graph is being captured after warm-up.
template <class Kern>
int set_smem(Kern k, size_t bytes) {
    static std::mutex mu;
    static std::map<std::pair<int, const void*>, size_t> high_water;  // keyed by (device, kernel address): the attribute is per device
    std::lock_guard<std::mutex> lock(mu);
    size_t& hw = high_water[std::make_pair(current_device(), reinterpret_cast<const void*>(k))];
    if (hw < 48 * 1024) hw = 48 * 1024;
    if (bytes > hw) {
        GRB_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        hw = bytes;
    }
    return 0;
}

HstuAttnArgs make_attn_args(const grb_hstu_dims* d, const grb_hstu_layer_params* p, const grb_hstu_seq* s, const LayerSaved& sv) {
    HstuAttnArgs a;
    memset(&a, 0, sizeof(a));
    const int D = d->D;
    a.q = sv.P + 2 * D; a.k = sv.P + 3 * D; a.v = sv.P + D;
    a.ldq = a.ldk = a.ldv = 4 * D;
    a.B = d->B; a.L = d->L; a.H = d->H;
    // uniform position buckets (the reference's behaviour) collapse to ONE effective bucket: the index matrix was built with
    // npos = 1, the tables shrink to 65 entries and the pointers are offset to the single live row of the [npos, H] table
    a.bias.wpos = p->pos_table + (s->pos_uniform ? (size_t)s->pos_bucket0 * d->H : 0);
    const bool has_time = p->time_table != nullptr && s->has_time && d->ntime > 0;
    a.bias.wtime = has_time ? p->time_table : nullptr;
    a.bias.bias_index = s->bias_index;
    a.bias.ldix = s->ld_index;
    a.bias.pos_uniform = s->pos_uniform;
    a.bias.pos_bucket0 = 0;
    a.bias.npos = s->pos_uniform ? 1 : d->npos;
    a.bias.ntime = has_time ? d->ntime : 0;
    a.o = sv.O; a.ldo = D;
    return a;
}

template <int DH>
int launch_hstu_attn_fwd(const HstuAttnArgs& a, cudaStream_t st) {
    size_t smem = sizeof(AttSmem<DH, 1>) + align_up((size_t)(a.bias.npos * 64 + 1) * 4, 16);
    GRB_TRY(set_smem(hstu_attn_fwd_kernel<DH>, smem));
    dim3 grid((a.L + ATT_BLK - 1) / ATT_BLK, a.H, a.B);
    launch_k(hstu_attn_fwd_kernel<DH>, grid, ATT_THREADS, smem, st, a);
    GRB_CUDA(cudaGetLastError());
    return 0;
}
// Fork/join helper: dQ and dK/dV are independent, both latency-bound at low occupancy -> run them concurrently (the side
// stream and the events are created on first use, i.e. during warm-up, never while a CUDA graph is being captured).
struct SideStream {
    cudaStream_t s = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
    bool ok = false;
    bool init() {
        if (ok) return true;
        if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess) return false;
        if (cudaEventCreateWithFlags(&fork, cudaEventDisableTiming) != cudaSuccess) return false;
        if (cudaEventCreateWithFlags(&join, cudaEventDisableTiming) != cudaSuccess) return false;
        ok = true;
        return true;
    }
};
SideStream& side_stream() {
    static thread_local SideStream ss;   // the backward runs on the autograd thread: one side stream per calling thread
    return ss;
}
// ---- deferred weight gradients.  dW / dE GEMMs are not on the critical path of a training step: nothing reads them before the
// optimizer.  With grb_set_defer_weight_grads(1) they go to a per-device side stream, forked where their operands are ready and
// joined by grb_join_deferred() (FlatAdam.step calls it), so they fill the SM tails of the epilogue-bound GEMMs and run next to the
// issue-bound attention kernels; the 620 MB dlogits stream of the head's dE GEMM overlaps the last block's backward.  The CALLER keeps
// the operand buffers (layer workspace, saved blob, head workspace) alive until the join.  Works under CUDA-graph capture (event
// fork / join pulls the side stream into the capture).
struct DeferStream {
    cudaStream_t s = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
    bool ok = false, pending = false;
};
std::mutex g_defer_mu;
bool g_defer_on = false;
DeferStream& defer_stream() {
    static DeferStream ds[64];
    return ds[current_device() & 63];
}
// run `launch(side_stream)` after everything enqueued on `st` so far; returns 0 / error code
template <class F>
int defer_run(cudaStream_t st, F&& launch) {
    std::lock_guard<std::mutex> lock(g_defer_mu);
    DeferStream& d = defer_stream();
    if (!d.ok) {
        GRB_CUDA(cudaStreamCreateWithFlags(&d.s, cudaStreamNonBlocking));
        GRB_CUDA(cudaEventCreateWithFlags(&d.fork, cudaEventDisableTiming));
        GRB_CUDA(cudaEventCreateWithFlags(&d.join, cudaEventDisableTiming));
        d.ok = true;
    }
    GRB_CUDA(cudaEventRecord(d.fork, st));
    GRB_CUDA(cudaStreamWaitEvent(d.s, d.fork, 0));
    GRB_TRY(launch(d.s));
    GRB_CUDA(cudaEventRecord(d.join, d.s));
    d.pending = true;
    return 0;
}
int join_pending(cudaStream_t st) {
    std::lock_guard<std::mutex> lock(g_defer_mu);
    DeferStream& d = defer_stream();
    if (d.ok && d.pending) {
        GRB_CUDA(cudaStreamWaitEvent(st, d.join, 0));
        d.pending = false;
    }
    return 0;
}
bool use_side_stream() {
    static int v = -1;
    if (v < 0) {
        // dQ and dK/dV side by side: +1.6 % step throughput at cfg-2 (1.786 -> 1.758 ms) once the weight-gradient GEMMs had moved
        // off the critical path; GRB_SIDE_STREAM=0 serialises them again
        const char* e = getenv("GRB_SIDE_STREAM");
        v = (e && strcmp(e, "0") == 0) ? 0 : 1;
    }
    return v == 1;
}

template <int DH>
int launch_hstu_attn_bwd(const HstuAttnArgs& a, cudaStream_t st) {
    dim3 grid((a.L + ATT_BLK - 1) / ATT_BLK, a.H, a.B);
    size_t posb = align_up((size_t)(a.bias.npos * 64 + 1) * 4, 16);  // combined bias table
    size_t smem_q = sizeof(AttSmem<DH>) + posb;
    GRB_TRY(set_smem(hstu_attn_bwd_dq_kernel<DH>, smem_q));
    SideStream& ss = side_stream();
    const bool forked = use_side_stream() && ss.init();
    if (forked) {
        GRB_CUDA(cudaEventRecord(ss.fork, st));
        GRB_CUDA(cudaStreamWaitEvent(ss.s, ss.fork, 0));
        launch_k(hstu_attn_bwd_dq_kernel<DH>, grid, ATT_THREADS, smem_q, ss.s, a);
        GRB_CUDA(cudaGetLastError());
        GRB_CUDA(cudaEventRecord(ss.join, ss.s));
    } else {
        launch_k(hstu_attn_bwd_dq_kernel<DH>, grid, ATT_THREADS, smem_q, st, a);
        GRB_CUDA(cudaGetLastError());
    }
    size_t smem_k = sizeof(AttSmemKV<DH>) + posb + (size_t)4 * (a.bias.ntime + 1 + (a.bias.pos_uniform ? 0 : a.bias.npos + 1)) * 32 * sizeof(float);
    const bool has_time = a.bias.wtime != nullptr && a.bias.ntime > 0, pos_uni = a.bias.pos_uniform != 0;
    auto go = [&](auto kern) -> int {
        GRB_TRY(set_smem(kern, smem_k));
        launch_k(kern, grid, ATT_THREADS, smem_k, st, a, (int)posb);
        return 0;
    };
    if (has_time && pos_uni) GRB_TRY(go(hstu_attn_bwd_dkdv_kernel<DH, true, true>));
    else if (has_time) GRB_TRY(go(hstu_attn_bwd_dkdv_kernel<DH, true, false>));
    else if (pos_uni) GRB_TRY(go(hstu_attn_bwd_dkdv_kernel<DH, false, true>));
    else GRB_TRY(go(hstu_attn_bwd_dkdv_kernel<DH, false, false>));
    GRB_CUDA(cudaGetLastError());
    if (forked) GRB_CUDA(cudaStreamWaitEvent(st, ss.join, 0));
    return 0;
}

// ---- tcgen05 attention path (attn_tc.cuh): the default whenever the position buckets are uniform (the reference's behaviour)
//      and head_dim is 32 or 64.  GRB_ATTN=mma selects the first-generation mma.sync kernels (they need the bias_index matrix).
// GRB_ATTN = tc | mma | auto (default).  auto: the tcgen05 kernels for seq_len > 256, the mma.sync kernels below - measured on
// B200 (scripts/bench_attn.py): with 128-row tiles and one thread per TMEM lane a 200-token sequence leaves 40 % of the lanes idle and a
// CTA lives for only a handful of tiles, so the 64-row mma.sync kernels (5 CTAs per SM) are still ahead there; from ~512 tokens on
// the tcgen05 path wins and needs no [B, L, L] index.  Read on every call so that a test can flip it.
int attn_mode() {
    const char* e = getenv("GRB_ATTN");
    if (e && strcmp(e, "mma") == 0) return 0;
    if (e && strcmp(e, "tc") == 0) return 1;
    return 2;
}
bool attn_tc_possible(const grb_hstu_dims* d, const grb_hstu_seq* s);
bool use_attn_tc(const grb_hstu_dims* d, const grb_hstu_seq* s) {
    const int mode = attn_mode();
    if (mode == 0 || (mode == 2 && d->L <= 256 && s->bias_index != nullptr)) return false;
    return attn_tc_possible(d, s);
}
bool attn_tc_possible(const grb_hstu_dims* d, const grb_hstu_seq* s) {
    const int dh = d->D / d->H;
    return s->pos_uniform && (dh == 32 || dh == 64) && d->D % 64 == 0 && s->pad != nullptr && s->time_thr != nullptr &&
           (s->timestamps == nullptr || !s->has_time || (s->rel32 != nullptr && s->wide != nullptr));
}
HstuTcArgs make_tc_args(const grb_hstu_dims* d, const float* pos_table, const float* time_table, const grb_hstu_seq* s) {
    HstuTcArgs a;
    memset(&a, 0, sizeof(a));
    const bool has_time = time_table != nullptr && s->has_time && s->timestamps != nullptr && d->ntime > 0;
    a.ts = has_time ? reinterpret_cast<const long long*>(s->timestamps) : nullptr;
    a.rel32 = has_time ? s->rel32 : nullptr;
    a.wide = s->wide;
    a.pad = s->pad;
    a.thr64 = reinterpret_cast<const long long*>(s->time_thr);
    a.wpos = pos_table + (size_t)s->pos_bucket0 * d->H;
    a.wtime = has_time ? time_table : nullptr;
    a.ntime = has_time ? d->ntime : 0;
    a.B = d->B; a.L = d->L; a.H = d->H; a.D = d->D;
    return a;
}
int launch_attn_tc_fwd(const grb_hstu_dims* d, const float* pos_table, const float* time_table, const grb_hstu_seq* s, const bf16* P, bf16* O,
                       cudaStream_t st) {
    const int D = d->D, dh = D / d->H;
    const size_t T = (size_t)d->B * d->L;
    HstuTcArgs a = make_tc_args(d, pos_table, time_table, s);
    a.o = O; a.ldo = D;
    CUtensorMap tmP;
    if (!make_tmap_bf16(&tmP, P, T, 4 * (size_t)D, 4 * (size_t)D, 64, 128)) return fail(GRB_EINVAL, "tensor map creation failed (attention P)");
    const int nqt = (d->L + 127) / 128;
    const unsigned grid = (unsigned)((D / 64) * d->B * nqt);
    if (dh == 32) {
        const size_t smem = AtcFwdSmem<32>::kBytes + 1024;
        GRB_TRY(set_smem(hstu_attn_tc_fwd_kernel<32>, smem));
        launch_k(hstu_attn_tc_fwd_kernel<32>, grid, ATC_THREADS, smem, st, tmP, a, nqt);
    } else {
        const size_t smem = AtcFwdSmem<64>::kBytes + 1024;
        GRB_TRY(set_smem(hstu_attn_tc_fwd_kernel<64>, smem));
        launch_k(hstu_attn_tc_fwd_kernel<64>, grid, ATC_THREADS, smem, st, tmP, a, nqt);
    }
    GRB_CUDA(cudaGetLastError());
    return 0;
}
// dzp columns V, Q, K <- gradients w.r.t. the pre-activations ; dq_acc: [T, D] fp32 scratch
int launch_attn_tc_bwd(const grb_hstu_dims* d, const float* pos_table, const float* time_table, const grb_hstu_seq* s, const bf16* P,
                       const bf16* zp, const bf16* dO, bf16* dzp, float* dwpos, float* dwtime, float* dq_acc, cudaStream_t st) {
    const int D = d->D, dh = D / d->H;
    const size_t T = (size_t)d->B * d->L;
    HstuTcArgs a = make_tc_args(d, pos_table, time_table, s);
    a.zk = zp ? zp + 3 * D : nullptr; a.zv = zp ? zp + D : nullptr; a.ldz = 4 * D;
    a.dk = dzp + 3 * D; a.dv = dzp + D; a.lddz = 4 * D;
    a.dq_acc = dq_acc;
    a.dwpos = dwpos + (size_t)s->pos_bucket0 * d->H;
    a.dwtime = a.wtime ? dwtime : nullptr;
    GRB_REQUIRE(a.wtime == nullptr || dwtime != nullptr, "time_table gradient pointer is null");
    CUtensorMap tmP, tmDO;
    if (!make_tmap_bf16(&tmP, P, T, 4 * (size_t)D, 4 * (size_t)D, 64, 128) || !make_tmap_bf16(&tmDO, dO, T, D, D, 64, 128))
        return fail(GRB_EINVAL, "tensor map creation failed (attention backward)");
    GRB_CUDA(cudaMemsetAsync(dq_acc, 0, T * D * sizeof(float), st));
    const int nqt = (d->L + 127) / 128;
    const unsigned grid = (unsigned)((D / 64) * d->B * nqt);
    if (dh == 32) {
        const size_t smem = AtcBwdSmem<32>::kBytes + 1024;
        GRB_TRY(set_smem(hstu_attn_tc_bwd_kernel<32>, smem));
        launch_k(hstu_attn_tc_bwd_kernel<32>, grid, ATC_THREADS, smem, st, tmP, tmDO, a, nqt);
    } else {
        const size_t smem = AtcBwdSmem<64>::kBytes + 1024;
        GRB_TRY(set_smem(hstu_attn_tc_bwd_kernel<64>, smem));
        launch_k(hstu_attn_tc_bwd_kernel<64>, grid, ATC_THREADS, smem, st, tmP, tmDO, a, nqt);
    }
    GRB_CUDA(cudaGetLastError());
    size_t blocks = (T * (D / 8) + 255) / 256;
    if (blocks > (size_t)sm_count() * 8) blocks = (size_t)sm_count() * 8;
    launch_k(hstu_dq_finish_kernel, (unsigned)blocks, 256, 0, st, (const float*)dq_acc, zp ? zp + 2 * D : (const bf16*)nullptr, 4 * D, dzp + 2 * D,
             4 * D, T, D);
    GRB_CUDA(cudaGetLastError());
    return 0;
}

template <int NP, class Args, class Kern>
int launch_row(Kern k, const Args& a, int T, cudaStream_t st) {
    launch_k(k, row_grid(T), ROW_THREADS, 0, st, a);
    GRB_CUDA(cudaGetLastError());
    return 0;
}
template <int NP, class Args, class Kern>
int launch_row_bwd(Kern k, const Args& a, int T, cudaStream_t st) {
    int need = (T + ROW_THREADS / 32 - 1) / (ROW_THREADS / 32);
    int cap = sm_count() * 3;
    launch_k(k, need < cap ? (need < 1 ? 1 : need) : cap, ROW_THREADS, 0, st, a);
    GRB_CUDA(cudaGetLastError());
    return 0;
}
#define GRB_ROW_BWD_DISPATCH(D, KERN, ARGS, T, ST)                                        \
    do {                                                                                  \
        if ((D) == 64) GRB_TRY((launch_row_bwd<1>(KERN<1>, ARGS, T, ST)));                \
        else if ((D) == 128) GRB_TRY((launch_row_bwd<2>(KERN<2>, ARGS, T, ST)));          \
        else if ((D) == 256) GRB_TRY((launch_row_bwd<4>(KERN<4>, ARGS, T, ST)));          \
        else return fail(GRB_EINVAL, "row kernels support D in {64,128,256}, got %d", (D)); \
    } while (0)
#define GRB_ROW_DISPATCH(D, KERN, ARGS, T, ST)                                            \
    do {                                                                                  \
        if ((D) == 64) GRB_TRY((launch_row<1>(KERN<1>, ARGS, T, ST)));                    \
        else if ((D) == 128) GRB_TRY((launch_row<2>(KERN<2>, ARGS, T, ST)));              \
        else if ((D) == 256) GRB_TRY((launch_row<4>(KERN<4>, ARGS, T, ST)));              \
        else return fail(GRB_EINVAL, "row kernels support D in {64,128,256}, got %d", (D)); \
    } while (0)

int cast_bf16(const float* in, bf16* out, size_t n, int D, const Dropout& drop, const float* row_scale, cudaStream_t st) {
    GRB_REQUIRE(D > 0 && D % 4 == 0 && n % (size_t)D == 0, "cast needs rows of a multiple-of-4 length D");
    int threads = 256;
    size_t blocks = (n / 4 + threads - 1) / threads;
    if (blocks > (size_t)sm_count() * 16) blocks = (size_t)sm_count() * 16;
    if (blocks < 1) blocks = 1;
    launch_k(cast_f32_bf16_kernel, (unsigned)blocks, threads, 0, st, in, out, n, D, drop, row_scale);
    GRB_CUDA(cudaGetLastError());
    return 0;
}
int cast_colsum(const float* in, bf16* out, int T, int D, const Dropout& drop, float* colsum_out, cudaStream_t st) {
    GRB_REQUIRE(D > 0 && D % 4 == 0, "cast needs rows of a multiple-of-4 length D");
    int cx = (D + 127) / 128;
    int cy = (8 * sm_count() + cx - 1) / cx;
    int maxy = (T + 31) / 32;
    if (cy > maxy) cy = maxy;
    if (cy < 1) cy = 1;
    launch_k(cast_colsum_f32_bf16_kernel, dim3(cx, cy), 256, 0, st, in, out, T, D, drop, colsum_out);
    GRB_CUDA(cudaGetLastError());
    return 0;
}
int colsum(const bf16* in, int T, int N, int ld, float* out, cudaStream_t st) {
    if (N % 8 != 0 || ld % 8 != 0) return fail(GRB_EINVAL, "colsum needs N and ld to be multiples of 8");
    int cx = (N + 255) / 256;
    int cy = (4 * sm_count() + cx - 1) / cx;
    int maxy = (T + 63) / 64;
    if (cy > maxy) cy = maxy;
    if (cy < 1) cy = 1;
    launch_k(colsum_bf16_kernel, dim3(cx, cy), 256, 0, st, in, T, N, ld, out);
    GRB_CUDA(cudaGetLastError());
    return 0;
}

constexpr uint32_t SITE_GATE = 0, SITE_FFN_HID = 1, SITE_FFN_OUT = 2, SITE_EMBED = 250, SITE_ATTN = 3;
inline uint32_t site_of(int layer, uint32_t which) { return (uint32_t)layer * 8u + which; }

}  // namespace

extern "C" {

const char* grb_last_error(void) { return g_err; }
int grb_version(void) { return 100; }
uint64_t grb_launch_count(void) { return (uint64_t)launch_counter(); }

int grb_check_device(int ordinal) {
    cudaDeviceProp prop;
    cudaError_t e = cudaGetDeviceProperties(&prop, ordinal);
    if (e != cudaSuccess) return fail(GRB_ENODEV, "cudaGetDeviceProperties(%d): %s", ordinal, cudaGetErrorString(e));
    if (prop.major != 10) return fail(GRB_ENODEV, "device %d is sm_%d%d; this library is built for sm_100a only", ordinal, prop.major, prop.minor);
    return 0;
}

size_t grb_hstu_layer_saved_bytes(const grb_hstu_dims* d) {
    if (check_dims(d)) return 0;
    return carve_saved(nullptr, (size_t)d->B * d->L, d->D).bytes;
}
size_t grb_hstu_layer_workspace_bytes(const grb_hstu_dims* d) {
    if (check_dims(d)) return 0;
    return carve_work(nullptr, (size_t)d->B * d->L, d->D).bytes;
}

int grb_hstu_layer_forward(const grb_hstu_dims* d, const grb_hstu_layer_params* p, const grb_hstu_seq* s, const float* x,
                           float* y, void* saved, void* stream) {
    GRB_TRY(check_dims(d));
    GRB_REQUIRE(p && s && x && y && saved, "null argument");
    GRB_REQUIRE(p->proj_w && p->proj_b && p->pos_table && p->ln1_g && p->ln1_b && p->ffn1_w && p->ffn1_b && p->ffn2_w &&
                    p->ffn2_b && p->ln2_g && p->ln2_b, "null parameter pointer");
    const bool attn_tc = use_attn_tc(d, s);
    GRB_REQUIRE(attn_tc || s->bias_index, "null sequence metadata: the mma.sync attention path needs bias_index");
    GRB_REQUIRE(attn_tc || (s->ld_index >= d->L && s->ld_index % 8 == 0 && aligned16(s->bias_index)),
                "bias_index pitch must be a multiple of 8 and >= L");
    GRB_REQUIRE(aligned16(x) && aligned16(y) && aligned16(saved) && aligned16(p->proj_w) && aligned16(p->ffn1_w) && aligned16(p->ffn2_w),
                "buffers must be 16-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int T = d->B * d->L, D = d->D;
    LayerSaved sv = carve_saved(saved, T, D);
    const Dropout nodrop = make_dropout(0.f, 0, 0);

    // 1. bf16 copy of the block input (GEMM operand; also the dWp operand in backward)
    GRB_TRY(cast_bf16(x, sv.xb, (size_t)T * D, D, nodrop, nullptr, st));
    // 2. P = silu(x Wp^T + bp) -> [U | V | Q | K]                                            (hstu.py:234-235)
    {
        GRB_CUDA(gemm_bias_act(1, sv.xb, (const bf16*)p->proj_w, p->proj_b, sv.zp, sv.P, T, 4 * D, D, nodrop, st));
    }
    // 3. O = silu(Q K^T + bias) V, causal + key padding                                      (hstu.py:244-267)
    GRB_TRY(join_pending(st));   // a bias-index matrix built on the side stream (deferred schedule) must be complete
    if (attn_tc) {
        GRB_TRY(launch_attn_tc_fwd(d, p->pos_table, p->time_table, s, sv.P, sv.O, st));
    } else {
        HstuAttnArgs a = make_attn_args(d, p, s, sv);
        if (D / d->H == 32) GRB_TRY(launch_hstu_attn_fwd<32>(a, st));
        else GRB_TRY(launch_hstu_attn_fwd<64>(a, st));
    }
    // 4. x1 = x + drop(LN1(O) * U) ; xn = LN2(x1)                                            (hstu.py:271-278)
    {
        LnGateFwdArgs a{sv.O, D, sv.P, 4 * D, x, p->ln1_g, p->ln1_b, p->ln2_g, p->ln2_b, sv.x1, sv.xn, sv.st1, sv.st2, T, D, 1e-5f,
                        make_dropout(d->dropout_p, d->seed, site_of(d->layer_index, SITE_GATE), d->seed_dev)};
        GRB_ROW_DISPATCH(D, ln_gate_fwd_kernel, a, T, st);
    }
    // 5. h = drop(silu(xn W1^T + b1))                                                        (hstu.py:210-212)
    {
        GRB_CUDA(gemm_bias_act(1, sv.xn, (const bf16*)p->ffn1_w, p->ffn1_b, sv.z1, sv.hact, T, 4 * D, D,
                               make_dropout(d->dropout_p, d->seed, site_of(d->layer_index, SITE_FFN_HID), d->seed_dev), st));
    }
    // 6. y = x1 + drop(h W2^T + b2)                                                          (hstu.py:213-214, :278)
    {
        GRB_CUDA(gemm_bias_res(sv.hact, (const bf16*)p->ffn2_w, p->ffn2_b, sv.x1, nullptr, y, T, D, 4 * D,
                               make_dropout(d->dropout_p, d->seed, site_of(d->layer_index, SITE_FFN_OUT), d->seed_dev), st));
    }
    return 0;
}

int grb_hstu_layer_backward(const grb_hstu_dims* d, const grb_hstu_layer_params* p, const grb_hstu_seq* s, const float* dy,
                            const void* saved, float* dx, const grb_hstu_layer_grads* g, void* workspace, void* stream) {
    GRB_TRY(check_dims(d));
    GRB_REQUIRE(p && s && dy && saved && dx && g && workspace, "null argument");
    GRB_REQUIRE(g->proj_w && g->proj_b && g->pos_table && g->ln1_g && g->ln1_b && g->ffn1_w && g->ffn1_b && g->ffn2_w && g->ffn2_b &&
                    g->ln2_g && g->ln2_b, "null gradient pointer");
    GRB_REQUIRE(aligned16(dy) && aligned16(dx) && aligned16(saved) && aligned16(workspace), "buffers must be 16-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int T = d->B * d->L, D = d->D;
    LayerSaved sv = carve_saved(const_cast<void*>(saved), T, D);
    LayerWork w = carve_work(workspace, T, D);
    const Dropout nodrop = make_dropout(0.f, 0, 0);
    const Dropout drop_out = make_dropout(d->dropout_p, d->seed, site_of(d->layer_index, SITE_FFN_OUT), d->seed_dev);
    const Dropout drop_hid = make_dropout(d->dropout_p, d->seed, site_of(d->layer_index, SITE_FFN_HID), d->seed_dev);
    const Dropout drop_gate = make_dropout(d->dropout_p, d->seed, site_of(d->layer_index, SITE_GATE), d->seed_dev);

    // FFN second linear
    GRB_TRY(cast_colsum(dy, w.dyb, T, D, drop_out, g->ffn2_b, st));   // dyb = bf16(dropmask(dy)) ; db2 += column sums
    {
        GRB_CUDA(gemm_dact(1, w.dyb, (const bf16*)p->ffn2_w, sv.z1, w.dz1, T, 4 * D, D, drop_hid, st));  // dz1 = dropmask(dyb W2) * silu'(z1)
    }
    // FFN first linear
    // bias gradients are off the critical path too: with deferred weight gradients the column sums run beside the main chain
    auto colsum_maybe_deferred = [&](const bf16* in, float* out) -> int {
        if (g_defer_on) return defer_run(st, [&](cudaStream_t side) -> int { return colsum(in, T, 4 * D, 4 * D, out, side); });
        return colsum(in, T, 4 * D, 4 * D, out, st);
    };
    GRB_TRY(colsum_maybe_deferred(w.dz1, g->ffn1_b));
    {
        GRB_CUDA(gemm_nn_f32(w.dz1, (const bf16*)p->ffn1_w, w.dxn, nullptr, 1.f, T, D, 4 * D, 4 * D, D, st));  // dxn = dz1 W1
    }
    // LN2 + residual + gate + LN1
    {
        LnGateBwdArgs a{dy, w.dxn, sv.x1, sv.st1, sv.st2, sv.O, D, sv.P, 4 * D, sv.zp, 4 * D, p->ln1_g, p->ln1_b, p->ln2_g,
                        w.dx1, w.dO, D, w.dzp, 4 * D, g->ln1_g, g->ln1_b, g->ln2_g, g->ln2_b, T, D, drop_gate};
        GRB_ROW_DISPATCH(D, ln_gate_bwd_kernel, a, T, st);
    }
    // attention backward -> gradients w.r.t. the V, Q, K pre-activations
    if (use_attn_tc(d, s)) {
        GRB_TRY(launch_attn_tc_bwd(d, p->pos_table, p->time_table, s, sv.P, sv.zp, w.dO, w.dzp, g->pos_table, g->time_table, w.dq_acc, st));
    } else {
        GRB_REQUIRE(s->bias_index, "null sequence metadata: the mma.sync attention path needs bias_index");
        HstuAttnArgs a = make_attn_args(d, p, s, sv);
        a.d_o = w.dO; a.lddo = D;
        a.zq = sv.zp + 2 * D; a.zk = sv.zp + 3 * D; a.zv = sv.zp + D; a.ldz = 4 * D;
        a.dq = w.dzp + 2 * D; a.dk = w.dzp + 3 * D; a.dv = w.dzp + D; a.lddq = 4 * D;
        a.dwpos = g->pos_table + (s->pos_uniform ? (size_t)s->pos_bucket0 * d->H : 0);
        a.dwtime = g->time_table;
        GRB_REQUIRE(a.bias.wtime == nullptr || g->time_table != nullptr, "time_table gradient pointer is null");
        if (D / d->H == 32) GRB_TRY(launch_hstu_attn_bwd<32>(a, st));
        else GRB_TRY(launch_hstu_attn_bwd<64>(a, st));
    }
    // projection
    GRB_TRY(colsum_maybe_deferred(w.dzp, g->proj_b));
    {
        GRB_CUDA(gemm_nn_f32(w.dzp, (const bf16*)p->proj_w, dx, w.dx1, 1.f, T, D, 4 * D, 4 * D, D, st));  // dx = dx1 + dzp Wp
    }
    {
        // the three weight gradients of the layer in ONE grouped launch: dW2 += dyb^T h, dW1 += dz1^T xn, dWp += dzp^T xb
        TnSpec specs[3] = {{w.dyb, sv.hact, g->ffn2_w, D, 4 * D, T, D, 4 * D, 4 * D},
                           {w.dz1, sv.xn, g->ffn1_w, 4 * D, D, T, 4 * D, D, D},
                           {w.dzp, sv.xb, g->proj_w, 4 * D, D, T, 4 * D, D, D}};
        if (g_defer_on) {
            GRB_TRY(defer_run(st, [&](cudaStream_t side) -> int {
                GRB_CUDA(launch_tc_tn_group(specs, 3, sm_count(), side));
                return 0;
            }));
        } else {
            GRB_CUDA(launch_tc_tn_group(specs, 3, sm_count(), st));
        }
    }
    (void)nodrop;
    return 0;
}

int grb_hstu_bias_index(const int64_t* timestamps, const uint8_t* pad, const int64_t* time_thr, const uint8_t* pos_bucket, int B, int L,
                        int npos, int ntime, uint16_t* out, int ld_index, void* stream) {
    GRB_REQUIRE(pad && time_thr && pos_bucket && out, "null argument");
    GRB_REQUIRE(B > 0 && L > 0 && B <= 65535 && L <= 65535, "bad shape B=%d L=%d", B, L);
    GRB_REQUIRE(ld_index >= L && ld_index % 8 == 0, "ld_index must be a multiple of 8 and >= L");
    GRB_REQUIRE(ntime >= 0 && ntime <= ATT_MAX_BUCKETS && npos >= 1 && npos <= ATT_MAX_BUCKETS, "bucket counts out of range");
    dim3 grid((ld_index + 255) / 256, (L + 7) / 8, B);
    auto go = [&](cudaStream_t s_) -> int {
        launch_k(hstu_bias_index_kernel, grid, 256, 0, s_, reinterpret_cast<const long long*>(timestamps), pad,
                 reinterpret_cast<const long long*>(time_thr), pos_bucket, L, ld_index, npos, ntime, out);
        GRB_CUDA(cudaGetLastError());
        return 0;
    };
    // the index matrix is first needed by the attention kernel of the first block: with the deferred schedule it is built beside
    // that block's cast + projection GEMM (grb_hstu_layer_forward joins before its attention launch)
    if (g_defer_on) return defer_run(static_cast<cudaStream_t>(stream), go);
    return go(static_cast<cudaStream_t>(stream));
}

int grb_set_defer_weight_grads(int on) {
    std::lock_guard<std::mutex> lock(g_defer_mu);
    g_defer_on = on != 0;
    return 0;
}
int grb_join_deferred(void* stream) { return join_pending(static_cast<cudaStream_t>(stream)); }

int grb_hstu_seq_prepare(const int64_t* timestamps, const uint8_t* pad, int B, int L, int32_t* rel32, uint8_t* wide, void* stream) {
    GRB_REQUIRE(timestamps && pad && rel32 && wide, "null argument");
    GRB_REQUIRE(B > 0 && L > 0, "bad shape B=%d L=%d", B, L);
    launch_k(hstu_seq_prep_kernel, (unsigned)B, 256, 0, static_cast<cudaStream_t>(stream), reinterpret_cast<const long long*>(timestamps), pad, L,
             reinterpret_cast<int*>(rel32), wide);
    GRB_CUDA(cudaGetLastError());
    return 0;
}

int grb_hstu_bucket_bytes_debug(const grb_hstu_seq* s, int B, int L, int ntime, uint8_t* out, void* stream) {
    GRB_REQUIRE(s && out && s->pad && s->time_thr, "null argument");
    GRB_REQUIRE(B > 0 && L > 0 && B <= 65535 && ntime >= 0 && ntime <= 64, "bad shape");
    HstuTcArgs a;
    memset(&a, 0, sizeof(a));
    const bool has_time = s->timestamps != nullptr && s->has_time && ntime > 0;
    GRB_REQUIRE(!has_time || (s->rel32 && s->wide), "rel32 / wide missing: call grb_hstu_seq_prepare first");
    a.ts = has_time ? reinterpret_cast<const long long*>(s->timestamps) : nullptr;
    a.rel32 = s->rel32; a.wide = s->wide; a.pad = s->pad;
    a.thr64 = reinterpret_cast<const long long*>(s->time_thr);
    a.ntime = has_time ? ntime : 0;
    a.B = B; a.L = L;
    dim3 grid((L + 31) / 32, (L + 127) / 128, B);
    launch_k(hstu_bucket_bytes_debug_kernel, grid, 128, 0, static_cast<cudaStream_t>(stream), a, out);
    GRB_CUDA(cudaGetLastError());
    return 0;
}

size_t grb_hstu_attention_scratch_bytes(const grb_hstu_dims* d) {
    if (check_dims(d)) return 0;
    return align_up((size_t)d->B * d->L * d->D * sizeof(float));
}
int grb_hstu_attention_forward(const grb_hstu_dims* d, const float* pos_table, const float* time_table, const grb_hstu_seq* s,
                               const void* P_bf16, void* O_bf16, void* stream) {
    GRB_TRY(check_dims(d));
    GRB_REQUIRE(pos_table && s && P_bf16 && O_bf16, "null argument");
    GRB_REQUIRE(attn_tc_possible(d, s), "the stand-alone attention entry points run the tcgen05 path: uniform position buckets, head_dim 32/64, "
                                        "pad / time_thr (and rel32 / wide with timestamps) required");
    GRB_REQUIRE(aligned16(P_bf16) && aligned16(O_bf16), "buffers must be 16-byte aligned");
    return launch_attn_tc_fwd(d, pos_table, time_table, s, (const bf16*)P_bf16, (bf16*)O_bf16, static_cast<cudaStream_t>(stream));
}
int grb_hstu_attention_backward(const grb_hstu_dims* d, const float* pos_table, const float* time_table, const grb_hstu_seq* s,
                                const void* P_bf16, const void* zp_bf16, const void* dO_bf16, void* dzp_bf16, float* dpos_table,
                                float* dtime_table, void* scratch, void* stream) {
    GRB_TRY(check_dims(d));
    GRB_REQUIRE(pos_table && s && P_bf16 && dO_bf16 && dzp_bf16 && dpos_table && scratch, "null argument");
    GRB_REQUIRE(attn_tc_possible(d, s), "the stand-alone attention entry points run the tcgen05 path");
    GRB_REQUIRE(aligned16(P_bf16) && aligned16(dO_bf16) && aligned16(dzp_bf16) && aligned16(scratch) && (zp_bf16 == nullptr || aligned16(zp_bf16)),
                "buffers must be 16-byte aligned");
    return launch_attn_tc_bwd(d, pos_table, time_table, s, (const bf16*)P_bf16, (const bf16*)zp_bf16, (const bf16*)dO_bf16, (bf16*)dzp_bf16,
                              dpos_table, dtime_table, (float*)scratch, static_cast<cudaStream_t>(stream));
}

int grb_collate_jagged(const int64_t* items, const int64_t* stamps, const int64_t* offsets, const int64_t* targets, int B, int L,
                       int64_t* out_input_ids, int64_t* out_targets, int64_t* out_timestamps, void* stream) {
    GRB_REQUIRE(items && offsets && targets && out_input_ids && out_targets, "null argument");
    GRB_REQUIRE(B > 0 && L > 0, "bad shape B=%d L=%d", B, L);
    const size_t n = (size_t)B * L;
    launch_k(collate_jagged_kernel, (unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream), reinterpret_cast<const long long*>(items),
             reinterpret_cast<const long long*>(stamps), reinterpret_cast<const long long*>(offsets), reinterpret_cast<const long long*>(targets), B, L,
             reinterpret_cast<long long*>(out_input_ids), reinterpret_cast<long long*>(out_targets), reinterpret_cast<long long*>(out_timestamps));
    GRB_CUDA(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------------ embedding
int grb_embed_forward(const int64_t* ids, const float* table, const float* pos_table, float* x, uint8_t* pad, int B, int L, int D,
                      float scale, int mask_pad_rows, float dropout_p, uint64_t seed, const uint64_t* seed_dev, void* stream) {
    GRB_REQUIRE(ids && table && x, "null argument");
    GRB_REQUIRE(B > 0 && L > 0 && D > 0 && D % 4 == 0, "bad shape");
    EmbedArgs a{reinterpret_cast<const long long*>(ids), table, pos_table, x, pad, B * L, L, D, scale, mask_pad_rows,
                make_dropout(dropout_p, seed, SITE_EMBED, seed_dev)};
    launch_k(embed_fwd_kernel, row_grid(B * L), ROW_THREADS, 0, static_cast<cudaStream_t>(stream), a);
    GRB_CUDA(cudaGetLastError());
    return 0;
}
int grb_embed_backward(const int64_t* ids, const float* dx, float* dtable, float* dpos_table, int B, int L, int D, float scale,
                       int mask_pad_rows, float dropout_p, uint64_t seed, const uint64_t* seed_dev, void* stream) {
    GRB_REQUIRE(ids && dx && dtable, "null argument");
    GRB_REQUIRE(D % 4 == 0 && aligned16(dx) && aligned16(dtable) && (dpos_table == nullptr || aligned16(dpos_table)),
                "embedding backward needs D %% 4 == 0 and 16-byte aligned buffers");
    EmbedBwdArgs a{reinterpret_cast<const long long*>(ids), dx, dtable, dpos_table, B * L, L, D, scale, mask_pad_rows,
                   make_dropout(dropout_p, seed, SITE_EMBED, seed_dev)};
    launch_k(embed_bwd_kernel, row_grid(B * L), ROW_THREADS, 0, static_cast<cudaStream_t>(stream), a);
    GRB_CUDA(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------------ head
namespace {
struct HeadWork {
    bf16* xf; float* stf; bf16* logits; float* dxf; float* scal;  // scal[0] = inv_count
    bf16* xs; float* row_sums; float2* row_stats;                  // fused CE: x / sum_row, per-row sums of G', {max, target logit}
    float* col_shift;                                              // fused CE: exponent shift of every token for the class-stationary dE pass
    void* ce_scratch;
    int ldl;
    size_t bytes;
};
HeadWork carve_head(void* base, size_t T, size_t D, size_t C) {
    HeadWork h;
    size_t off = 0;
    char* b = static_cast<char*>(base);
    auto take = [&](size_t n) { char* p = b ? b + off : nullptr; off += align_up(n); return p; };
    h.ldl = (int)((C + 7) / 8 * 8);
    h.xf = (bf16*)take(T * D * 2);
    h.stf = (float*)take(T * 2 * 4);
    h.dxf = (float*)take(T * D * 4);
    h.scal = (float*)take(64);
    h.xs = (bf16*)take(T * D * 2);
    h.row_sums = (float*)take(4 * T * 4);   // [2][T] sums of G' per class half, then [2][T] target-logit partials (one-sweep CE)
    h.row_stats = (float2*)take(T * 8);
    h.col_shift = (float*)take(((T + 127) / 128) * 128 * 4);
    h.ce_scratch = take(ce_scratch_bytes((int)T));
    h.logits = (bf16*)take(T * (size_t)h.ldl * 2);
    h.bytes = off;
    return h;
}
}  // namespace

size_t grb_head_workspace_bytes(int T, int D, int C) { return carve_head(nullptr, T, D, C).bytes; }

int grb_head_loss_forward_backward(const float* x, const float* ln_g, const float* ln_b, float ln_eps, const void* table_bf16,
                                   const int64_t* targets, int T, int D, int C, float* loss, float* dx, float* dtable, float* dln_g,
                                   float* dln_b, void* workspace, void* stream) {
    GRB_REQUIRE(x && ln_g && ln_b && table_bf16 && targets && loss && workspace, "null argument");
    GRB_REQUIRE(T > 0 && C > 1 && (D == 64 || D == 128 || D == 256), "bad shape T=%d D=%d C=%d", T, D, C);
    const bool want_grad = dx != nullptr;
    GRB_REQUIRE(!want_grad || (dtable && dln_g && dln_b), "null gradient pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    HeadWork h = carve_head(workspace, T, D, C);
    // the target count (one CTA, latency-bound) depends on the targets only: with the deferred schedule it runs beside the final
    // LayerNorm and is joined before the fused CE kernel
    const bool count_aside = g_defer_on;
    // D <= 128: no [T, C] tensor reaches HBM - dX' accumulates in TMEM beside the CE sweep and dE comes from a class-stationary pass
    // that recomputes G.  D = 256 (or GRB_CE=store): G' is stored and dE is a TN GEMM.
    const bool keep_g = D <= 128 && want_grad && !ce_store_forced();
    const int ce_mode = keep_g ? ce_mode_env() : (int)CE_STORE_G;
    auto count = [&](cudaStream_t s_) -> int {
        launch_k(ce_count_kernel, 1, 1024, 0, s_, reinterpret_cast<const long long*>(targets), T, h.scal, loss);
        GRB_CUDA(cudaGetLastError());
        return 0;
    };
    if (count_aside) GRB_TRY(defer_run(st, count));
    {
        LnFwdArgs a{x, ln_g, ln_b, h.xf, nullptr, h.stf, T, D, ln_eps};
        GRB_ROW_DISPATCH(D, ln_fwd_kernel, a, T, st);
    }
    if (count_aside) GRB_TRY(join_pending(st));
    else GRB_TRY(count(st));
    bool fused_dx = false;
    {
        // fused: logits are never materialised; (D <= 128) h.dxf = G' E, and h.logits receives G' only when a dE GEMM needs it
        const long long* tg = reinterpret_cast<const long long*>(targets);                                  // (hstu.py:137-146)
        const bf16* tb = (const bf16*)table_bf16;
        if (D == 64) GRB_CUDA(launch_tc_ce<1>(h.xf, tb, h.logits, ce_mode, T, C, h.ldl, tg, h.scal, h.row_sums, h.row_stats, h.dxf, &fused_dx, h.ce_scratch, sm_count(), st));
        else if (D == 128) GRB_CUDA(launch_tc_ce<2>(h.xf, tb, h.logits, ce_mode, T, C, h.ldl, tg, h.scal, h.row_sums, h.row_stats, h.dxf, &fused_dx, h.ce_scratch, sm_count(), st));
        else GRB_CUDA(launch_tc_ce<4>(h.xf, tb, h.logits, CE_STORE_G, T, C, h.ldl, tg, h.scal, h.row_sums, h.row_stats, h.dxf, &fused_dx, h.ce_scratch, sm_count(), st));
    }
    {
        // normalisation pass of the fused CE (rowwise.cuh ce_finish_kernel): loss, and - with gradients - dxf, x / sum_row, the one-hot
        // term of dE.  Without the dX fusion (D = 256) dxf' = G' E comes from a GEMM first.
        if (want_grad && !fused_dx) GRB_CUDA(gemm_nn_f32(h.logits, (const bf16*)table_bf16, h.dxf, nullptr, 1.f, T, D, C, h.ldl, D, st));
        CeFinishArgs fa{h.row_sums, h.row_stats, ce_mode == CE_ONE_SWEEP ? h.row_sums + (size_t)2 * T : nullptr,
                        reinterpret_cast<const long long*>(targets), h.scal, h.xf, (const bf16*)table_bf16,
                        want_grad ? h.dxf : nullptr, (want_grad && !keep_g) ? h.xs : nullptr, keep_g ? h.col_shift : nullptr,
                        want_grad ? dtable : nullptr, loss, T, D};
        launch_k(ce_finish_kernel, row_grid(T), ROW_THREADS, 0, st, fa);
        GRB_CUDA(cudaGetLastError());
    }
    if (!want_grad) return 0;
    {
        if (keep_g) {
            // dE[C,D] += G^T xf with G recomputed class block by class block (tc_ce.cuh CE_ACCUM_T); off the critical path like the
            // other weight gradients
            auto accum = [&](cudaStream_t s_) -> int {
                if (D == 64) GRB_CUDA(launch_tc_ce_accum_t<1>(h.xf, (const bf16*)table_bf16, h.col_shift, dtable, T, C, sm_count(), s_));
                else GRB_CUDA(launch_tc_ce_accum_t<2>(h.xf, (const bf16*)table_bf16, h.col_shift, dtable, T, C, sm_count(), s_));
                return 0;
            };
            if (g_defer_on) GRB_TRY(defer_run(st, accum));
            else GRB_TRY(accum(st));
        } else {
            TnSpec spec{h.logits, h.xs, dtable, C, D, T, h.ldl, D, D};  // dE[C,D] += G'^T (xf / sum_row) = dlogits^T xf
            if (g_defer_on) {
                GRB_TRY(defer_run(st, [&](cudaStream_t side) -> int {
                    GRB_CUDA(launch_tc_tn_group(&spec, 1, sm_count(), side));
                    return 0;
                }));
            } else {
                GRB_CUDA(launch_tc_tn_group(&spec, 1, sm_count(), st));
            }
        }
    }
    {
        LnBwdArgs a{h.dxf, x, h.stf, ln_g, nullptr, dx, dln_g, dln_b, T, D};
        GRB_ROW_BWD_DISPATCH(D, ln_bwd_kernel, a, T, st);
    }
    return 0;
}

int grb_head_logits(const float* x, const float* ln_g, const float* ln_b, float ln_eps, const void* table_bf16, int T, int D, int C,
                    float* logits, void* workspace, void* stream) {
    GRB_REQUIRE(x && ln_g && ln_b && table_bf16 && logits && workspace, "null argument");
    GRB_REQUIRE(T > 0 && C > 1 && (D == 64 || D == 128 || D == 256), "bad shape T=%d D=%d C=%d", T, D, C);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    HeadWork h = carve_head(workspace, T, D, C);
    {
        LnFwdArgs a{x, ln_g, ln_b, h.xf, nullptr, h.stf, T, D, ln_eps};
        GRB_ROW_DISPATCH(D, ln_fwd_kernel, a, T, st);
    }
    GRB_CUDA(gemm_nt_f32_plain(h.xf, (const bf16*)table_bf16, logits, T, C, D, st));
    return 0;
}

int grb_eval_rank_metrics(const float* logits, const int64_t* targets, int B, int C, float* metrics, int32_t* ranks, void* stream) {
    GRB_REQUIRE(logits && targets && metrics, "null argument");
    GRB_REQUIRE(B > 0 && C > 1, "bad shape B=%d C=%d", B, C);
    launch_k(eval_rank_kernel, (unsigned)B, 256, 0, static_cast<cudaStream_t>(stream), logits, C, reinterpret_cast<const long long*>(targets), metrics,
             reinterpret_cast<int*>(ranks));
    GRB_CUDA(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------------ SASRec attention
namespace {
int sas_args(const grb_sasrec_dims* d, SasAttnArgs& a) {
    GRB_REQUIRE(d && d->B > 0 && d->L > 0 && d->H > 0 && d->D % d->H == 0, "bad dims");
    int dh = d->D / d->H;
    GRB_REQUIRE(dh == 32 || dh == 64, "head_dim %d unsupported (32, 64)", dh);
    GRB_REQUIRE(d->D % 8 == 0, "embed_dim must be a multiple of 8");
    memset(&a, 0, sizeof(a));
    a.ld = d->D; a.B = d->B; a.L = d->L; a.H = d->H;
    a.scale = 1.f / sqrtf((float)dh);
    a.drop = make_dropout(d->dropout_p, d->seed, site_of(d->layer_index, SITE_ATTN), d->seed_dev);
    return 0;
}
}  // namespace

int grb_sasrec_attention_forward(const grb_sasrec_dims* d, const void* q, const void* k, const void* v, const uint8_t* pad, void* out,
                                 float* lse, void* stream) {
    SasAttnArgs a;
    GRB_TRY(sas_args(d, a));
    GRB_REQUIRE(q && k && v && pad && out && lse, "null argument");
    a.q = (const bf16*)q; a.k = (const bf16*)k; a.v = (const bf16*)v; a.pad = pad; a.out = (bf16*)out; a.lse = lse;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    dim3 grid((a.L + ATT_BLK - 1) / ATT_BLK, a.H, a.B);
    if (d->D / d->H == 32) {
        GRB_TRY(set_smem(sas_attn_fwd_kernel<32>, sizeof(SasSmem<32>)));
        launch_k(sas_attn_fwd_kernel<32>, grid, ATT_THREADS, sizeof(SasSmem<32>), st, a);
    } else {
        GRB_TRY(set_smem(sas_attn_fwd_kernel<64>, sizeof(SasSmem<64>)));
        launch_k(sas_attn_fwd_kernel<64>, grid, ATT_THREADS, sizeof(SasSmem<64>), st, a);
    }
    GRB_CUDA(cudaGetLastError());
    return 0;
}

int grb_sasrec_attention_backward(const grb_sasrec_dims* d, const void* q, const void* k, const void* v, const uint8_t* pad,
                                  const void* out, const float* lse, const void* dout, void* dq, void* dk, void* dv, void* stream) {
    SasAttnArgs a;
    GRB_TRY(sas_args(d, a));
    GRB_REQUIRE(q && k && v && pad && out && lse && dout && dq && dk && dv, "null argument");
    a.q = (const bf16*)q; a.k = (const bf16*)k; a.v = (const bf16*)v; a.pad = pad;
    a.out = (bf16*)const_cast<void*>(out); a.lse = const_cast<float*>(lse); a.d_out = (const bf16*)dout;
    a.dq = (bf16*)dq; a.dk = (bf16*)dk; a.dv = (bf16*)dv;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    dim3 grid((a.L + ATT_BLK - 1) / ATT_BLK, a.H, a.B);
    if (d->D / d->H == 32) {
        GRB_TRY(set_smem(sas_attn_bwd_dq_kernel<32>, sizeof(SasSmem<32>)));
        GRB_TRY(set_smem(sas_attn_bwd_dkdv_kernel<32>, sizeof(SasSmem<32>)));
        launch_k(sas_attn_bwd_dq_kernel<32>, grid, ATT_THREADS, sizeof(SasSmem<32>), st, a);
        launch_k(sas_attn_bwd_dkdv_kernel<32>, grid, ATT_THREADS, sizeof(SasSmem<32>), st, a);
    } else {
        GRB_TRY(set_smem(sas_attn_bwd_dq_kernel<64>, sizeof(SasSmem<64>)));
        GRB_TRY(set_smem(sas_attn_bwd_dkdv_kernel<64>, sizeof(SasSmem<64>)));
        launch_k(sas_attn_bwd_dq_kernel<64>, grid, ATT_THREADS, sizeof(SasSmem<64>), st, a);
        launch_k(sas_attn_bwd_dkdv_kernel<64>, grid, ATT_THREADS, sizeof(SasSmem<64>), st, a);
    }
    GRB_CUDA(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------------ generic fused linear pieces
int grb_linear_forward(const void* x_bf16, const void* w_bf16, const float* bias, int T, int N, int K, int act, void* z_bf16,
                       void* act_bf16, float dropout_p, uint64_t seed, const uint64_t* seed_dev, uint32_t site, void* stream) {
    GRB_REQUIRE(x_bf16 && w_bf16 && bias && z_bf16, "null argument");
    GRB_REQUIRE(T > 0 && N % 8 == 0 && K % 8 == 0, "N and K must be multiples of 8");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    Dropout drop = make_dropout(dropout_p, seed, site, seed_dev);
    GRB_REQUIRE(act >= 0 && act <= 2, "unknown activation %d", act);
    GRB_REQUIRE(act == 0 || act_bf16, "act output is null");
    GRB_CUDA(gemm_bias_act(act, (const bf16*)x_bf16, (const bf16*)w_bf16, bias, (bf16*)z_bf16, (bf16*)act_bf16, T, N, K, drop, st));
    return 0;
}
int grb_linear_residual_forward(const void* x_bf16, const void* w_bf16, const float* bias, const float* residual, const float* row_scale,
                                int T, int N, int K, float* y, float dropout_p, uint64_t seed, const uint64_t* seed_dev, uint32_t site,
                                void* stream) {
    GRB_REQUIRE(x_bf16 && w_bf16 && bias && residual && y, "null argument");
    GRB_REQUIRE(T > 0 && N % 8 == 0 && K % 8 == 0, "N and K must be multiples of 8");
    GRB_CUDA(gemm_bias_res((const bf16*)x_bf16, (const bf16*)w_bf16, bias, residual, row_scale, y, T, N, K,
                           make_dropout(dropout_p, seed, site, seed_dev), static_cast<cudaStream_t>(stream)));
    return 0;
}
int grb_linear_backward(const void* dy_bf16, const void* w_bf16, const void* x_bf16, int T, int N, int K, float* dx_f32,
                        const float* dx_residual, float* dw, float* db, void* stream) {
    GRB_REQUIRE(dy_bf16 && w_bf16, "null argument");
    GRB_REQUIRE(T > 0 && N % 8 == 0 && K % 8 == 0, "N and K must be multiples of 8");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (db) GRB_TRY(colsum((const bf16*)dy_bf16, T, N, N, db, st));
    if (dw) {
        GRB_REQUIRE(x_bf16, "x is null");
        GRB_CUDA(gemm_tn_atomic((const bf16*)dy_bf16, (const bf16*)x_bf16, dw, N, K, T, N, K, st));
    }
    if (dx_f32) {
        GRB_CUDA(gemm_nn_f32((const bf16*)dy_bf16, (const bf16*)w_bf16, dx_f32, dx_residual, 1.f, T, K, N, N, K, st));
    }
    return 0;
}

namespace {
__global__ void dact_kernel(bf16* g, const bf16* z, size_t n, int act) {
    pdl_wait();
    size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 2;
    size_t stride = (size_t)gridDim.x * blockDim.x * 2;
    for (; i < n; i += stride) {
        float2 gv = unpack_bf16(*reinterpret_cast<const uint32_t*>(g + i));
        float2 zv = unpack_bf16(*reinterpret_cast<const uint32_t*>(z + i));
        float d0 = act == 1 ? dsiluf(zv.x) : (zv.x > 0.f ? 1.f : 0.f);
        float d1 = act == 1 ? dsiluf(zv.y) : (zv.y > 0.f ? 1.f : 0.f);
        *reinterpret_cast<uint32_t*>(g + i) = pack_bf16(gv.x * d0, gv.y * d1);
    }
}
}  // namespace
int grb_dact(const void* g_bf16_in_out, const void* z_bf16, size_t n, int act, void* stream) {
    GRB_REQUIRE(g_bf16_in_out && z_bf16 && n % 2 == 0 && (act == 1 || act == 2), "bad argument");
    size_t blocks = (n / 2 + 255) / 256;
    if (blocks > (size_t)sm_count() * 16) blocks = (size_t)sm_count() * 16;
    launch_k(dact_kernel, (unsigned)(blocks ? blocks : 1), 256, 0, static_cast<cudaStream_t>(stream), (bf16*)const_cast<void*>(g_bf16_in_out), (const bf16*)z_bf16, n, act);
    GRB_CUDA(cudaGetLastError());
    return 0;
}

int grb_linear_dact_backward(const void* dy_bf16, const void* w_bf16, const void* z_bf16, int T, int N, int K, int act, float dropout_p,
                             uint64_t seed, const uint64_t* seed_dev, uint32_t site, void* g_bf16, void* stream) {
    GRB_REQUIRE(dy_bf16 && w_bf16 && z_bf16 && g_bf16, "null argument");
    GRB_REQUIRE(T > 0 && N % 8 == 0 && K % 8 == 0 && (act == 1 || act == 2), "bad argument");
    GRB_CUDA(gemm_dact(act, (const bf16*)dy_bf16, (const bf16*)w_bf16, (const bf16*)z_bf16, (bf16*)g_bf16, T, K, N,
                       make_dropout(dropout_p, seed, site, seed_dev), static_cast<cudaStream_t>(stream)));
    return 0;
}
int grb_cast_rows_f32_to_bf16(const float* in, void* out_bf16, int T, int D, const float* row_scale, float dropout_p, uint64_t seed,
                              const uint64_t* seed_dev, uint32_t site, void* stream) {
    GRB_REQUIRE(in && out_bf16 && T > 0 && D > 0 && D % 4 == 0, "bad argument");
    return cast_bf16(in, (bf16*)out_bf16, (size_t)T * D, D, make_dropout(dropout_p, seed, site, seed_dev), row_scale,
                     static_cast<cudaStream_t>(stream));
}

int grb_layernorm_forward(const float* x, const float* g, const float* b, float eps, int T, int D, void* y_bf16, float* y_f32,
                          float* stats, void* stream) {
    GRB_REQUIRE(x && g && b && (y_bf16 || y_f32), "null argument");
    LnFwdArgs a{x, g, b, (bf16*)y_bf16, y_f32, stats, T, D, eps};
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    GRB_ROW_DISPATCH(D, ln_fwd_kernel, a, T, st);
    return 0;
}
int grb_layernorm_backward(const float* dy, const float* x, const float* stats, const float* g, const float* residual, int T, int D,
                           float* dx, float* dg, float* db, void* stream) {
    GRB_REQUIRE(dy && x && stats && g && dx && dg && db, "null argument");
    LnBwdArgs a{dy, x, stats, g, residual, dx, dg, db, T, D};
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    GRB_ROW_DISPATCH(D, ln_bwd_kernel, a, T, st);
    return 0;
}

int grb_split3_f32_to_bf16(const float* in, void* out_bf16, size_t rows, int K, int operand, void* stream) {
    GRB_REQUIRE(in && out_bf16 && K > 0 && (operand == 0 || operand == 1), "bad argument");
    if (rows == 0) return 0;
    size_t blocks = (rows * (size_t)K + 255) / 256;
    if (blocks > (size_t)sm_count() * 16) blocks = (size_t)sm_count() * 16;
    launch_k(split3_f32_bf16_kernel, (unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream), in, (bf16*)out_bf16, rows, K, operand);
    GRB_CUDA(cudaGetLastError());
    return 0;
}
static int linear_f32x3(const bf16* xs, const bf16* ws, const float* bias, const float* res2, int T, int N, int K, int act, float* y, int ldy,
                        cudaStream_t st) {
    const int K6 = 6 * K;
    // Two accumulators.  The tensor core adds each K = 16 group into the fp32 accumulator with truncation, an error relative to
    // the running sum per step: 288 steps over the six-term K (K = 768) measured 2e-5.  The five small cross terms (<= 2^-8 of
    // the result) are therefore summed on their own (their truncation is 2^-8 smaller), and the hi*hi term, K/16 steps, is
    // added to that sum in the epilogue of a second pass together with bias, activation and residual.  y doubles as the scratch of pass 1.
    GRB_CUDA((launch_tc_gemm<0, 0>(xs + K, ws + K, T, N, 5 * K, K6, K6, 1, TcEpiF32{nullptr, ldy, 1.f}, y, nullptr, ldy, sm_count(), st)));
    if (act == 1) GRB_CUDA((launch_tc_gemm<0, 0>(xs, ws, T, N, K, K6, K6, 1, TcEpiActResF32<1>{y, ldy, bias, res2}, y, nullptr, ldy, sm_count(), st)));
    else GRB_CUDA((launch_tc_gemm<0, 0>(xs, ws, T, N, K, K6, K6, 1, TcEpiActResF32<0>{y, ldy, bias, res2}, y, nullptr, ldy, sm_count(), st)));
    return 0;
}
int grb_linear_f32x3_forward(const void* x_split_bf16, const void* w_split_bf16, int T, int N, int K, int act, float* y, void* stream) {
    GRB_REQUIRE(x_split_bf16 && w_split_bf16 && y, "null argument");
    GRB_REQUIRE(T > 0 && N % 4 == 0 && K % 8 == 0 && (act == 0 || act == 1), "bad shape T=%d N=%d K=%d act=%d", T, N, K, act);
    GRB_REQUIRE(aligned16(x_split_bf16) && aligned16(w_split_bf16) && aligned16(y), "buffers must be 16-byte aligned");
    return linear_f32x3((const bf16*)x_split_bf16, (const bf16*)w_split_bf16, nullptr, nullptr, T, N, K, act, y, N, static_cast<cudaStream_t>(stream));
}
int grb_linear_f32x3_bias_forward(const void* x_split_bf16, const void* w_split_bf16, const float* bias, const float* residual, int T, int N,
                                  int K, int act, float* y, int ldy, void* stream) {
    GRB_REQUIRE(x_split_bf16 && w_split_bf16 && y, "null argument");
    GRB_REQUIRE(T > 0 && N > 0 && ldy >= N && ldy % 4 == 0 && K % 8 == 0 && (act == 0 || act == 1), "bad shape T=%d N=%d K=%d ldy=%d act=%d", T, N, K, ldy, act);
    GRB_REQUIRE(aligned16(x_split_bf16) && aligned16(w_split_bf16) && aligned16(y) && (!residual || aligned16(residual)), "buffers must be 16-byte aligned");
    return linear_f32x3((const bf16*)x_split_bf16, (const bf16*)w_split_bf16, bias, residual, T, N, K, act, y, ldy, static_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------------------------------------------ fp32-exact HSTU block, forward
struct LayerF32Work {
    bf16* xs; float* P; float* O; float* x1; float* xn; float* h; bf16* hs; size_t bytes;
};
static LayerF32Work carve_f32(void* base, size_t T, size_t D) {
    LayerF32Work w;
    size_t off = 0;
    auto take = [&](size_t n) { void* p = base ? (char*)base + off : nullptr; off += (n + 255) & ~size_t(255); return p; };
    w.xs = (bf16*)take(T * 6 * D * 2);
    w.P = (float*)take(T * 4 * D * 4);
    w.O = (float*)take(T * D * 4);
    w.x1 = (float*)take(T * D * 4);
    w.xn = (float*)take(T * D * 4);
    w.h = (float*)take(T * 4 * D * 4);
    w.hs = (bf16*)take(T * 24 * D * 2);
    w.bytes = off;
    return w;
}
size_t grb_hstu_layer_f32_workspace_bytes(const grb_hstu_dims* d) {
    if (!d || d->B <= 0 || d->L <= 0 || d->D <= 0) return 0;
    return carve_f32(nullptr, (size_t)d->B * d->L, d->D).bytes;
}
int grb_hstu_layer_forward_f32(const grb_hstu_dims* d, const grb_hstu_layer_params_f32* p, const grb_hstu_seq* s, const float* x, float* y,
                               void* workspace, void* stream) {
    GRB_TRY(check_dims(d));
    GRB_REQUIRE(p && s && x && y && workspace, "null argument");
    GRB_REQUIRE(p->proj_w_split && p->proj_b && p->pos_table && p->ln1_g && p->ln1_b && p->ffn1_w_split && p->ffn1_b && p->ffn2_w_split &&
                    p->ffn2_b && p->ln2_g && p->ln2_b, "null parameter pointer");
    GRB_REQUIRE(s->bias_index && s->ld_index >= d->L && s->ld_index % 8 == 0, "the fp32 path reads the [B, L, ld] bias index matrix");
    GRB_REQUIRE(aligned16(x) && aligned16(y) && aligned16(workspace), "buffers must be 16-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int T = d->B * d->L, D = d->D, DH = D / d->H;
    LayerF32Work w = carve_f32(workspace, T, D);
    GRB_TRY(join_pending(st));
    // P = silu(x Wp^T + bp)                                                                   (hstu.py:234-235)
    GRB_TRY(grb_split3_f32_to_bf16(x, w.xs, T, D, 0, stream));
    GRB_TRY(linear_f32x3(w.xs, (const bf16*)p->proj_w_split, p->proj_b, nullptr, T, 4 * D, D, 1, w.P, 4 * D, st));
    // O = silu(Q K^T + bias) V                                                                (hstu.py:244-267)
    {
        HstuAttnF32Args a{w.P, 4 * D, d->B, d->L, d->H, {}, w.O};
        // same conventions as make_attn_args(): uniform position buckets collapse to one effective bucket
        a.bias.wpos = p->pos_table + (s->pos_uniform ? (size_t)s->pos_bucket0 * d->H : 0);
        const bool has_time = p->time_table != nullptr && s->has_time && d->ntime > 0;
        a.bias.wtime = has_time ? p->time_table : nullptr;
        a.bias.bias_index = s->bias_index; a.bias.ldix = s->ld_index;
        a.bias.npos = s->pos_uniform ? 1 : d->npos; a.bias.ntime = has_time ? d->ntime : 0;
        a.bias.pos_uniform = s->pos_uniform; a.bias.pos_bucket0 = 0;
        int rc = DH == 32 ? launch_hstu_attn_f32<32>(a, st) : launch_hstu_attn_f32<64>(a, st);
        GRB_REQUIRE(rc == 0, "fp32 attention launch failed");
    }
    // x1 = x + LN1(O) * U ; xn = LN2(x1)                                                      (hstu.py:271-278)
    {
        LnGateF32Args a{w.O, w.P, 4 * D, x, p->ln1_g, p->ln1_b, p->ln2_g, p->ln2_b, w.x1, w.xn, T, 1e-5f};
        const int grid = row_grid(T);
        if (D == 64) launch_k(ln_gate_f32_kernel<2>, grid, 256, 0, st, a);
        else if (D == 128) launch_k(ln_gate_f32_kernel<4>, grid, 256, 0, st, a);
        else launch_k(ln_gate_f32_kernel<8>, grid, 256, 0, st, a);
        GRB_CUDA(cudaGetLastError());
    }
    // y = x1 + (silu(xn W1^T + b1) W2^T + b2)                                                 (hstu.py:210-214, :278)
    GRB_TRY(grb_split3_f32_to_bf16(w.xn, w.xs, T, D, 0, stream));
    GRB_TRY(linear_f32x3(w.xs, (const bf16*)p->ffn1_w_split, p->ffn1_b, nullptr, T, 4 * D, D, 1, w.h, 4 * D, st));
    GRB_TRY(grb_split3_f32_to_bf16(w.h, w.hs, T, 4 * D, 0, stream));
    GRB_TRY(linear_f32x3(w.hs, (const bf16*)p->ffn2_w_split, p->ffn2_b, w.x1, T, D, 4 * D, 0, y, D, st));
    return 0;
}
int grb_layernorm_f32_forward(const float* x, const float* g, const float* b, float eps, int T, int D, float* y, void* stream) {
    GRB_REQUIRE(x && g && b && y && T > 0 && (D == 64 || D == 128 || D == 256), "bad argument T=%d D=%d", T, D);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int grid = row_grid(T);
    if (D == 64) launch_k(ln_f32_kernel<2>, grid, 256, 0, st, x, g, b, y, T, eps);
    else if (D == 128) launch_k(ln_f32_kernel<4>, grid, 256, 0, st, x, g, b, y, T, eps);
    else launch_k(ln_f32_kernel<8>, grid, 256, 0, st, x, g, b, y, T, eps);
    GRB_CUDA(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------------ T5-style attention core (TIGER)
static int t5_args(T5AttnArgs& a, const void* q, const void* k, const void* v, int B, int Lq, int Lk, int H, int DH, int ldq, int ldk, int ldv,
                   const float* bias, const int32_t* bucket, int nb, const uint8_t* key_pad, int causal, float scale, float p, uint64_t seed,
                   const uint64_t* seed_dev, uint32_t site) {
    GRB_REQUIRE(q && k && v, "null argument");
    GRB_REQUIRE(B > 0 && Lq > 0 && Lk > 0 && H > 0 && (DH == 32 || DH == 64), "bad shape B=%d Lq=%d Lk=%d H=%d head_dim=%d", B, Lq, Lk, H, DH);
    GRB_REQUIRE(ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0 && aligned16(q) && aligned16(k) && aligned16(v), "rows must be 16-byte aligned");
    GRB_REQUIRE((bias == nullptr) == (bucket == nullptr) && (!bias || (nb > 0 && nb <= 1024)), "bias table and bucket map go together");
    GRB_REQUIRE(p >= 0.f && p < 1.f, "dropout_p out of range");
    memset(&a, 0, sizeof(a));
    a.q = (const bf16*)q; a.k = (const bf16*)k; a.v = (const bf16*)v; a.ldq = ldq; a.ldk = ldk; a.ldv = ldv;
    a.B = B; a.Lq = Lq; a.Lk = Lk; a.H = H; a.bias = bias; a.bucket = bucket; a.nb = bias ? nb : 0; a.key_pad = key_pad; a.causal = causal;
    a.scale = scale; a.drop = make_dropout(p, seed, site, seed_dev);
    return 0;
}
int grb_t5_attention_forward(const void* q, const void* k, const void* v, int B, int Lq, int Lk, int H, int head_dim, int ldq, int ldk, int ldv,
                             const float* bias, const int32_t* bucket, int num_buckets, const uint8_t* key_pad, int causal, float scale,
                             float dropout_p, uint64_t seed, const uint64_t* seed_dev, uint32_t site, void* out, int ldo, float* lse,
                             void* stream) {
    T5AttnArgs a;
    GRB_TRY(t5_args(a, q, k, v, B, Lq, Lk, H, head_dim, ldq, ldk, ldv, bias, bucket, num_buckets, key_pad, causal, scale, dropout_p, seed, seed_dev, site));
    GRB_REQUIRE(out && lse && ldo % 8 == 0 && aligned16(out), "bad output");
    a.out = (bf16*)out; a.ldo = ldo; a.lse = lse;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    dim3 grid((Lq + T5_ROWS - 1) / T5_ROWS, B * H);
    if (head_dim == 32) {
        const size_t smem = t5_fwd_smem<32>(a.nb);
        GRB_TRY(set_smem(t5_attn_fwd_kernel<32>, smem));
        launch_k(t5_attn_fwd_kernel<32>, grid, T5_THREADS, smem, st, a);
    } else {
        const size_t smem = t5_fwd_smem<64>(a.nb);
        GRB_TRY(set_smem(t5_attn_fwd_kernel<64>, smem));
        launch_k(t5_attn_fwd_kernel<64>, grid, T5_THREADS, smem, st, a);
    }
    GRB_CUDA(cudaGetLastError());
    return 0;
}
int grb_t5_attention_backward(const void* q, const void* k, const void* v, int B, int Lq, int Lk, int H, int head_dim, int ldq, int ldk, int ldv,
                              const float* bias, const int32_t* bucket, int num_buckets, const uint8_t* key_pad, int causal, float scale,
                              float dropout_p, uint64_t seed, const uint64_t* seed_dev, uint32_t site, const void* out, int ldo,
                              const float* lse, const void* dout, int lddo, void* dq, int lddq, float* dk, float* dv, float* dbias,
                              void* stream) {
    T5AttnArgs a;
    GRB_TRY(t5_args(a, q, k, v, B, Lq, Lk, H, head_dim, ldq, ldk, ldv, bias, bucket, num_buckets, key_pad, causal, scale, dropout_p, seed, seed_dev, site));
    GRB_REQUIRE(out && lse && dout && dq && dk && dv && ldo % 8 == 0 && lddo % 8 == 0 && lddq % 8 == 0, "bad argument");
    GRB_REQUIRE(aligned16(out) && aligned16(dout) && aligned16(dq), "rows must be 16-byte aligned");
    a.out = (bf16*)const_cast<void*>(out); a.ldo = ldo; a.lse = const_cast<float*>(lse); a.dout = (const bf16*)dout; a.lddo = lddo;
    a.dq = (bf16*)dq; a.lddq = lddq; a.dk = dk; a.dv = dv; a.dbias = bias ? dbias : nullptr;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    GRB_CUDA(cudaMemsetAsync(dk, 0, (size_t)B * Lk * H * head_dim * sizeof(float), st));
    GRB_CUDA(cudaMemsetAsync(dv, 0, (size_t)B * Lk * H * head_dim * sizeof(float), st));
    dim3 grid((Lq + T5_ROWS - 1) / T5_ROWS, B * H);
    if (head_dim == 32) {
        const size_t smem = t5_bwd_smem<32>(a.nb);
        GRB_TRY(set_smem(t5_attn_bwd_kernel<32>, smem));
        launch_k(t5_attn_bwd_kernel<32>, grid, T5_THREADS, smem, st, a);
    } else {
        const size_t smem = t5_bwd_smem<64>(a.nb);
        GRB_TRY(set_smem(t5_attn_bwd_kernel<64>, smem));
        launch_k(t5_attn_bwd_kernel<64>, grid, T5_THREADS, smem, st, a);
    }
    GRB_CUDA(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------------ TIGER constrained beam step
int grb_trie_log_softmax(const float* logits, int rows, int V, const int32_t* node, const int32_t* child_off, const int32_t* child_tok,
                         int n_nodes, int use_trie, int vocab_offset, int num_embeddings, float temperature, float* probs, float* logp,
                         void* stream) {
    GRB_REQUIRE(logits && probs && logp && rows >= 0 && V > 0 && V <= 1 << 20, "bad argument rows=%d V=%d", rows, V);
    GRB_REQUIRE(!use_trie || (node && child_off && n_nodes > 0), "trie arrays missing");
    GRB_REQUIRE(temperature > 0.f, "temperature must be positive");
    if (rows == 0) return 0;
    TrieCsr t{child_off, child_tok, nullptr, n_nodes};
    const size_t smem = (size_t)((V + 31) / 32) * 4;
    launch_k(trie_log_softmax_kernel, rows, 256, smem, static_cast<cudaStream_t>(stream), logits, V, node, t, use_trie, vocab_offset,
             num_embeddings, temperature, probs, logp);
    GRB_CUDA(cudaGetLastError());
    return 0;
}
int grb_beam_select(const int64_t* beam_seqs, const float* beam_logps, const int64_t* cand_tok, const float* cand_logp, const int32_t* nodes,
                    const int32_t* child_off, const int32_t* child_tok, const int32_t* child_node, int n_nodes, int B, int K, int KK, int S,
                    int64_t* new_seqs, float* new_logps, int32_t* new_nodes, void* stream) {
    GRB_REQUIRE(beam_logps && cand_tok && cand_logp && new_seqs && new_logps && (S == 0 || beam_seqs), "null argument");
    GRB_REQUIRE(B >= 0 && K >= 1 && K <= 32 && KK >= 1 && K * KK <= BEAM_MAX_CAND && S >= 0, "bad shape B=%d K=%d KK=%d S=%d (K <= 32, K*KK <= 1024)", B, K, KK, S);
    GRB_REQUIRE(!new_nodes || (nodes && child_off && child_tok && child_node && n_nodes > 0), "trie arrays missing");
    if (B == 0) return 0;
    BeamSelectArgs a{reinterpret_cast<const long long*>(beam_seqs), beam_logps, reinterpret_cast<const long long*>(cand_tok), cand_logp, nodes,
                     TrieCsr{child_off, child_tok, child_node, n_nodes}, K, KK, S, reinterpret_cast<long long*>(new_seqs), new_logps, new_nodes};
    launch_k(beam_select_kernel, B, BEAM_MAX_CAND, 0, static_cast<cudaStream_t>(stream), a);
    GRB_CUDA(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------------ optimizer / casts
int grb_cast_f32_to_bf16(const float* in, void* out_bf16, size_t n, void* stream) {
    GRB_REQUIRE(in && out_bf16, "null argument");
    if (n == 0) return 0;
    size_t blocks = (n + 255) / 256;
    if (blocks > (size_t)sm_count() * 16) blocks = (size_t)sm_count() * 16;
    launch_k(cast_flat_f32_bf16_kernel, (unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream), in, (bf16*)out_bf16, n);
    GRB_CUDA(cudaGetLastError());
    return 0;
}
int grb_adam_step(float* p, float* g, float* m, float* v, void* p_bf16, size_t n, float* state, float lr, float beta1, float beta2,
                  float eps, float weight_decay, float grad_scale, int zero_grad, void* stream) {
    GRB_REQUIRE(p && g && m && v && state, "null argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    launch_k(adam_tick_kernel, 1, 1, 0, st, state, beta1, beta2);
    GRB_CUDA(cudaGetLastError());
    if (n == 0) return 0;
    AdamArgs a{p, g, m, v, (bf16*)p_bf16, n, state, lr, beta1, beta2, eps, weight_decay, grad_scale, zero_grad};
    size_t blocks = (n + 255) / 256;
    if (blocks > (size_t)sm_count() * 16) blocks = (size_t)sm_count() * 16;
    launch_k(adam_step_kernel, (unsigned)blocks, 256, 0, st, a);
    GRB_CUDA(cudaGetLastError());
    return 0;
}

int grb_dp_adam_step(float* p, float* g, float* m, float* v, void* p_bf16, const void* mc_g, void* mc_p, void* mc_p_bf16,
                     const void* peer_g, const void* peer_p, const void* peer_p_bf16, const void* peer_sig, void* sig, void* epoch,
                     size_t n, int rank, int world, float* state, float lr, float beta1, float beta2, float eps, float weight_decay,
                     float grad_scale, void* stream) {
    GRB_REQUIRE(p && g && m && v && p_bf16 && peer_sig && sig && epoch && state, "null argument");
    GRB_REQUIRE(world >= 2 && world <= 32 && rank >= 0 && rank < world, "bad rank/world %d/%d", rank, world);
    GRB_REQUIRE(n > 0 && n % ((size_t)8 * world) == 0, "n must be a multiple of 8 * world");
    const bool mc = mc_g != nullptr && mc_p != nullptr && mc_p_bf16 != nullptr;
    GRB_REQUIRE(mc || (peer_g && peer_p && peer_p_bf16), "neither multicast addresses nor peer pointer arrays given");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    launch_k(adam_tick_kernel, 1, 1, 0, st, state, beta1, beta2);
    GRB_CUDA(cudaGetLastError());
    launch_k(dp_barrier_kernel, 1, 32, 0, st, reinterpret_cast<unsigned* const*>(peer_sig), reinterpret_cast<unsigned*>(sig),
             reinterpret_cast<unsigned*>(epoch), rank, world, 0);
    GRB_CUDA(cudaGetLastError());
    DpAdamArgs a{p, g, m, v, (bf16*)p_bf16, (const float*)mc_g, (float*)mc_p, (bf16*)mc_p_bf16,
                 reinterpret_cast<const float* const*>(peer_g), reinterpret_cast<float* const*>(peer_p), reinterpret_cast<bf16* const*>(peer_p_bf16),
                 n, rank, world, state, lr, beta1, beta2, eps, weight_decay, grad_scale};
    size_t blocks = (n / world / 8 + 255) / 256;
    if (blocks > (size_t)sm_count() * 4) blocks = (size_t)sm_count() * 4;
    if (blocks < 1) blocks = 1;
    if (mc) launch_k(dp_adam_kernel<true>, (unsigned)blocks, 256, 0, st, a);
    else launch_k(dp_adam_kernel<false>, (unsigned)blocks, 256, 0, st, a);
    GRB_CUDA(cudaGetLastError());
    launch_k(dp_barrier_kernel, 1, 32, 0, st, reinterpret_cast<unsigned* const*>(peer_sig), reinterpret_cast<unsigned*>(sig),
             reinterpret_cast<unsigned*>(epoch), rank, world, 1);
    GRB_CUDA(cudaGetLastError());
    GRB_CUDA(cudaMemsetAsync(g, 0, n * sizeof(float), st));
    return 0;
}

namespace {
__global__ void assert_unit_scalar_kernel(const float* v) {
    pdl_wait();
    if (*v != 1.0f) {
        printf("genrec_b200: the loss was back-propagated with gradient %g, but FlatAdam(unit_loss_grad=True) promised 1\n", (double)*v);
        __trap();
    }
}
}  // namespace
int grb_assert_unit_scalar(const float* value, void* stream) {
    GRB_REQUIRE(value, "null argument");
    launch_k(assert_unit_scalar_kernel, 1, 1, 0, static_cast<cudaStream_t>(stream), value);
    GRB_CUDA(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------------ RQ-VAE
int grb_rq_residual_argmin(const float* x, const float* codebooks, int64_t N, int D, int K, int levels, float commitment, int64_t* ids,
                           float* emb, float* res, float* loss, float* res_out, void* stream) {
    GRB_REQUIRE(x && codebooks && ids, "null argument");
    GRB_REQUIRE(N >= 0 && levels >= 1 && K >= 2 && K % 2 == 0, "bad shape N=%lld K=%d levels=%d", (long long)N, K, levels);
    GRB_REQUIRE(D == 32 || D == 64, "latent dim %d unsupported (32, 64)", D);
    GRB_REQUIRE((size_t)K * (D + 1) * 4 <= 200 * 1024, "codebook level does not fit shared memory (K=%d, D=%d)", K, D);
    GRB_REQUIRE(aligned16(x) && aligned16(codebooks), "buffers must be 16-byte aligned");
    if (N == 0) return 0;
    RqArgs a{x, codebooks, reinterpret_cast<long long*>(ids), emb, res, loss, res_out, (long long)N, K, levels, commitment};
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    GRB_REQUIRE(emb == nullptr || aligned16(emb), "emb must be 16-byte aligned");
    GRB_REQUIRE(res == nullptr || aligned16(res), "res must be 16-byte aligned");
    // Three kernels (rq_argmin.cuh).  Default: the register-blocked tile kernel (D = 32, K a multiple of 256, tile fits shared
    // memory).  GRB_RQ = tile | split | thread forces one; split / thread are the earlier generations, kept as cross-checks
    // (tests/test_rq_gpu.py compares all three) and for the shapes the tile kernel does not cover.
    const char* rq_env = getenv("GRB_RQ");
    const bool force_thread = rq_env != nullptr && strcmp(rq_env, "thread") == 0;
    const bool force_split = rq_env != nullptr && strcmp(rq_env, "split") == 0;
    {
        const bool stage = emb != nullptr || res != nullptr;
        const size_t smem = rq_tile_smem_bytes(D, K, levels, stage);
        if (!force_thread && !force_split && D == 32 && K % 256 == 0 && smem <= 220 * 1024) {
            GRB_TRY(set_smem(rq_residual_argmin_tile_kernel<32>, smem));
            const unsigned grid = (unsigned)((N + RQT_ROWS - 1) / RQT_ROWS);
            launch_k(rq_residual_argmin_tile_kernel<32>, grid, RQT_THREADS, smem, st, a);
            GRB_CUDA(cudaGetLastError());
            return 0;
        }
    }
    const bool legacy = force_thread || (!force_split && N > (int64_t)sm_count() * RQ_THREADS * 4);
    if (!legacy && K % 8 == 0) {
        // four threads per row (see rq_argmin.cuh); two rows per thread once there is more than a wave of work (FMA : LDS = 8 : 1)
        const int rows = (D == 32 && N > (int64_t)sm_count() * RQ_ROWS_PER_CTA * 4) ? 2 : 1;
        const size_t base = ((size_t)K * D + ((K + 3) & ~3)) * sizeof(float);
        const size_t stage = (emb || res) ? (size_t)2 * RQ_ROWS_PER_CTA * rows * D * levels * sizeof(float) : 0;
        const bool staged = stage > 0 && base + stage <= 200 * 1024;
        const size_t smem = base + (staged ? stage : 0);
        const unsigned grid = (unsigned)((N + (int64_t)RQ_ROWS_PER_CTA * rows - 1) / ((int64_t)RQ_ROWS_PER_CTA * rows));
        auto go = [&](auto kern) -> int {
            GRB_TRY(set_smem(kern, smem));
            launch_k(kern, grid, RQ_THREADS, smem, st, a);
            return 0;
        };
        if (D == 32) {
            if (rows == 2) GRB_TRY(staged ? go(rq_residual_argmin_split_kernel<32, 2, true>) : go(rq_residual_argmin_split_kernel<32, 2, false>));
            else GRB_TRY(staged ? go(rq_residual_argmin_split_kernel<32, 1, true>) : go(rq_residual_argmin_split_kernel<32, 1, false>));
        } else {
            GRB_TRY(staged ? go(rq_residual_argmin_split_kernel<64, 1, true>) : go(rq_residual_argmin_split_kernel<64, 1, false>));
        }
        GRB_CUDA(cudaGetLastError());
        return 0;
    }
    size_t smem = (size_t)K * (D + 1) * sizeof(float);
    if (D == 32) {
        // two rows per thread once there is more than a wave of work; one row per thread for small N (more CTAs)
        if (N > (int64_t)sm_count() * RQ_THREADS * 2) {
            unsigned grid = (unsigned)((N + 2 * RQ_THREADS - 1) / (2 * RQ_THREADS));
            GRB_TRY(set_smem(rq_residual_argmin_kernel<32, 2>, smem));
            launch_k(rq_residual_argmin_kernel<32, 2>, grid, RQ_THREADS, smem, st, a);
        } else {
            unsigned grid = (unsigned)((N + RQ_THREADS - 1) / RQ_THREADS);
            GRB_TRY(set_smem(rq_residual_argmin_kernel<32, 1>, smem));
            launch_k(rq_residual_argmin_kernel<32, 1>, grid, RQ_THREADS, smem, st, a);
        }
    } else {
        unsigned grid = (unsigned)((N + RQ_THREADS - 1) / RQ_THREADS);
        GRB_TRY(set_smem(rq_residual_argmin_kernel<64, 1>, smem));
        launch_k(rq_residual_argmin_kernel<64, 1>, grid, RQ_THREADS, smem, st, a);
    }
    GRB_CUDA(cudaGetLastError());
    return 0;
}

}  // extern "C"
