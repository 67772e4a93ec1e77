// C ABI (include/milagro_bls_b200.h) and host-side orchestration of the verification path.
// Single translation unit: the device headers carry __constant__ tables with internal linkage.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <dlfcn.h>
#include <nccl.h>   // types only: the library is bound at run time (dlopen), see nccl()

#include <algorithm>
#include <condition_variable>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/milagro_bls_b200.h"
#undef B3_OK
#undef B3_ERR_INVALID_POINT
#undef B3_ERR_INVALID_YFLAG
#include "kernels.cuh"

static const uint8_t kDstG2[] = "BLS_SIG_BLS12381G2_XMD:SHA-256_SSWU_RO_POP_";   // A/bls381/proof_of_possession.rs:38
static const size_t kDstG2Len = 43;

#define B3_MAX_MARKS 24
// sets from which the key aggregation uses 4 lanes per set instead of 8 (less shuffle-tree overhead, twice the latency)
static const size_t kAggG4Min = 4096;
#define B3_MSM_MIN_SETS 512     // below this, S = sum [c_j] sig_j uses n separate ladders + a tree
#define B3_N_STAGES 12
// stage ids (b3_ctx_stage_ms / b3_stage_name)
enum { ST_SIG_CHECK = 0, ST_AGGREGATE, ST_G1_MUL, ST_HASH_TO_G2, ST_G2_MUL_SUM, ST_MILLER, ST_FP12_PRODUCT, ST_FINAL_EXP, ST_COPY, ST_MILLER_LINES, ST_MILLER_LINES_SUMS, ST_END };
static const char* kStageNames[B3_N_STAGES] = {"g2_parse_subgroup_check", "g1_aggregate", "g1_scalar_mul_affine", "hash_to_g2_affine",
                                               "g2_scalar_mul_sum", "miller_accumulate", "miller_chain", "final_exp", "parse_copies", "miller_lines",
                                               "miller_lines_signature_sums", "end"};

struct dev_buf {
    void* p = nullptr;
    size_t cap = 0;
};

struct b3_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    std::string err;
    uint64_t launches = 0;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};   // 0/1: whole call, 2/3: Miller kernel
    float last_ms[2] = {0.f, 0.f};
    // stage spans of the most recent verification call: span i = [span_a[i], span_b[i]] on the stream the stage ran on
    cudaEvent_t span_a[B3_MAX_MARKS], span_b[B3_MAX_MARKS];
    int span_id[B3_MAX_MARKS];
    int n_spans = 0;
    float stage_ms[B3_N_STAGES];
    // independent stages of verify_multiple run concurrently on aux streams (fork/join by events) unless serial != 0
    cudaStream_t aux[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr, ev_fork2 = nullptr, ev_fork3 = nullptr, ev_join[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_sync = nullptr;  // blocking-sync event: the host thread of a call SLEEPS while it waits (see sync())
    bool sig_pending = false;       // the subgroup checks of the call run on aux[0] beside the closing chain: join before reading first_bad
    int serial = 0;
    int latency_mode = 0;           // chain kernels: 0 = replicated lanes (quad.cuh) when this is the only call in flight on the device, 1 = always, 2 = never
    bool wide_now = false;          // decision for the call being enqueued
    int trusted = 0;                // 1: key / signature arrays come from the library's own validated outputs: skip the on-curve checks of the aggregation kernels
    int item_kernel = 0;            // b3_verify_batch finishing kernel: 0 = by batch size, 1 = CTA per item, 3 = lane pair per item
    // scratch (grown on demand, reused across calls)
    dev_buf in_a, in_b, in_c, in_d, in_e, in_f;      // staged host inputs
    dev_buf g1j, g1j2, g1a, g2a_sig, g2j, g2j2, g2j_h, g2a, g2q, g1pp, qinf, f12a, f12b, lines, status, ok, misc, outb;
    dev_buf msm;                    // the signature MSM's digit sort: per-window index lists and bucket starts
    dev_buf part;                   // this rank's packed partial (sharded calls)
    dev_buf loc_lines, loc_qinf, loc_pp;   // b3_verify_multiple_locate only: signature lines, their qinf, unscaled keys in pairing form
    dev_buf in_g, grp;              // grouped calls: the sets' message indices; the sort by message and the group bounds
    uint8_t* d_dst = nullptr;
    void* pin = nullptr;            // pinned host staging for the status read-back of a verify_multiple call
    size_t pin_cap = 0;
    long long h_init[2] = {0, 0};   // source of the small host-to-device initialisations (must outlive the async copy)
    size_t pre_n = (size_t)-1;      // number of signatures parsed + checked by b3_sig_precheck, (size_t)-1 = none
    size_t loc_n = (size_t)-1;      // n of the whole verify_multiple call b3_verify_multiple_locate may read, (size_t)-1 = none
    bool loc_accept = false;        // ... and whether that call accepted
    size_t loc_np = 0;              // ... the pair count of its line table (the stride of H's lines)
    const uint32_t* loc_idx = nullptr;   // ... and for a grouped call the message index of every set (H's pair), else null
};

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            ctx->err = std::string(#call) + ": " + cudaGetErrorString(_e);                         \
            return B3_ERR_CUDA;                                                                    \
        }                                                                                          \
    } while (0)
#define CKR(expr)                      \
    do {                               \
        int _r = (expr);               \
        if (_r != B3_OK) return _r;    \
    } while (0)

static int ensure(b3_ctx* ctx, dev_buf& b, size_t bytes) {
    if (bytes <= b.cap) return B3_OK;
    if (b.p) CK(cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
    size_t cap = bytes + bytes / 4 + 256;
    CK(cudaMalloc(&b.p, cap));
    b.cap = cap;
    return B3_OK;
}
static inline unsigned nblk(size_t n, int tpb = B3_TPB) { return (unsigned)((n + tpb - 1) / tpb); }
#define LAUNCH(kern, grid, block, ...)                       \
    do {                                                     \
        kern<<<(grid), (block), 0, ctx->stream>>>(__VA_ARGS__); \
        ctx->launches++;                                     \
    } while (0)

#define LAUNCH_ON(strm, kern, grid, block, ...)              \
    do {                                                     \
        kern<<<(grid), (block), 0, (strm)>>>(__VA_ARGS__);   \
        ctx->launches++;                                     \
    } while (0)
// A chain kernel over n items in the lane layout P, or in the replicated layout W when `wide` (quad.cuh): kern_of(L) is the
// kernel's instantiation for layout L, which runs n << L::shift threads.
template <class P, class W, class KernOf, class... A>
static void launch_lanes(b3_ctx* ctx, cudaStream_t strm, bool wide, size_t n, KernOf kern_of, A... args) {
    if (wide) LAUNCH_ON(strm, kern_of(W()), nblk(n << W::shift), B3_TPB, args...);
    else LAUNCH_ON(strm, kern_of(P()), nblk(n << P::shift), B3_TPB, args...);
}
// An aggregation kernel over n_sets sets with G lanes per set: kern_of(std::integral_constant<int, G>) is its instantiation.
// Enough lanes to fill the chip, few enough to keep the shuffle tree short (4 from g4_min sets: the tree runs at <= half the
// lanes, so fewer lanes per set waste less).
template <class KernOf, class... A>
static void launch_agg(b3_ctx* ctx, cudaStream_t strm, size_t n_sets, size_t total_keys, size_t g4_min, KernOf kern_of, A... args) {
    const size_t avg = total_keys / n_sets;
    if (n_sets >= g4_min || avg <= 8) LAUNCH_ON(strm, kern_of(std::integral_constant<int, 4>()), nblk(n_sets * 4), B3_TPB, args...);
    else if (n_sets >= 2048 || avg <= 32) LAUNCH_ON(strm, kern_of(std::integral_constant<int, 8>()), nblk(n_sets * 8), B3_TPB, args...);
    else LAUNCH_ON(strm, kern_of(std::integral_constant<int, 32>()), nblk(n_sets * 32), B3_TPB, args...);
}

extern "C" void b3_ctx_destroy(b3_ctx* ctx);
extern "C" int b3_ctx_create(int device, b3_ctx** out) {
    if (!out) return B3_ERR_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) return B3_ERR_CUDA;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return B3_ERR_CUDA;
    if (prop.major != 10) return B3_ERR_CUDA;        // sm_100a code only: no other path exists
    if (cudaSetDevice(device) != cudaSuccess) return B3_ERR_CUDA;
    b3_ctx* ctx = new b3_ctx();
    ctx->device = device;
    for (int i = 0; i < B3_MAX_MARKS; i++) { ctx->span_a[i] = nullptr; ctx->span_b[i] = nullptr; }
    // Priorities (lower number = served first): the context's own stream carries the END of every call (Miller
    // accumulation, closing chain, final exponentiation -- single-CTA kernels that must not queue behind the wide kernels
    // of other contexts' batches), aux[2] the longest dependent chain of a batch (hash_to_G2 -> Miller point chains).
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    const int prio_mid = prio_hi < prio_lo ? prio_hi + 1 : prio_hi;
    bool ok = cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, prio_hi) == cudaSuccess;
    for (int i = 0; ok && i < 4; i++) ok = cudaEventCreate(&ctx->ev[i]) == cudaSuccess;
    for (int i = 0; ok && i < B3_MAX_MARKS; i++) ok = cudaEventCreate(&ctx->span_a[i]) == cudaSuccess && cudaEventCreate(&ctx->span_b[i]) == cudaSuccess;
    for (int i = 0; ok && i < 4; i++)
        ok = cudaStreamCreateWithPriority(&ctx->aux[i], cudaStreamNonBlocking, i == 2 ? prio_mid : prio_lo) == cudaSuccess &&
             cudaEventCreateWithFlags(&ctx->ev_join[i], cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&ctx->ev_fork2, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&ctx->ev_fork3, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&ctx->ev_sync, cudaEventDisableTiming | cudaEventBlockingSync) == cudaSuccess;
    for (int i = 0; i < B3_N_STAGES; i++) ctx->stage_ms[i] = 0.f;
    ok = ok && cudaMalloc((void**)&ctx->d_dst, 256) == cudaSuccess;
    ok = ok && cudaMemcpy(ctx->d_dst, kDstG2, kDstG2Len, cudaMemcpyHostToDevice) == cudaSuccess;
    if (!ok) {                                        // one exit for every partial construction: destroy skips what is null
        cudaGetLastError();
        b3_ctx_destroy(ctx);
        return B3_ERR_CUDA;
    }
    *out = ctx;
    return B3_OK;
}
extern "C" void b3_ctx_destroy(b3_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (int i = 0; i < 4; i++) if (ctx->aux[i]) cudaStreamSynchronize(ctx->aux[i]);
    dev_buf* bufs[] = {&ctx->in_a, &ctx->in_b, &ctx->in_c, &ctx->in_d, &ctx->in_e, &ctx->in_f, &ctx->g1j, &ctx->g1j2, &ctx->g1a,
                       &ctx->g2a_sig, &ctx->g2j, &ctx->g2j2, &ctx->g2j_h, &ctx->g2a, &ctx->g2q, &ctx->g1pp, &ctx->qinf, &ctx->lines, &ctx->f12a, &ctx->f12b, &ctx->status, &ctx->ok,
                       &ctx->misc, &ctx->outb, &ctx->msm, &ctx->part, &ctx->loc_lines, &ctx->loc_qinf, &ctx->loc_pp, &ctx->in_g, &ctx->grp};
    if (ctx->pin) cudaFreeHost(ctx->pin);
    for (dev_buf* b : bufs) if (b->p) cudaFree(b->p);
    if (ctx->d_dst) cudaFree(ctx->d_dst);
    for (int i = 0; i < 4; i++) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    for (int i = 0; i < B3_MAX_MARKS; i++) {
        if (ctx->span_a[i]) cudaEventDestroy(ctx->span_a[i]);
        if (ctx->span_b[i]) cudaEventDestroy(ctx->span_b[i]);
    }
    for (int i = 0; i < 4; i++) {
        if (ctx->aux[i]) cudaStreamDestroy(ctx->aux[i]);
        if (ctx->ev_join[i]) cudaEventDestroy(ctx->ev_join[i]);
    }
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_fork2) cudaEventDestroy(ctx->ev_fork2);
    if (ctx->ev_fork3) cudaEventDestroy(ctx->ev_fork3);
    if (ctx->ev_sync) cudaEventDestroy(ctx->ev_sync);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    cudaGetLastError();
    delete ctx;
}
extern "C" const char* b3_last_error(b3_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }
extern "C" void* b3_ctx_stream(b3_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
extern "C" uint64_t b3_ctx_launch_count(b3_ctx* ctx) { return ctx ? ctx->launches : 0; }
extern "C" float b3_ctx_last_kernel_ms(b3_ctx* ctx, int which) { return (ctx && which >= 0 && which < 2) ? ctx->last_ms[which] : 0.f; }
extern "C" float b3_ctx_stage_ms(b3_ctx* ctx, int stage) { return (ctx && stage >= 0 && stage < B3_N_STAGES) ? ctx->stage_ms[stage] : 0.f; }
extern "C" const char* b3_stage_name(int stage) { return (stage >= 0 && stage < B3_N_STAGES) ? kStageNames[stage] : ""; }
extern "C" int b3_stage_count(void) { return B3_N_STAGES - 1; }
extern "C" void b3_ctx_set_serial(b3_ctx* ctx, int serial) { if (ctx) ctx->serial = serial; }
extern "C" void b3_ctx_set_item_kernel(b3_ctx* ctx, int which) { if (ctx) ctx->item_kernel = which; }
extern "C" void b3_ctx_set_trusted_points(b3_ctx* ctx, int trusted) { if (ctx) ctx->trusted = trusted; }
extern "C" void b3_ctx_set_latency_mode(b3_ctx* ctx, int mode) { if (ctx && mode >= 0 && mode <= 2) ctx->latency_mode = mode; }
// verification calls in flight per device (all contexts of the process): a call that is alone on its GPU cannot fill it with
// one item per set, so its chain kernels run in the replicated form (twice the lanes per item, ~25 % more arithmetic);
// with several calls in flight the plain kernels give the higher throughput.
#include <atomic>
static std::atomic<int> g_calls_in_flight[64];
struct call_guard {
    b3_ctx* ctx;
    explicit call_guard(b3_ctx* c, size_t n) : ctx(c) {
        const int others = g_calls_in_flight[ctx->device & 63].fetch_add(1);
        ctx->wide_now = ctx->latency_mode == 1 || (ctx->latency_mode == 0 && others == 0 && n <= 16384);
    }
    ~call_guard() { g_calls_in_flight[ctx->device & 63].fetch_sub(1); }
};
static void mark_reset(b3_ctx* ctx) { ctx->n_spans = 0; }
// open a stage span on `strm`; returns the span index (or -1 when the table is full)
static int span_begin(b3_ctx* ctx, int id, cudaStream_t strm) {
    if (ctx->n_spans >= B3_MAX_MARKS) return -1;
    int i = ctx->n_spans++;
    ctx->span_id[i] = id;
    cudaEventRecord(ctx->span_a[i], strm);
    return i;
}
static void span_end(b3_ctx* ctx, int i, cudaStream_t strm) {
    if (i >= 0) cudaEventRecord(ctx->span_b[i], strm);
}
// after a stream synchronize: fold the spans into per-stage durations
static void mark_collect(b3_ctx* ctx) {
    for (int i = 0; i < B3_N_STAGES; i++) ctx->stage_ms[i] = 0.f;
    for (int i = 0; i < ctx->n_spans; i++) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ctx->span_a[i], ctx->span_b[i]) == cudaSuccess) ctx->stage_ms[ctx->span_id[i]] += ms;
    }
    cudaGetLastError();
}

static int h2d(b3_ctx* ctx, dev_buf& b, const void* src, size_t bytes) {
    CKR(ensure(ctx, b, bytes ? bytes : 1));
    if (bytes) CK(cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return B3_OK;
}
static int d2h(b3_ctx* ctx, void* dst, const void* src, size_t bytes) {
    if (bytes) CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return B3_OK;
}
// Wait for the context's stream.  The waiting host thread BLOCKS on a blocking-sync event instead of spinning in
// cudaStreamSynchronize: the drop-in model is one host thread per call in flight (eight per GPU in bench.py), and on an
// 8-GPU box 64 spinning threads on 32 cores starve the threads that launch kernels (measured: 8.1 M sets/s at N = 8
// spinning).  B3_SPIN_SYNC=1 restores the spinning wait.
static int sync(b3_ctx* ctx) {
    static const bool spin = getenv("B3_SPIN_SYNC") && atoi(getenv("B3_SPIN_SYNC")) != 0;
    if (spin) {
        CK(cudaStreamSynchronize(ctx->stream));
    } else {
        CK(cudaEventRecord(ctx->ev_sync, ctx->stream));
        CK(cudaEventSynchronize(ctx->ev_sync));
    }
    CK(cudaGetLastError());
    return B3_OK;
}
// point arrays handed over as DEVICE pointers must be 16-byte aligned (the kernels read and write them with LDG.128 /
// STG.128); cudaMalloc'ed arrays and any record-aligned offset into them are
static int dev_aligned(b3_ctx* ctx, const void* p) {
    if ((reinterpret_cast<uintptr_t>(p) & 15u) == 0) return B3_OK;
    ctx->err = "device point arrays must be 16-byte aligned";
    return B3_ERR_ARG;
}
static int begin(b3_ctx* ctx) {
    if (!ctx) return B3_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    ctx->wide_now = false;                    // set per call by the call_guard of the verify_multiple entries
    ctx->loc_n = (size_t)-1;                  // any call may overwrite what b3_verify_multiple_locate reads (vm_whole re-enables it)
    return B3_OK;
}

// ---------------------------------------------------------------------------------------------- generic pieces
// product of n Fp12 values in `a` (scratch `b`), result left in *res (device pointer into a or b)
static int fp12_product(b3_ctx* ctx, fp12* a, fp12* b, size_t n, fp12** res) {
    fp12 *src = a, *dst = b;
    while (n > 1) {
        size_t m = (n + 1) / 2;
        LAUNCH(k_fp12_mul_pairs, nblk(m), B3_TPB, src, n, dst);
        fp12* t = src; src = dst; dst = t;
        n = m;
    }
    *res = src;
    return B3_OK;
}
// sum of n G2 points in `a` (scratch `b`) by a pairwise tree, result left in *res; with keep > 1 the tree stops at `keep`
// points, each the sum of n / keep consecutive inputs when n / keep is a power of two
static int g2_sum(b3_ctx* ctx, g2_jac* a, g2_jac* b, size_t n, g2_jac** res, cudaStream_t strm = nullptr, size_t keep = 1) {
    g2_jac *src = a, *dst = b;
    if (!strm) strm = ctx->stream;
    while (n > keep) {
        size_t m = (n + 1) / 2;
        LAUNCH_ON(strm, k_g2_add_pairs, nblk(2 * m), B3_TPB, src, n, dst);
        g2_jac* t = src; src = dst; dst = t;
        n = m;
    }
    *res = src;
    return B3_OK;
}
// Split multi-Miller loop (pairing.cuh), step 1: point chains of pairs [first, first + count) of an n_pairs product
// -> lines in HBM (68 x n_pairs x 288 B) and qinf (n_pairs x u32).  May be issued on any stream as soon as those q's exist.
static int miller_lines(b3_ctx* ctx, cudaStream_t strm, const g2_jac* q, size_t n_pairs, size_t first, size_t count, dev_buf& lines, dev_buf& qinf) {
    if (count == 0) return B3_OK;
    int sp = span_begin(ctx, count <= 64 && first > 0 ? ST_MILLER_LINES_SUMS : ST_MILLER_LINES, strm);   // the few pairs of the signature MSM are timed apart
    // few pairs (the window sums of the signature MSM): always latency-bound
    launch_lanes<lanes_pair, lanes_quad>(ctx, strm, ctx->wide_now || count <= 64, count, [](auto L) { return k_miller_lines<decltype(L)>; },
                                         q, n_pairs, first, count, (fp2*)lines.p, (uint32_t*)qinf.p);
    span_end(ctx, sp, strm);
    return B3_OK;
}
static int miller_reserve(b3_ctx* ctx, size_t n_pairs, dev_buf& lines, dev_buf& qinf) {
    CKR(ensure(ctx, lines, sizeof(fp2) * 3 * B3_MILLER_SLOTS * (n_pairs ? n_pairs : 1)));
    CKR(ensure(ctx, qinf, 4 * (n_pairs ? n_pairs : 1)));
    return B3_OK;
}
// steps 2 and 3 (context stream): per-slot accumulation over all pairs, one cooperative closing chain -> *res
// K pairs per accumulating six-lane group, 20 groups per CTA (k_miller_accum)
static void miller_shape(size_t n_pairs, size_t* chunks_out, unsigned* K_out) {
    static const unsigned kTargetK = getenv("B3_ACC_K") ? (unsigned)atoi(getenv("B3_ACC_K")) : 32u;
    size_t chunks = (n_pairs + (size_t)B3_ACC_GROUPS * kTargetK - 1) / ((size_t)B3_ACC_GROUPS * kTargetK);
    if (chunks < 1) chunks = 1;
    if (chunks > 64) chunks = 64;
    unsigned K = (unsigned)((n_pairs + chunks * B3_ACC_GROUPS - 1) / (chunks * B3_ACC_GROUPS));
    if (K < 1) K = 1;
    *chunks_out = chunks;
    *K_out = K;
}
static int miller_finish_reserve(b3_ctx* ctx, size_t n_pairs) {
    size_t chunks;
    unsigned K;
    miller_shape(n_pairs, &chunks, &K);
    return ensure(ctx, ctx->f12a, sizeof(fp12) * (B3_MILLER_SLOTS * (chunks + 1) + 2));
}
// step 2: the accumulation kernel (wide: fills the GPU); step 3 (miller_close): slot products and the closing chain (one CTA)
static int miller_accumulate(b3_ctx* ctx, const g1_pp* p, size_t n_pairs, fp12** res) {
    size_t chunks;
    unsigned K;
    miller_shape(n_pairs, &chunks, &K);
    CKR(miller_finish_reserve(ctx, n_pairs));
    fp12* partial = (fp12*)ctx->f12a.p;
    fp12* slotvals = partial + B3_MILLER_SLOTS * chunks;
    fp12* out = slotvals + B3_MILLER_SLOTS;
    *res = out;
    if (n_pairs == 0) return B3_OK;
    CK(cudaEventRecord(ctx->ev[2], ctx->stream));
    int sp = span_begin(ctx, ST_MILLER, ctx->stream);
    LAUNCH(k_miller_accum, dim3((unsigned)chunks, B3_MILLER_SLOTS), B3_TPB, (const fp2*)ctx->lines.p, (const uint32_t*)ctx->qinf.p, p, n_pairs, K, partial);
    span_end(ctx, sp, ctx->stream);
    CK(cudaEventRecord(ctx->ev[3], ctx->stream));
    return B3_OK;
}
static int miller_close(b3_ctx* ctx, size_t n_pairs) {
    size_t chunks;
    unsigned K;
    miller_shape(n_pairs, &chunks, &K);
    fp12* partial = (fp12*)ctx->f12a.p;
    fp12* slotvals = partial + B3_MILLER_SLOTS * chunks;
    fp12* out = slotvals + B3_MILLER_SLOTS;
    if (n_pairs == 0) {
        LAUNCH(k_fp12_set_one, 1, 1, out);
        return B3_OK;
    }
    int sp = span_begin(ctx, ST_FP12_PRODUCT, ctx->stream);
    if (chunks > 1) {
        LAUNCH(k_miller_slots, B3_MILLER_SLOTS, B3_COOP_THREADS, (const fp12*)partial, (unsigned)chunks, slotvals);
        LAUNCH(k_miller_chain, 1, B3_COOP_THREADS, (const fp12*)slotvals, 1u, out);
    } else {
        LAUNCH(k_miller_chain, 1, B3_COOP_THREADS, (const fp12*)partial, 1u, out);
    }
    span_end(ctx, sp, ctx->stream);
    return B3_OK;
}
static int miller_finish(b3_ctx* ctx, const g1_pp* p, size_t n_pairs, fp12** res) {
    CKR(miller_accumulate(ctx, p, n_pairs, res));
    return miller_close(ctx, n_pairs);
}
// whole product on the context stream
static int miller_product(b3_ctx* ctx, const g2_jac* q, const g1_pp* p, size_t n_pairs, fp12** res) {
    CKR(miller_reserve(ctx, n_pairs, ctx->lines, ctx->qinf));
    CKR(miller_lines(ctx, ctx->stream, q, n_pairs, 0, n_pairs, ctx->lines, ctx->qinf));
    return miller_finish(ctx, p, n_pairs, res);
}
// final exponentiation of *m -> accept / gt on the host
static int finish(b3_ctx* ctx, const fp12* m, int* accept, uint8_t* gt576) {
    CKR(ensure(ctx, ctx->outb, 576 + 16));
    uint8_t* d_gt = (uint8_t*)ctx->outb.p;
    int32_t* d_one = (int32_t*)(d_gt + 576);
    int sp = span_begin(ctx, ST_FINAL_EXP, ctx->stream);
    LAUNCH(k_final_exp, 1, B3_COOP_THREADS, m, d_gt, d_one);
    span_end(ctx, sp, ctx->stream);
    CK(cudaEventRecord(ctx->ev[1], ctx->stream));
    int32_t one = 0;
    uint8_t gt[576];
    CKR(d2h(ctx, &one, d_one, 4));
    CKR(d2h(ctx, gt, d_gt, 576));
    CKR(sync(ctx));
    cudaEventElapsedTime(&ctx->last_ms[0], ctx->ev[0], ctx->ev[1]);
    if (cudaEventElapsedTime(&ctx->last_ms[1], ctx->ev[2], ctx->ev[3]) != cudaSuccess) ctx->last_ms[1] = 0.f;
    cudaGetLastError();
    mark_collect(ctx);
    if (gt576) memcpy(gt576, gt, 576);
    if (accept) *accept = one ? 1 : 0;
    return B3_OK;
}
// host copy of a status array; returns the first non-zero code or B3_OK
static int first_status(b3_ctx* ctx, const int32_t* d_status, size_t n) {
    std::vector<int32_t> h(n);
    CKR(d2h(ctx, h.data(), d_status, 4 * n));
    CKR(sync(ctx));
    for (size_t i = 0; i < n; i++) if (h[i]) return h[i];
    return B3_OK;
}
// G1 key aggregation on `strm`
static int launch_g1_aggregate(b3_ctx* ctx, cudaStream_t strm, const uint8_t* d_pks, const uint32_t* d_off, size_t n_sets, size_t total_keys,
                               g1_jac* d_out, int32_t* d_status) {
    if (n_sets == 0) return B3_OK;
    const int chk = ctx->trusted ? 0 : 1;
    launch_agg(ctx, strm, n_sets, total_keys, kAggG4Min, [](auto g) { return k_g1_aggregate<decltype(g)::value>; }, d_pks, d_off, n_sets, d_out,
               d_status, chk);
    return B3_OK;
}

// ---------------------------------------------------------------------------------------------- serialisation API
extern "C" int b3_g1_decompress(b3_ctx* ctx, const uint8_t* in48, size_t n, int validate, uint8_t* out96, int32_t* status) {
    CKR(begin(ctx));
    if (n == 0) return B3_OK;
    if (!in48 || !out96 || !status) return B3_ERR_ARG;
    CKR(h2d(ctx, ctx->in_a, in48, 48 * n));
    CKR(ensure(ctx, ctx->outb, 96 * n));
    CKR(ensure(ctx, ctx->status, 4 * n));
    LAUNCH(k_g1_decompress, nblk(n), B3_TPB, (const uint8_t*)ctx->in_a.p, n, validate, (uint8_t*)ctx->outb.p, (int32_t*)ctx->status.p);
    CKR(d2h(ctx, out96, ctx->outb.p, 96 * n));
    CKR(d2h(ctx, status, ctx->status.p, 4 * n));
    return sync(ctx);
}
extern "C" int b3_g2_decompress(b3_ctx* ctx, const uint8_t* in96, size_t n, uint8_t* out192, int32_t* status) {
    CKR(begin(ctx));
    if (n == 0) return B3_OK;
    if (!in96 || !out192 || !status) return B3_ERR_ARG;
    CKR(h2d(ctx, ctx->in_a, in96, 96 * n));
    CKR(ensure(ctx, ctx->outb, 192 * n));
    CKR(ensure(ctx, ctx->status, 4 * n));
    LAUNCH(k_g2_decompress, nblk(n), B3_TPB, (const uint8_t*)ctx->in_a.p, n, (uint8_t*)ctx->outb.p, (int32_t*)ctx->status.p);
    CKR(d2h(ctx, out192, ctx->outb.p, 192 * n));
    CKR(d2h(ctx, status, ctx->status.p, 4 * n));
    return sync(ctx);
}
extern "C" int b3_g1_compress(b3_ctx* ctx, const uint8_t* in96, size_t n, uint8_t* out48, int32_t* status) {
    CKR(begin(ctx));
    if (n == 0) return B3_OK;
    if (!in96 || !out48 || !status) return B3_ERR_ARG;
    CKR(h2d(ctx, ctx->in_a, in96, 96 * n));
    CKR(ensure(ctx, ctx->outb, 48 * n));
    CKR(ensure(ctx, ctx->status, 4 * n));
    LAUNCH(k_g1_compress, nblk(n), B3_TPB, (const uint8_t*)ctx->in_a.p, n, (uint8_t*)ctx->outb.p, (int32_t*)ctx->status.p);
    CKR(d2h(ctx, out48, ctx->outb.p, 48 * n));
    CKR(d2h(ctx, status, ctx->status.p, 4 * n));
    return sync(ctx);
}
extern "C" int b3_g2_compress(b3_ctx* ctx, const uint8_t* in192, size_t n, uint8_t* out96, int32_t* status) {
    CKR(begin(ctx));
    if (n == 0) return B3_OK;
    if (!in192 || !out96 || !status) return B3_ERR_ARG;
    CKR(h2d(ctx, ctx->in_a, in192, 192 * n));
    CKR(ensure(ctx, ctx->outb, 96 * n));
    CKR(ensure(ctx, ctx->status, 4 * n));
    LAUNCH(k_g2_compress, nblk(n), B3_TPB, (const uint8_t*)ctx->in_a.p, n, (uint8_t*)ctx->outb.p, (int32_t*)ctx->status.p);
    CKR(d2h(ctx, out96, ctx->outb.p, 96 * n));
    CKR(d2h(ctx, status, ctx->status.p, 4 * n));
    return sync(ctx);
}
extern "C" int b3_g1_validate(b3_ctx* ctx, const uint8_t* in96, size_t n, int32_t* status, int32_t* valid) {
    CKR(begin(ctx));
    if (n == 0) return B3_OK;
    if (!in96 || !status || !valid) return B3_ERR_ARG;
    CKR(h2d(ctx, ctx->in_a, in96, 96 * n));
    CKR(ensure(ctx, ctx->g1j, sizeof(g1_jac) * n));
    CKR(ensure(ctx, ctx->status, 4 * n));
    CKR(ensure(ctx, ctx->ok, 4 * n));
    LAUNCH(k_g1_parse, nblk(n), B3_TPB, (const uint8_t*)ctx->in_a.p, n, (g1_jac*)ctx->g1j.p, (int32_t*)ctx->status.p, 1);
    LAUNCH(k_g1_key_validate, nblk(n), B3_TPB, (const g1_jac*)ctx->g1j.p, (const int32_t*)ctx->status.p, n, (int32_t*)ctx->ok.p);
    CKR(d2h(ctx, status, ctx->status.p, 4 * n));
    CKR(d2h(ctx, valid, ctx->ok.p, 4 * n));
    return sync(ctx);
}
extern "C" int b3_g2_subgroup_check(b3_ctx* ctx, const uint8_t* in192, size_t n, int32_t* status, int32_t* ok) {
    CKR(begin(ctx));
    if (n == 0) return B3_OK;
    if (!in192 || !status || !ok) return B3_ERR_ARG;
    CKR(h2d(ctx, ctx->in_a, in192, 192 * n));
    CKR(ensure(ctx, ctx->g2a_sig, sizeof(g2_aff) * n));
    CKR(ensure(ctx, ctx->status, 4 * n));
    CKR(ensure(ctx, ctx->ok, 4 * n));
    LAUNCH(k_g2_parse, nblk(n), B3_TPB, (const uint8_t*)ctx->in_a.p, n, (g2_aff*)ctx->g2a_sig.p, (int32_t*)ctx->status.p, 1);
    LAUNCH(k_g2_subgroup<lanes_pair>, nblk(2 * n), B3_TPB, (const g2_aff*)ctx->g2a_sig.p, (const int32_t*)ctx->status.p, n, (int32_t*)ctx->ok.p);
    CKR(d2h(ctx, status, ctx->status.p, 4 * n));
    CKR(d2h(ctx, ok, ctx->ok.p, 4 * n));
    return sync(ctx);
}

// ---------------------------------------------------------------------------------------------- aggregation API
extern "C" int b3_g1_aggregate_dev(b3_ctx* ctx, const uint8_t* pks96_dev, const uint32_t* off_dev, size_t n_sets, uint8_t* out96_dev,
                                   int32_t* status_dev) {
    CKR(begin(ctx));
    if (n_sets == 0) return B3_OK;
    CKR(dev_aligned(ctx, pks96_dev));
    CKR(dev_aligned(ctx, out96_dev));
    CKR(ensure(ctx, ctx->g1j, sizeof(g1_jac) * n_sets));
    CKR(ensure(ctx, ctx->g1a, sizeof(g1_aff) * n_sets));
    uint32_t total = 0;
    CK(cudaMemcpyAsync(&total, off_dev + n_sets, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CKR(sync(ctx));
    CKR(launch_g1_aggregate(ctx, ctx->stream, pks96_dev, off_dev, n_sets, total, (g1_jac*)ctx->g1j.p, status_dev));
    LAUNCH(k_g1_to_affine, nblk((n_sets + norm_per(n_sets) - 1) / norm_per(n_sets)), B3_TPB, (const g1_jac*)ctx->g1j.p, n_sets, (g1_aff*)ctx->g1a.p, norm_per(n_sets));
    LAUNCH(k_g1_aff_to_wire, nblk(n_sets), B3_TPB, (const g1_aff*)ctx->g1a.p, n_sets, out96_dev);
    return sync(ctx);
}
extern "C" int b3_g1_aggregate(b3_ctx* ctx, const uint8_t* pks96, const uint32_t* off, size_t n_sets, uint8_t* out96, int32_t* status) {
    CKR(begin(ctx));
    if (n_sets == 0) return B3_OK;
    if (!off || !out96 || !status) return B3_ERR_ARG;
    size_t total = off[n_sets];
    CKR(h2d(ctx, ctx->in_a, pks96, 96 * total));
    CKR(h2d(ctx, ctx->in_b, off, 4 * (n_sets + 1)));
    CKR(ensure(ctx, ctx->outb, 96 * n_sets));
    CKR(ensure(ctx, ctx->status, 4 * n_sets));
    CKR(b3_g1_aggregate_dev(ctx, (const uint8_t*)ctx->in_a.p, (const uint32_t*)ctx->in_b.p, n_sets, (uint8_t*)ctx->outb.p, (int32_t*)ctx->status.p));
    CKR(d2h(ctx, out96, ctx->outb.p, 96 * n_sets));
    CKR(d2h(ctx, status, ctx->status.p, 4 * n_sets));
    return sync(ctx);
}
extern "C" int b3_g2_aggregate(b3_ctx* ctx, const uint8_t* sigs192, const uint32_t* off, size_t n_sets, uint8_t* out192, int32_t* status) {
    CKR(begin(ctx));
    if (n_sets == 0) return B3_OK;
    if (!off || !out192 || !status) return B3_ERR_ARG;
    size_t total = off[n_sets];
    CKR(h2d(ctx, ctx->in_a, sigs192, 192 * total));
    CKR(h2d(ctx, ctx->in_b, off, 4 * (n_sets + 1)));
    CKR(ensure(ctx, ctx->outb, 192 * n_sets));
    CKR(ensure(ctx, ctx->status, 4 * n_sets));
    CKR(ensure(ctx, ctx->g2j, sizeof(g2_jac) * n_sets));
    CKR(ensure(ctx, ctx->g2a, sizeof(g2_aff) * n_sets));
    const int chk = ctx->trusted ? 0 : 1;
    launch_agg(ctx, ctx->stream, n_sets, total, 16384, [](auto g) { return k_g2_aggregate<decltype(g)::value>; }, (const uint8_t*)ctx->in_a.p,
               (const uint32_t*)ctx->in_b.p, n_sets, (g2_jac*)ctx->g2j.p, (int32_t*)ctx->status.p, chk);
    LAUNCH(k_g2_to_affine, nblk((n_sets + norm_per(n_sets) - 1) / norm_per(n_sets)), B3_TPB, (const g2_jac*)ctx->g2j.p, n_sets, (g2_aff*)ctx->g2a.p, norm_per(n_sets));
    LAUNCH(k_g2_aff_to_wire, nblk(n_sets), B3_TPB, (const g2_aff*)ctx->g2a.p, n_sets, (uint8_t*)ctx->outb.p);
    CKR(d2h(ctx, out192, ctx->outb.p, 192 * n_sets));
    CKR(d2h(ctx, status, ctx->status.p, 4 * n_sets));
    return sync(ctx);
}

// ---------------------------------------------------------------------------------------------- hash_to_g2 API
static int stage_dst(b3_ctx* ctx, const uint8_t* dst, size_t dst_len, const uint8_t** d_dst, uint32_t* len) {
    if (!dst) { *d_dst = ctx->d_dst; *len = (uint32_t)kDstG2Len; return B3_OK; }
    if (dst_len > 255) return B3_ERR_HASH_TO_FIELD;    // oversize-DST hashing is never reached through milagro_bls
    CKR(h2d(ctx, ctx->misc, dst, dst_len));
    *d_dst = (const uint8_t*)ctx->misc.p;
    *len = (uint32_t)dst_len;
    return B3_OK;
}
// hash_to_curve_g2 left in Jacobian coordinates (pair members of the Miller loop are never normalised)
static int hash_to_g2_jac_dev(b3_ctx* ctx, cudaStream_t strm, const uint8_t* d_msgs, const uint32_t* d_off, size_t n, g2_jac* d_out) {
    LAUNCH_ON(strm, k_hash_to_g2, nblk(2 * n), B3_TPB, d_msgs, d_off, n, (const uint8_t*)ctx->d_dst, (uint32_t)kDstG2Len, d_out);
    return B3_OK;
}
static int hash_to_g2_affine_dev(b3_ctx* ctx, cudaStream_t strm, const uint8_t* d_msgs, const uint32_t* d_off, size_t n, const uint8_t* d_dst,
                                 uint32_t dst_len, g2_aff* d_out) {
    CKR(ensure(ctx, ctx->g2j_h, sizeof(g2_jac) * n));
    LAUNCH_ON(strm, k_hash_to_g2, nblk(2 * n), B3_TPB, d_msgs, d_off, n, d_dst, dst_len, (g2_jac*)ctx->g2j_h.p);
    LAUNCH_ON(strm, k_g2_to_affine, nblk((n + norm_per(n) - 1) / norm_per(n)), B3_TPB, (const g2_jac*)ctx->g2j_h.p, n, d_out, norm_per(n));
    return B3_OK;
}
extern "C" int b3_hash_to_g2_dev(b3_ctx* ctx, const uint8_t* msgs_dev, const uint32_t* off_dev, size_t n, uint8_t* out192_dev) {
    CKR(begin(ctx));
    if (n == 0) return B3_OK;
    CKR(dev_aligned(ctx, out192_dev));
    CKR(ensure(ctx, ctx->g2a, sizeof(g2_aff) * n));
    CK(cudaEventRecord(ctx->ev[0], ctx->stream));
    mark_reset(ctx);
    int sp = span_begin(ctx, ST_HASH_TO_G2, ctx->stream);
    CKR(hash_to_g2_affine_dev(ctx, ctx->stream, msgs_dev, off_dev, n, ctx->d_dst, (uint32_t)kDstG2Len, (g2_aff*)ctx->g2a.p));
    span_end(ctx, sp, ctx->stream);
    sp = span_begin(ctx, ST_COPY, ctx->stream);
    LAUNCH(k_g2_aff_to_wire, nblk(n), B3_TPB, (const g2_aff*)ctx->g2a.p, n, out192_dev);
    span_end(ctx, sp, ctx->stream);
    CK(cudaEventRecord(ctx->ev[1], ctx->stream));
    CKR(sync(ctx));
    mark_collect(ctx);
    cudaEventElapsedTime(&ctx->last_ms[0], ctx->ev[0], ctx->ev[1]);
    return B3_OK;
}
extern "C" int b3_hash_to_g2(b3_ctx* ctx, const uint8_t* msgs, const uint32_t* off, size_t n, const uint8_t* dst, size_t dst_len, uint8_t* out192) {
    CKR(begin(ctx));
    if (n == 0) return B3_OK;
    if (!off || !out192) return B3_ERR_ARG;
    const uint8_t* d_dst;
    uint32_t dl;
    CKR(stage_dst(ctx, dst, dst_len, &d_dst, &dl));
    CKR(h2d(ctx, ctx->in_a, msgs, off[n]));
    CKR(h2d(ctx, ctx->in_b, off, 4 * (n + 1)));
    CKR(ensure(ctx, ctx->g2a, sizeof(g2_aff) * n));
    CKR(ensure(ctx, ctx->outb, 192 * n));
    CKR(hash_to_g2_affine_dev(ctx, ctx->stream, (const uint8_t*)ctx->in_a.p, (const uint32_t*)ctx->in_b.p, n, d_dst, dl, (g2_aff*)ctx->g2a.p));
    LAUNCH(k_g2_aff_to_wire, nblk(n), B3_TPB, (const g2_aff*)ctx->g2a.p, n, (uint8_t*)ctx->outb.p);
    CKR(d2h(ctx, out192, ctx->outb.p, 192 * n));
    return sync(ctx);
}

// ---------------------------------------------------------------------------------------------- verification
// Shared tail of Signature::verify / fast_aggregate_verify* : pairs (sig, -G1), (H(msg), key).
//   d_sig: parsed signature (g2_aff), d_key: key as g1_jac.  reject_inf_key: the aggregate-key-at-infinity rule.
static int verify_two_pairs(b3_ctx* ctx, const g2_aff* d_sig, const int32_t* d_sig_ok, const g1_jac* d_key, int reject_inf_key,
                            const uint8_t* msg, size_t msg_len, int* accept, uint8_t* gt576) {
    uint32_t off[2] = {0, (uint32_t)msg_len};
    CKR(h2d(ctx, ctx->in_c, msg, msg_len));
    CKR(h2d(ctx, ctx->in_d, off, 8));
    CKR(ensure(ctx, ctx->g2q, sizeof(g2_jac) * 2));
    CKR(ensure(ctx, ctx->g1pp, sizeof(g1_pp) * 2));
    g2_jac* q = (g2_jac*)ctx->g2q.p;
    g1_pp* p = (g1_pp*)ctx->g1pp.p;
    // pair 0: (sig, -G1)
    LAUNCH(k_g2_aff_to_jac, 1, B3_TPB, d_sig, 1, q);
    LAUNCH(k_set_neg_g1_pp, 1, 1, p);
    // pair 1: (H(msg), key)
    CKR(hash_to_g2_jac_dev(ctx, ctx->stream, (const uint8_t*)ctx->in_c.p, (const uint32_t*)ctx->in_d.p, 1, q + 1));
    LAUNCH(k_g1_jac_to_pp, 1, B3_TPB, d_key, 1, p + 1);
    fp12* res;
    CKR(miller_product(ctx, q, p, 2, &res));
    int ok = 0;
    CKR(finish(ctx, res, &ok, gt576));
    int32_t sig_ok = 0;
    g1_pp key;
    CKR(d2h(ctx, &sig_ok, d_sig_ok, 4));
    CKR(d2h(ctx, &key, p + 1, sizeof(g1_pp)));
    CKR(sync(ctx));
    if (!sig_ok) ok = 0;
    if (reject_inf_key && key.inf) ok = 0;
    if (accept) *accept = ok;
    return B3_OK;
}
static int parse_sig(b3_ctx* ctx, const uint8_t* sig192) {
    CKR(h2d(ctx, ctx->in_a, sig192, 192));
    CKR(ensure(ctx, ctx->g2a_sig, sizeof(g2_aff)));
    CKR(ensure(ctx, ctx->status, 4 * 4));
    CKR(ensure(ctx, ctx->ok, 4 * 4));
    LAUNCH(k_g2_parse, 1, B3_TPB, (const uint8_t*)ctx->in_a.p, 1, (g2_aff*)ctx->g2a_sig.p, (int32_t*)ctx->status.p, 1);
    LAUNCH(k_g2_subgroup<lanes_pair>, 1, B3_TPB, (const g2_aff*)ctx->g2a_sig.p, (const int32_t*)ctx->status.p, 1, (int32_t*)ctx->ok.p);
    return first_status(ctx, (const int32_t*)ctx->status.p, 1);
}
extern "C" int b3_fast_aggregate_verify(b3_ctx* ctx, const uint8_t sig192[192], const uint8_t* pks96, size_t n_pks, const uint8_t* msg,
                                        size_t msg_len, int* accept, uint8_t* gt576) {
    CKR(begin(ctx));
    if (accept) *accept = 0;
    if (!sig192 || (!msg && msg_len)) return B3_ERR_ARG;
    if (n_pks == 0) return B3_OK;                       // M/src/aggregates.rs:179-181
    CK(cudaEventRecord(ctx->ev[0], ctx->stream));
    mark_reset(ctx);
    CKR(parse_sig(ctx, sig192));
    uint32_t off[2] = {0, (uint32_t)n_pks};
    CKR(h2d(ctx, ctx->in_b, pks96, 96 * n_pks));
    CKR(h2d(ctx, ctx->in_e, off, 8));
    CKR(ensure(ctx, ctx->g1j, sizeof(g1_jac) * 2));
    int32_t* d_st = (int32_t*)ctx->status.p + 1;
    CKR(launch_g1_aggregate(ctx, ctx->stream, (const uint8_t*)ctx->in_b.p, (const uint32_t*)ctx->in_e.p, 1, n_pks, (g1_jac*)ctx->g1j.p, d_st));
    CKR(first_status(ctx, d_st, 1));
    return verify_two_pairs(ctx, (const g2_aff*)ctx->g2a_sig.p, (const int32_t*)ctx->ok.p, (const g1_jac*)ctx->g1j.p, 1, msg, msg_len, accept, gt576);
}
static int verify_single_key(b3_ctx* ctx, const uint8_t* sig192, const uint8_t* pk96, int reject_inf, const uint8_t* msg, size_t msg_len,
                             int* accept, uint8_t* gt576) {
    CKR(begin(ctx));
    if (accept) *accept = 0;
    if (!sig192 || !pk96 || (!msg && msg_len)) return B3_ERR_ARG;
    CK(cudaEventRecord(ctx->ev[0], ctx->stream));
    mark_reset(ctx);
    CKR(parse_sig(ctx, sig192));
    CKR(h2d(ctx, ctx->in_b, pk96, 96));
    CKR(ensure(ctx, ctx->g1j, sizeof(g1_jac) * 2));
    int32_t* d_st = (int32_t*)ctx->status.p + 1;
    LAUNCH(k_g1_parse, 1, B3_TPB, (const uint8_t*)ctx->in_b.p, 1, (g1_jac*)ctx->g1j.p, d_st, 1);
    CKR(first_status(ctx, d_st, 1));
    return verify_two_pairs(ctx, (const g2_aff*)ctx->g2a_sig.p, (const int32_t*)ctx->ok.p, (const g1_jac*)ctx->g1j.p, reject_inf, msg, msg_len, accept, gt576);
}
extern "C" int b3_verify(b3_ctx* ctx, const uint8_t sig192[192], const uint8_t pk96[96], const uint8_t* msg, size_t msg_len, int* accept,
                         uint8_t* gt576) {
    return verify_single_key(ctx, sig192, pk96, 0, msg, msg_len, accept, gt576);
}
extern "C" int b3_fast_aggregate_verify_pre_aggregated(b3_ctx* ctx, const uint8_t sig192[192], const uint8_t apk96[96], const uint8_t* msg,
                                                       size_t msg_len, int* accept, uint8_t* gt576) {
    return verify_single_key(ctx, sig192, apk96, 1, msg, msg_len, accept, gt576);
}

extern "C" int b3_aggregate_verify(b3_ctx* ctx, const uint8_t sig192[192], const uint8_t* pks96, const uint8_t* msgs, const uint32_t* msg_off,
                                   size_t n, int* accept, uint8_t* gt576) {
    CKR(begin(ctx));
    if (accept) *accept = 0;
    if (n == 0) return B3_OK;                            // M/src/aggregates.rs:132-134
    if (!sig192 || !pks96 || !msg_off) return B3_ERR_ARG;
    CK(cudaEventRecord(ctx->ev[0], ctx->stream));
    mark_reset(ctx);
    CKR(parse_sig(ctx, sig192));
    CKR(h2d(ctx, ctx->in_b, pks96, 96 * n));
    CKR(h2d(ctx, ctx->in_c, msgs, msg_off[n]));
    CKR(h2d(ctx, ctx->in_d, msg_off, 4 * (n + 1)));
    CKR(ensure(ctx, ctx->g1j, sizeof(g1_jac) * n));
    CKR(ensure(ctx, ctx->g1pp, sizeof(g1_pp) * (n + 1)));
    CKR(ensure(ctx, ctx->g2q, sizeof(g2_jac) * (n + 1)));
    CKR(ensure(ctx, ctx->status, 4 * (n + 4)));
    int32_t* d_st = (int32_t*)ctx->status.p + 4;
    LAUNCH(k_g1_parse, nblk(n), B3_TPB, (const uint8_t*)ctx->in_b.p, n, (g1_jac*)ctx->g1j.p, d_st, 1);
    CKR(first_status(ctx, d_st, n));
    g2_jac* q = (g2_jac*)ctx->g2q.p;
    g1_pp* p = (g1_pp*)ctx->g1pp.p;
    LAUNCH(k_g1_jac_to_pp, nblk(n), B3_TPB, (const g1_jac*)ctx->g1j.p, n, p);
    CKR(hash_to_g2_jac_dev(ctx, ctx->stream, (const uint8_t*)ctx->in_c.p, (const uint32_t*)ctx->in_d.p, n, q));
    LAUNCH(k_g2_aff_to_jac, 1, B3_TPB, (const g2_aff*)ctx->g2a_sig.p, 1, q + n);
    LAUNCH(k_set_neg_g1_pp, 1, 1, p + n);
    fp12* res;
    CKR(miller_product(ctx, q, p, n + 1, &res));
    int ok = 0;
    CKR(finish(ctx, res, &ok, gt576));
    int32_t sig_ok = 0;
    CKR(d2h(ctx, &sig_ok, ctx->ok.p, 4));
    CKR(sync(ctx));
    if (accept) *accept = (ok && sig_ok) ? 1 : 0;
    return B3_OK;
}

// ---- batched per-item verification (SURVEY.md 8(f)3): n independent items, one accept bit each ------------------------
#define B3_ITEMS_PAIR_MIN 2048
// Finishing kernel of n items on the context stream (k_items_finish*: pair 0 of item i = pair first0 + i of the np0-pair
// table lines0, pair 1 = pair first1 + i of lines1, or pair idx1[i] when idx1 is not null).  CTA per item: ~1.5 ms per wave
// of 2 x 148 items; lane pair per item: one item's latency (~12 ms) for any batch that fits the machine (17 ms at 16384 items,
// 33 ms at 32768) -- the crossover is near 2.3 k items
static void items_finish(b3_ctx* ctx, const fp2* lines0, const uint32_t* qinf0, size_t np0, size_t first0, const fp2* lines1, const uint32_t* qinf1,
                         size_t np1, size_t first1, const uint32_t* idx1, const g1_pp* keys, size_t n, const int32_t* st_sig, const int32_t* st_key, int key_rule,
                         int32_t* accept, int32_t* status, uint8_t* gt) {
    const bool per_pair = ctx->item_kernel == 3 || (ctx->item_kernel == 0 && n >= B3_ITEMS_PAIR_MIN);
    if (per_pair)
        LAUNCH(k_items_finish_p, (unsigned)((2 * n + B3_ITEMS_PAIR_TPB - 1) / B3_ITEMS_PAIR_TPB), B3_ITEMS_PAIR_TPB, lines0, qinf0, np0, first0,
               lines1, qinf1, np1, first1, idx1, keys, n, st_sig, st_key, (const int32_t*)ctx->ok.p, key_rule, accept, status, gt);
    else
        LAUNCH(k_items_finish, (unsigned)n, B3_COOP_THREADS, lines0, qinf0, np0, first0, lines1, qinf1, np1, first1, idx1, keys, st_sig, st_key,
               (const int32_t*)ctx->ok.p, key_rule, accept, status, gt);
}
static int verify_batch_core(b3_ctx* ctx, int mode, const uint8_t* d_sigs, const uint8_t* d_pks, const uint32_t* d_pk_off, size_t total_keys,
                             const uint8_t* d_msgs, const uint32_t* d_msg_off, size_t n, int32_t* d_accept, int32_t* d_status, uint8_t* d_gt) {
    CKR(ensure(ctx, ctx->g2a_sig, sizeof(g2_aff) * n));
    CKR(ensure(ctx, ctx->status, 4 * (2 * n + 8)));
    CKR(ensure(ctx, ctx->ok, 4 * (n + 8)));
    CKR(ensure(ctx, ctx->g1j, sizeof(g1_jac) * n));
    CKR(ensure(ctx, ctx->g1pp, sizeof(g1_pp) * n));
    CKR(ensure(ctx, ctx->g2q, sizeof(g2_jac) * 2 * n));
    CKR(miller_reserve(ctx, 2 * n, ctx->lines, ctx->qinf));
    int32_t* d_st_sig = (int32_t*)ctx->status.p;
    int32_t* d_st_key = d_st_sig + n + 4;
    g2_jac* q = (g2_jac*)ctx->g2q.p;              // q[0 .. n) = signatures, q[n .. 2n) = H(msg)
    g1_pp* keys = (g1_pp*)ctx->g1pp.p;
    cudaStream_t sm = ctx->stream;
    cudaStream_t s0 = ctx->serial ? sm : ctx->aux[0], s1 = ctx->serial ? sm : ctx->aux[1], s2 = ctx->serial ? sm : ctx->aux[2];
    int sp;
    if (!ctx->serial) {
        CK(cudaEventRecord(ctx->ev_fork, sm));
        CK(cudaStreamWaitEvent(s1, ctx->ev_fork, 0));
        CK(cudaStreamWaitEvent(s2, ctx->ev_fork, 0));
    }
    // H_i = hash_to_curve_g2(msg_i) and its point chain: the longest dependent chain, issued first
    sp = span_begin(ctx, ST_HASH_TO_G2, s2);
    CKR(hash_to_g2_jac_dev(ctx, s2, d_msgs, d_msg_off, n, q + n));
    span_end(ctx, sp, s2);
    CKR(miller_lines(ctx, s2, q, 2 * n, n, n, ctx->lines, ctx->qinf));
    // signatures: parse + on-curve, then the subgroup checks (aux0) beside their point chains (main)
    sp = span_begin(ctx, ST_COPY, sm);
    LAUNCH_ON(sm, k_g2_parse, nblk(n), B3_TPB, d_sigs, n, (g2_aff*)ctx->g2a_sig.p, d_st_sig, 1);
    LAUNCH_ON(sm, k_g2_aff_to_jac, nblk(n), B3_TPB, (const g2_aff*)ctx->g2a_sig.p, n, q);
    span_end(ctx, sp, sm);
    if (!ctx->serial) {
        CK(cudaEventRecord(ctx->ev_fork2, sm));
        CK(cudaStreamWaitEvent(s0, ctx->ev_fork2, 0));
    }
    sp = span_begin(ctx, ST_SIG_CHECK, s0);
    LAUNCH_ON(s0, k_g2_subgroup<lanes_pair>, nblk(2 * n), B3_TPB, (const g2_aff*)ctx->g2a_sig.p, (const int32_t*)d_st_sig, n, (int32_t*)ctx->ok.p);
    span_end(ctx, sp, s0);
    CKR(miller_lines(ctx, sm, q, 2 * n, 0, n, ctx->lines, ctx->qinf));
    // keys: aggregate (fast_aggregate_verify) or parse (verify / pre-aggregated) -> pairing form
    sp = span_begin(ctx, ST_AGGREGATE, s1);
    if (mode == B3_ITEM_FAST_AGGREGATE) {
        CKR(launch_g1_aggregate(ctx, s1, d_pks, d_pk_off, n, total_keys, (g1_jac*)ctx->g1j.p, d_st_key));
    } else {
        LAUNCH_ON(s1, k_g1_parse, nblk(n), B3_TPB, d_pks, n, (g1_jac*)ctx->g1j.p, d_st_key, 1);
    }
    LAUNCH_ON(s1, k_g1_jac_to_pp, nblk(n), B3_TPB, (const g1_jac*)ctx->g1j.p, n, keys);
    span_end(ctx, sp, s1);
    if (!ctx->serial) {
        cudaStream_t auxs[3] = {s0, s1, s2};
        for (int k = 0; k < 3; k++) {
            CK(cudaEventRecord(ctx->ev_join[k], auxs[k]));
            CK(cudaStreamWaitEvent(sm, ctx->ev_join[k], 0));
        }
    }
    CK(cudaEventRecord(ctx->ev[2], sm));
    sp = span_begin(ctx, ST_FINAL_EXP, sm);
    const fp2* lines = (const fp2*)ctx->lines.p;
    const uint32_t* qinf = (const uint32_t*)ctx->qinf.p;
    items_finish(ctx, lines, qinf, 2 * n, 0, lines, qinf, 2 * n, n, nullptr, keys, n, d_st_sig, d_st_key, mode == B3_ITEM_VERIFY ? B3_KEY_INF_PAIR : B3_KEY_INF_REJECT,
                 d_accept, d_status, d_gt);
    span_end(ctx, sp, sm);
    CK(cudaEventRecord(ctx->ev[3], sm));
    return B3_OK;
}
static int verify_batch_done(b3_ctx* ctx) {
    CK(cudaEventRecord(ctx->ev[1], ctx->stream));
    CKR(sync(ctx));
    mark_collect(ctx);
    cudaEventElapsedTime(&ctx->last_ms[0], ctx->ev[0], ctx->ev[1]);
    if (cudaEventElapsedTime(&ctx->last_ms[1], ctx->ev[2], ctx->ev[3]) != cudaSuccess) ctx->last_ms[1] = 0.f;
    cudaGetLastError();
    return B3_OK;
}
extern "C" int b3_verify_batch_dev(b3_ctx* ctx, int mode, const uint8_t* sigs192_dev, const uint8_t* pks96_dev, const uint32_t* pk_off_dev,
                                   const uint8_t* msgs_dev, const uint32_t* msg_off_dev, size_t n, int32_t* accept_dev, int32_t* status_dev,
                                   uint8_t* gt576_dev) {
    CKR(begin(ctx));
    if (n == 0) return B3_OK;
    if (mode < B3_ITEM_VERIFY || mode > B3_ITEM_PRE_AGGREGATED || n > 0x3fffffffu) return B3_ERR_ARG;
    if (!sigs192_dev || !pks96_dev || !msg_off_dev || !accept_dev || !status_dev || (mode == B3_ITEM_FAST_AGGREGATE && !pk_off_dev)) return B3_ERR_ARG;
    CKR(dev_aligned(ctx, sigs192_dev));
    CKR(dev_aligned(ctx, pks96_dev));
    CKR(dev_aligned(ctx, gt576_dev));
    CK(cudaEventRecord(ctx->ev[0], ctx->stream));
    mark_reset(ctx);
    size_t total_keys = n;
    if (mode == B3_ITEM_FAST_AGGREGATE) {
        uint32_t t = 0;
        CK(cudaMemcpyAsync(&t, pk_off_dev + n, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CKR(sync(ctx));
        total_keys = t;
    }
    CKR(verify_batch_core(ctx, mode, sigs192_dev, pks96_dev, pk_off_dev, total_keys, msgs_dev, msg_off_dev, n, accept_dev, status_dev, gt576_dev));
    return verify_batch_done(ctx);
}
extern "C" int b3_verify_batch(b3_ctx* ctx, int mode, const uint8_t* sigs192, const uint8_t* pks96, const uint32_t* pk_off, const uint8_t* msgs,
                               const uint32_t* msg_off, size_t n, int32_t* accept, int32_t* status, uint8_t* gt576) {
    CKR(begin(ctx));
    if (n == 0) return B3_OK;
    if (mode < B3_ITEM_VERIFY || mode > B3_ITEM_PRE_AGGREGATED || n > 0x3fffffffu) return B3_ERR_ARG;
    if (!sigs192 || !pks96 || !msg_off || !accept || !status || (mode == B3_ITEM_FAST_AGGREGATE && !pk_off)) return B3_ERR_ARG;
    CK(cudaEventRecord(ctx->ev[0], ctx->stream));
    mark_reset(ctx);
    const size_t total_keys = mode == B3_ITEM_FAST_AGGREGATE ? pk_off[n] : n;
    CKR(h2d(ctx, ctx->in_a, sigs192, 192 * n));
    CKR(h2d(ctx, ctx->in_b, pks96, 96 * total_keys));
    if (mode == B3_ITEM_FAST_AGGREGATE) CKR(h2d(ctx, ctx->in_e, pk_off, 4 * (n + 1)));
    CKR(h2d(ctx, ctx->in_c, msgs, msg_off[n]));
    CKR(h2d(ctx, ctx->in_d, msg_off, 4 * (n + 1)));
    CKR(ensure(ctx, ctx->outb, (gt576 ? 576 * n : 0) + 8 * n + 16));
    uint8_t* d_gt = gt576 ? (uint8_t*)ctx->outb.p : nullptr;        // first: the GT records are written with STG.128
    int32_t* d_accept = (int32_t*)((uint8_t*)ctx->outb.p + (gt576 ? 576 * n : 0));
    int32_t* d_status = d_accept + n;
    CKR(verify_batch_core(ctx, mode, (const uint8_t*)ctx->in_a.p, (const uint8_t*)ctx->in_b.p, (const uint32_t*)ctx->in_e.p, total_keys,
                          (const uint8_t*)ctx->in_c.p, (const uint32_t*)ctx->in_d.p, n, d_accept, d_status, d_gt));
    CKR(d2h(ctx, accept, d_accept, 4 * n));
    CKR(d2h(ctx, status, d_status, 4 * n));
    if (gt576) CKR(d2h(ctx, gt576, d_gt, 576 * n));
    return verify_batch_done(ctx);
}

// ---------------------------------------------------------------------------------------------- key table
// Device-resident table of decoded public keys (SURVEY.md 8(f)1): PublicKey::from_bytes -- decompression + key_validate,
// M/src/keys.rs:140-147 -- is paid once per validator; verification calls then name keys by u32 index (4 B instead of 96 B
// per key over PCIe, and no parsing / Montgomery conversion / curve check per use).  A table belongs to one device and is
// read-only during verification, so any number of contexts of that device may use it concurrently.
struct b3_keytable {
    int device = 0;
    size_t n = 0, cap = 0;
    key_entry* d = nullptr;
};
extern "C" int b3_keytable_create(b3_ctx* ctx, size_t capacity, b3_keytable** out) {
    CKR(begin(ctx));
    if (!out) return B3_ERR_ARG;
    *out = nullptr;
    b3_keytable* t = new b3_keytable();
    t->device = ctx->device;
    t->cap = capacity ? capacity : 1;
    if (cudaMalloc((void**)&t->d, sizeof(key_entry) * t->cap) != cudaSuccess) {
        ctx->err = "cudaMalloc(key table)";
        cudaGetLastError();
        delete t;
        return B3_ERR_CUDA;
    }
    *out = t;
    return B3_OK;
}
extern "C" void b3_keytable_destroy(b3_keytable* t) {
    if (!t) return;
    cudaSetDevice(t->device);
    if (t->d) cudaFree(t->d);
    delete t;
}
extern "C" size_t b3_keytable_size(const b3_keytable* t) { return t ? t->n : 0; }
// Appends n keys (compressed != 0: 48-byte ZCash-compressed = PublicKey::from_bytes / from_bytes_unchecked; else 96-byte
// uncompressed = from_uncompressed_bytes; validate != 0 adds key_validate).  status[i] (nullable) = B3_OK or the AmclError
// code; a rejected key still occupies its slot (marked invalid: any set that names it fails with that error), so that
// indices stay aligned with the caller's validator numbering.  *first_index (nullable) = index of keys[0] in the table.
extern "C" int b3_keytable_append(b3_ctx* ctx, b3_keytable* t, const uint8_t* keys, size_t n, int compressed, int validate, int32_t* status,
                                  size_t* first_index) {
    CKR(begin(ctx));
    if (!t || t->device != ctx->device || (n && !keys)) return B3_ERR_ARG;
    if (first_index) *first_index = t->n;
    if (n == 0) return B3_OK;
    if (t->n + n > t->cap) {                            // grow (geometric): old entries are copied device to device
        size_t cap = t->cap * 2 > t->n + n ? t->cap * 2 : t->n + n;
        key_entry* d = nullptr;
        CK(cudaMalloc((void**)&d, sizeof(key_entry) * cap));
        CK(cudaMemcpyAsync(d, t->d, sizeof(key_entry) * t->n, cudaMemcpyDeviceToDevice, ctx->stream));
        CKR(sync(ctx));
        cudaFree(t->d);
        t->d = d;
        t->cap = cap;
    }
    CKR(h2d(ctx, ctx->in_a, keys, (compressed ? 48 : 96) * n));
    CKR(ensure(ctx, ctx->status, 4 * n));
    LAUNCH(k_keytable_build, nblk(n), B3_TPB, (const uint8_t*)ctx->in_a.p, n, compressed, validate, t->d + t->n, (int32_t*)ctx->status.p);
    if (status) CKR(d2h(ctx, status, ctx->status.p, 4 * n));
    CKR(sync(ctx));
    t->n += n;
    return B3_OK;
}
// table entries idx[0..n) back in the 96-byte wire format (what PublicKey::as_uncompressed_bytes returns, M/src/keys.rs:163-165)
extern "C" int b3_keytable_get(b3_ctx* ctx, const b3_keytable* t, const uint32_t* idx, size_t n, uint8_t* out96, int32_t* status) {
    CKR(begin(ctx));
    if (!t || t->device != ctx->device) return B3_ERR_ARG;
    if (n == 0) return B3_OK;
    if (!idx || !out96 || !status) return B3_ERR_ARG;
    CKR(h2d(ctx, ctx->in_a, idx, 4 * n));
    CKR(ensure(ctx, ctx->outb, 96 * n));
    CKR(ensure(ctx, ctx->status, 4 * n));
    LAUNCH(k_keytable_get, nblk(n), B3_TPB, (const key_entry*)t->d, t->n, (const uint32_t*)ctx->in_a.p, n, (uint8_t*)ctx->outb.p, (int32_t*)ctx->status.p);
    CKR(d2h(ctx, out96, ctx->outb.p, 96 * n));
    CKR(d2h(ctx, status, ctx->status.p, 4 * n));
    return sync(ctx);
}
static int launch_g1_aggregate_idx(b3_ctx* ctx, cudaStream_t strm, const b3_keytable* t, const uint32_t* d_idx, const uint32_t* d_off, size_t n_sets,
                                   size_t total_keys, g1_jac* d_out, int32_t* d_status) {
    if (n_sets == 0) return B3_OK;
    launch_agg(ctx, strm, n_sets, total_keys, kAggG4Min, [](auto g) { return k_g1_aggregate_idx<decltype(g)::value>; }, (const key_entry*)t->d,
               t->n, d_idx, d_off, n_sets, d_out, d_status);
    return B3_OK;
}
// AggregatePublicKey::into_aggregate over table indices (M/src/aggregates.rs:46-56)
extern "C" int b3_g1_aggregate_indexed(b3_ctx* ctx, const b3_keytable* t, const uint32_t* key_idx, const uint32_t* off, size_t n_sets, uint8_t* out96,
                                       int32_t* status) {
    CKR(begin(ctx));
    if (!t || t->device != ctx->device) return B3_ERR_ARG;
    if (n_sets == 0) return B3_OK;
    if (!off || !out96 || !status || (off[n_sets] && !key_idx)) return B3_ERR_ARG;
    const size_t total = off[n_sets];
    CKR(h2d(ctx, ctx->in_a, key_idx, 4 * total));
    CKR(h2d(ctx, ctx->in_b, off, 4 * (n_sets + 1)));
    CKR(ensure(ctx, ctx->outb, 96 * n_sets));
    CKR(ensure(ctx, ctx->status, 4 * n_sets));
    CKR(ensure(ctx, ctx->g1j, sizeof(g1_jac) * n_sets));
    CKR(ensure(ctx, ctx->g1a, sizeof(g1_aff) * n_sets));
    CKR(launch_g1_aggregate_idx(ctx, ctx->stream, t, (const uint32_t*)ctx->in_a.p, (const uint32_t*)ctx->in_b.p, n_sets, total, (g1_jac*)ctx->g1j.p,
                                (int32_t*)ctx->status.p));
    LAUNCH(k_g1_to_affine, nblk((n_sets + norm_per(n_sets) - 1) / norm_per(n_sets)), B3_TPB, (const g1_jac*)ctx->g1j.p, n_sets, (g1_aff*)ctx->g1a.p, norm_per(n_sets));
    LAUNCH(k_g1_aff_to_wire, nblk(n_sets), B3_TPB, (const g1_aff*)ctx->g1a.p, n_sets, (uint8_t*)ctx->outb.p);
    CKR(d2h(ctx, out96, ctx->outb.p, 96 * n_sets));
    CKR(d2h(ctx, status, ctx->status.p, 4 * n_sets));
    return sync(ctx);
}

// ---------------------------------------------------------------------------------------------- verify_multiple
// Inputs of one verify_multiple call; everything device-resident unless named h_.
struct vm_in {
    const uint8_t* d_sigs = nullptr;        // n x 192 B wire format (unused when `prechecked`)
    const uint8_t* d_pks = nullptr;         // keys as 96-byte records ...
    const uint8_t* h_pks = nullptr;         // ... copied from here on the aggregation stream (host-pointer entries)
    const b3_keytable* tbl = nullptr;       // or: key table + indices
    const uint32_t* d_idx = nullptr;
    const uint32_t* h_idx = nullptr;
    const uint32_t* d_pk_off = nullptr;     // null: one key (or index) per set
    size_t total_keys = 0;
    const uint8_t* d_msgs = nullptr;
    const uint32_t* d_msg_off = nullptr;
    size_t n_hash = 0;                      // messages hashed: n, or the n_msgs of a grouped call
    const uint32_t* d_msg_idx = nullptr;    // grouped call: message of set j (n_hash messages); null: message j
    const uint64_t* d_scalars = nullptr;
    size_t n = 0;
    long long index_base = 0;
    bool prechecked = false;                // parsed signatures and ok[] are already in the context (b3_sig_precheck)
    bool defer_sig = false;                 // run the subgroup checks beside the serial tail of the call instead of at its start (whole calls)
};
#define B3_FB_NONE 0x7fffffffffffffffLL
// pairs of the batch product over n sets: the n_hash messages' H_k (k < n_hash), then the signature sum S, or its 8 window
// sums from B3_MSM_MIN_SETS sets up
static size_t vm_pairs(size_t n, size_t n_hash) { return n == 0 ? 0 : n_hash + (n >= B3_MSM_MIN_SETS ? B3_MSM_WINDOWS : 1); }
// one table entry per set (pre-aggregated keys held in the table)
__global__ void __launch_bounds__(B3_TPB) k_g1_from_table(const key_entry* __restrict__ table, size_t n_table, const uint32_t* __restrict__ idx, size_t n,
                                                          g1_jac* out, int32_t* status) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t k = idx[i];
    g1_aff a;
    int e = B3_ERR_INVALID_POINT;
    if (k < n_table) {
        key_entry ent;
        key_entry_load(ent, table + k);
        e = key_entry_point(a, ent);
    }
    g1_jac j;
    if (e) pt_set_inf(j); else pt_from_aff(j, a);
    out[i] = j;
    status[i] = e;
}
// The forked region: the stages below are independent of each other; unless ctx->serial they run concurrently:
//   main : parse signatures (... and, after the join, the end of the call: accumulation, closing chain)
//   aux0 : subgroup checks of the parsed signatures               aux1 : aggregate keys -> P_j = [c_j] apk_j
//   aux2 : H_k = hash_to_curve_g2(msg_k) -> their point chains    aux3 : S = sum_j [c_j] sig_j -> its point chains
// (a grouped call hashes each of its n_hash messages once, and aux1 sums the P_j of the sets naming message k into pair k)
// No allocation happens in here (every buffer is sized by the caller before the fork).
static int vm_sig_checks(b3_ctx* ctx, const vm_in& in, const int32_t* d_st_sig, long long* d_first_bad);
static int vm_stages(b3_ctx* ctx, const vm_in& in, size_t n_total, int32_t* d_st_sig, int32_t* d_st_key, long long* d_first_bad, int32_t* d_zero,
                     int32_t* d_range) {
    const size_t n = in.n, nh = in.n_hash;
    g2_jac* q = (g2_jac*)ctx->g2q.p;
    g1_pp* p = (g1_pp*)ctx->g1pp.p;
    cudaStream_t sm = ctx->stream;
    cudaStream_t s0 = ctx->serial ? sm : ctx->aux[0], s1 = ctx->serial ? sm : ctx->aux[1], s2 = ctx->serial ? sm : ctx->aux[2];
    cudaStream_t s3 = ctx->serial ? sm : ctx->aux[3];
    int sp;
    if (!ctx->serial) {
        CK(cudaEventRecord(ctx->ev_fork, sm));
        CK(cudaStreamWaitEvent(s1, ctx->ev_fork, 0));
        CK(cudaStreamWaitEvent(s2, ctx->ev_fork, 0));
    }
    // 4. H_j = hash_to_curve_g2(msg_j) (M/src/aggregates.rs:290) and its Miller point chain: the longest dependent chain of
    //    the batch, so it is issued FIRST (blocks are dispatched in launch order) on the high-priority stream
    sp = span_begin(ctx, ST_HASH_TO_G2, s2);
    CKR(hash_to_g2_jac_dev(ctx, s2, in.d_msgs, in.d_msg_off, nh, q));
    span_end(ctx, sp, s2);
    CKR(miller_lines(ctx, s2, q, n_total, 0, nh, ctx->lines, ctx->qinf));   // the point chains need only H_k
    // 1. signatures: parse + on-curve (main), subgroup check (M/src/aggregates.rs:274-276) on aux0 -- unless b3_sig_precheck
    //    already left the parsed signatures and their ok[] in the context
    if (!in.prechecked) {
        sp = span_begin(ctx, ST_COPY, sm);
        LAUNCH_ON(sm, k_g2_parse, nblk(n), B3_TPB, in.d_sigs, n, (g2_aff*)ctx->g2a_sig.p, d_st_sig, 1);
        span_end(ctx, sp, sm);
    }
    if (!ctx->serial) {
        CK(cudaEventRecord(ctx->ev_fork2, sm));
        CK(cudaStreamWaitEvent(s3, ctx->ev_fork2, 0));
    }
    // subgroup checks: a WHOLE call (in.defer_sig) runs them beside its closing chain and final exponentiation, when the GPU is
    // otherwise idle (vm_enqueue) -- nothing before the accept bit needs their result; a PARTIAL call needs first_bad in its
    // partial record right after the closing chain, so its checks start here, with the call
    if (!in.defer_sig) CKR(vm_sig_checks(ctx, in, d_st_sig, d_first_bad));
    // 2. aggregate public keys; 3. P_j = [c_j] apk_j (M/src/aggregates.rs:293)
    // grouped: the sets sorted by message first (it needs only msg_idx, so it runs while the keys are copied)
    const uint32_t m = (uint32_t)nh;
    uint32_t *perm = nullptr, *pos = nullptr, *lo = nullptr, *hi = nullptr;
    if (in.d_msg_idx) {
        uint32_t* w = (uint32_t*)ctx->grp.p;               // [perm0 | perm1 | pos] n each, then [lo | hi] m each
        pos = w + 2 * n;
        lo = w + 3 * n;
        hi = lo + m;
        int passes = 1;                                    // 8-bit digits of the largest index
        while (passes < 4 && ((m - 1) >> (8 * passes)) != 0) passes++;
        sp = span_begin(ctx, ST_G1_MUL, s1);
        for (int t = 0; t < passes; t++) {
            uint32_t* out = w + (size_t)(t & 1) * n;
            LAUNCH_ON(s1, k_grp_sort, 1, 1024, in.d_msg_idx, n, m, 8u * t, t ? (const uint32_t*)perm : nullptr, out, t == passes - 1 ? pos : nullptr,
                      t == 0 ? d_range : nullptr);
            perm = out;
        }
        CK(cudaMemsetAsync(lo, 0, 8 * (size_t)m, s1));
        LAUNCH_ON(s1, k_grp_bounds, nblk(n), B3_TPB, in.d_msg_idx, perm, n, m, lo, hi);
        span_end(ctx, sp, s1);
    }
    // host-pointer entries: the keys (96 % of the input bytes) or their indices are copied on THIS stream, so the transfer
    // overlaps hash_to_G2 and the signature work instead of preceding them
    if (in.h_pks) CK(cudaMemcpyAsync((void*)in.d_pks, in.h_pks, 96 * in.total_keys, cudaMemcpyHostToDevice, s1));
    if (in.h_idx) CK(cudaMemcpyAsync((void*)in.d_idx, in.h_idx, 4 * in.total_keys, cudaMemcpyHostToDevice, s1));
    sp = span_begin(ctx, ST_AGGREGATE, s1);
    if (in.tbl) {
        if (in.d_pk_off) CKR(launch_g1_aggregate_idx(ctx, s1, in.tbl, in.d_idx, in.d_pk_off, n, in.total_keys, (g1_jac*)ctx->g1j.p, d_st_key));
        else LAUNCH_ON(s1, k_g1_from_table, nblk(n), B3_TPB, (const key_entry*)in.tbl->d, in.tbl->n, in.d_idx, n, (g1_jac*)ctx->g1j.p, d_st_key);
    } else if (in.d_pk_off) {
        CKR(launch_g1_aggregate(ctx, s1, in.d_pks, in.d_pk_off, n, in.total_keys, (g1_jac*)ctx->g1j.p, d_st_key));
    } else {
        LAUNCH_ON(s1, k_g1_parse, nblk(n), B3_TPB, in.d_pks, n, (g1_jac*)ctx->g1j.p, d_st_key, 1);
    }
    span_end(ctx, sp, s1);
    sp = span_begin(ctx, ST_G1_MUL, s1);
    if (in.d_msg_idx) {                   // [c_j] apk_j at the set's sorted position, a segmented tree per message, H_k's G1 member
        g1_jac* a = (g1_jac*)ctx->g1j2.p;
        launch_lanes<lanes_thread, lanes_pair>(ctx, s1, ctx->wide_now, n, [](auto L) { return k_g1_mul_u64<decltype(L), g1_out_at>; },
                                               (const g1_jac*)ctx->g1j.p, in.d_scalars, n, g1_out_at{a, pos}, d_zero);
        for (size_t step = 1; step < n; step <<= 1)
            LAUNCH_ON(s1, k_grp_sum_level, nblk(n), B3_TPB, a, in.d_msg_idx, perm, lo, hi, n, m, step);
        LAUNCH_ON(s1, k_grp_to_pp, nblk(m), B3_TPB, (const g1_jac*)a, lo, hi, m, p);
    } else {
        launch_lanes<lanes_thread, lanes_pair>(ctx, s1, ctx->wide_now, n, [](auto L) { return k_g1_mul_u64<decltype(L), g1_out_pp>; },
                                               (const g1_jac*)ctx->g1j.p, in.d_scalars, n, g1_out_pp{p}, d_zero);
    }
    span_end(ctx, sp, s1);
    // 5. S = sum_j [c_j] sig_j (M/src/aggregates.rs:303), on aux3: the context's own (highest-priority) stream is left to the
    //    end of the call
    sp = span_begin(ctx, ST_G2_MUL_SUM, s3);
    g2_jac* s;
    if (n >= B3_MSM_MIN_SETS) {           // bucket method: 8 window sums, each its own pair against -[2^(8w)] G1
        const unsigned nr = msm_ranges(n);
        uint32_t* idx = (uint32_t*)ctx->msm.p;
        uint32_t* start = idx + B3_MSM_WINDOWS * n;
        LAUNCH_ON(s3, k_msm_sort, B3_MSM_WINDOWS, 1024, in.d_scalars, n, idx, start);
        LAUNCH_ON(s3, k_msm_walk, nblk(2 * (size_t)B3_MSM_WINDOWS * nr), B3_TPB, (const g2_aff*)ctx->g2a_sig.p, idx, start, n, nr, msm_step(n),
                  (g2_jac*)ctx->g2j.p);
        CKR(g2_sum(ctx, (g2_jac*)ctx->g2j.p, (g2_jac*)ctx->g2j2.p, (size_t)B3_MSM_WINDOWS * nr, &s, s3, B3_MSM_WINDOWS));
        LAUNCH_ON(s3, k_msm_pairs, 1, 32, s, q + nh, p + nh);
    } else {
        LAUNCH_ON(s3, k_g2_mul_u64, nblk(2 * n), B3_TPB, (const g2_aff*)ctx->g2a_sig.p, in.d_scalars, n, (g2_jac*)ctx->g2j.p);
        CKR(g2_sum(ctx, (g2_jac*)ctx->g2j.p, (g2_jac*)ctx->g2j2.p, n, &s, s3));
        CK(cudaMemcpyAsync(q + nh, s, sizeof(g2_jac), cudaMemcpyDeviceToDevice, s3));
        LAUNCH_ON(s3, k_set_neg_g1_pp, 1, 1, p + nh);
    }
    span_end(ctx, sp, s3);
    CKR(miller_lines(ctx, s3, q, n_total, nh, n_total - nh, ctx->lines, ctx->qinf));   // ... and the window sums / S
    if (!ctx->serial) {
        cudaStream_t auxs[4] = {s0, s1, s2, s3};
        for (int k = 1; k < 4; k++) {
            CK(cudaEventRecord(ctx->ev_join[k], auxs[k]));
            CK(cudaStreamWaitEvent(sm, ctx->ev_join[k], 0));
        }
        (void)s0;
    }
    return B3_OK;
}
// 1b. subgroup_check_g2 of every signature (M/src/aggregates.rs:274-276) and the index of the first failure.  Nothing before the
//     accept bit needs the result, so the checks are forked off AFTER the accumulation kernel has been launched: they run on
//     aux0 beside the closing chain and the final exponentiation -- single-CTA kernels that leave the GPU idle -- instead of
//     competing with hash_to_G2 at the start of the call.  vm_join_sig() makes the context stream wait for them.
static int vm_sig_checks(b3_ctx* ctx, const vm_in& in, const int32_t* d_st_sig, long long* d_first_bad) {
    const size_t n = in.n;
    cudaStream_t s0 = ctx->serial ? ctx->stream : ctx->aux[0];
    if (!ctx->serial) {
        CK(cudaEventRecord(ctx->ev_fork3, ctx->stream));
        CK(cudaStreamWaitEvent(s0, ctx->ev_fork3, 0));
    }
    // beside the tail the plain kernel is used even in latency mode: at 8192 sets it has 128 CTAs, which leaves SMs free for
    // the single CTA of the closing chain / final exponentiation (the replicated form fills every SM and halves their speed)
    const bool wide = ctx->wide_now && !in.defer_sig;
    int sp = span_begin(ctx, ST_SIG_CHECK, s0);
    if (!in.prechecked)
        launch_lanes<lanes_pair, lanes_quad>(ctx, s0, wide, n, [](auto L) { return k_g2_subgroup<decltype(L)>; }, (const g2_aff*)ctx->g2a_sig.p,
                                             d_st_sig, n, (int32_t*)ctx->ok.p);
    LAUNCH_ON(s0, k_first_bad, nblk(n), B3_TPB, (const int32_t*)ctx->ok.p, n, in.index_base, d_first_bad);
    span_end(ctx, sp, s0);
    if (!ctx->serial) {
        CK(cudaEventRecord(ctx->ev_join[0], s0));
        ctx->sig_pending = true;
    }
    return B3_OK;
}
static int vm_join_sig(b3_ctx* ctx) {
    if (ctx->sig_pending) {
        ctx->sig_pending = false;
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_join[0], 0));
    }
    return B3_OK;
}
// an error inside the forked region leaves aux streams running (possibly still reading the caller's host buffers): drain them
static void vm_drain(b3_ctx* ctx) {
    ctx->sig_pending = false;
    for (int i = 0; i < 4; i++) cudaStreamSynchronize(ctx->aux[i]);
    cudaStreamSynchronize(ctx->stream);
    cudaGetLastError();
}
// Enqueues the whole partial verification (everything up to this rank's Miller product, left in *res) WITHOUT synchronising;
// the input statuses travel to pinned host memory behind it and are read by vm_collect() after the caller's synchronise.
static int vm_enqueue(b3_ctx* ctx, const vm_in& in, fp12** res, long long** d_first_bad_out) {
    const size_t n = in.n;
    if (in.tbl && in.tbl->device != ctx->device) return B3_ERR_ARG;
    if (in.prechecked && ctx->pre_n != n) {
        ctx->err = "b3_sig_precheck of the same signatures must precede a *_checked call on this context";
        return B3_ERR_ARG;
    }
    const size_t nh = in.n_hash;
    const size_t n_total = vm_pairs(n, nh);
    // every buffer of the call is sized HERE, before the fork (ensure() may free / allocate, which synchronises the device)
    const size_t nr = n >= B3_MSM_MIN_SETS ? msm_ranges(n) : 0;     // ranges of the signature MSM per window
    CKR(ensure(ctx, ctx->g2a_sig, sizeof(g2_aff) * (n + 1)));
    CKR(ensure(ctx, ctx->status, 4 * (2 * n + 8)));
    CKR(ensure(ctx, ctx->ok, 4 * (n + 8)));
    CKR(ensure(ctx, ctx->g1j, sizeof(g1_jac) * (n + 1)));
    CKR(ensure(ctx, ctx->g1pp, sizeof(g1_pp) * (nh + B3_MSM_WINDOWS)));
    CKR(ensure(ctx, ctx->g2q, sizeof(g2_jac) * (nh + B3_MSM_WINDOWS)));
    if (in.d_msg_idx) {
        CKR(ensure(ctx, ctx->g1j2, sizeof(g1_jac) * (n + 1)));
        CKR(ensure(ctx, ctx->grp, 4 * (3 * n + 2 * nh)));
    }
    CKR(ensure(ctx, ctx->g2j, sizeof(g2_jac) * std::max(n + 1, B3_MSM_WINDOWS * nr)));
    CKR(ensure(ctx, ctx->g2j2, sizeof(g2_jac) * std::max(n + 2, B3_MSM_WINDOWS * nr / 2)));
    if (nr) CKR(ensure(ctx, ctx->msm, 4 * (B3_MSM_WINDOWS * n + B3_MSM_WINDOWS * 257)));
    CKR(ensure(ctx, ctx->misc, 64));
    CKR(miller_reserve(ctx, n_total, ctx->lines, ctx->qinf));
    CKR(miller_finish_reserve(ctx, n_total));
    if (ctx->pin_cap < 4 * (2 * n + 8) + 16) {
        if (ctx->pin) cudaFreeHost(ctx->pin);
        ctx->pin = nullptr;
        ctx->pin_cap = 0;
        const size_t cap = 4 * (2 * n + 8) + 16 + 4096;
        CK(cudaMallocHost(&ctx->pin, cap));
        ctx->pin_cap = cap;
    }
    int32_t* d_st_sig = (int32_t*)ctx->status.p;
    int32_t* d_st_key = d_st_sig + n + 4;
    long long* d_first_bad = (long long*)ctx->misc.p;
    int32_t* d_zero = (int32_t*)((uint8_t*)ctx->misc.p + 8);
    int32_t* d_range = d_zero + 1;                            // grouped: a message index >= n_hash
    ctx->h_init[0] = B3_FB_NONE;
    ctx->h_init[1] = 0;
    CK(cudaMemcpyAsync(d_first_bad, ctx->h_init, 16, cudaMemcpyHostToDevice, ctx->stream));
    if (n > 0) {
        const int rc = vm_stages(ctx, in, n_total, d_st_sig, d_st_key, d_first_bad, d_zero, d_range);
        if (rc != B3_OK) { vm_drain(ctx); return rc; }
    }
    // 6. Miller loops over the n + 8 (or n + 1) pairs: accumulation, then -- beside the subgroup checks -- the closing chain
    CKR(miller_accumulate(ctx, (const g1_pp*)ctx->g1pp.p, n_total, res));
    if (n > 0 && in.defer_sig) {
        const int rc = vm_sig_checks(ctx, in, d_st_sig, d_first_bad);
        if (rc != B3_OK) { vm_drain(ctx); return rc; }
    }
    CKR(miller_close(ctx, n_total));
    *d_first_bad_out = d_first_bad;
    if (n > 0) CK(cudaMemcpyAsync(ctx->pin, ctx->status.p, 4 * (2 * n + 8), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync((uint8_t*)ctx->pin + 4 * (2 * n + 8), d_zero, 8, cudaMemcpyDeviceToHost, ctx->stream));
    ctx->pre_n = (size_t)-1;                                  // a precheck is consumed by the call that follows it
    return B3_OK;
}
// after the stream synchronise: wire-format errors of the inputs (cannot happen for values that came out of the reference's
// own types), the zero-scalar flag and the message-index flag of a grouped call
static int vm_collect(b3_ctx* ctx, size_t n) {
    const int32_t* h = (const int32_t*)ctx->pin;
    if (h[2 * n + 8]) { ctx->err = "batch scalar 0: the draw rule of M/src/aggregates.rs:280-286 never yields it"; return B3_ERR_ARG; }
    if (h[2 * n + 9]) { ctx->err = "msg_idx: a message index >= n_msgs"; return B3_ERR_ARG; }
    for (size_t i = 0; i < n; i++) {
        if (h[i]) return h[i];
        if (h[n + 4 + i] && h[n + 4 + i] != B3_ERR_AGGREGATE_EMPTY_POINTS) return h[n + 4 + i];
    }
    return B3_OK;
}
static int scalars_nonzero(b3_ctx* ctx, const uint64_t* scalars, size_t n) {
    for (size_t i = 0; i < n; i++)
        if (scalars[i] == 0) { ctx->err = "batch scalar 0: the draw rule of M/src/aggregates.rs:280-286 never yields it"; return B3_ERR_ARG; }
    return B3_OK;
}
// final exponentiation of *res + accept bit, in the same stream synchronise as the partial
static int vm_finish_whole(b3_ctx* ctx, size_t n, fp12* res, long long* d_fb, int* accept, int64_t* first_bad, uint8_t* gt576) {
    CKR(ensure(ctx, ctx->outb, 576 + 16));
    uint8_t* d_gt = (uint8_t*)ctx->outb.p;
    int32_t* d_one = (int32_t*)(d_gt + 576);
    int sp = span_begin(ctx, ST_FINAL_EXP, ctx->stream);
    LAUNCH(k_final_exp, 1, B3_COOP_THREADS, (const fp12*)res, d_gt, d_one);
    span_end(ctx, sp, ctx->stream);
    CKR(vm_join_sig(ctx));
    CK(cudaEventRecord(ctx->ev[1], ctx->stream));
    int32_t one = 0;
    long long fb = 0;
    uint8_t gt[576];
    CKR(d2h(ctx, &one, d_one, 4));
    CKR(d2h(ctx, gt, d_gt, 576));
    CKR(d2h(ctx, &fb, d_fb, 8));
    CKR(sync(ctx));
    cudaEventElapsedTime(&ctx->last_ms[0], ctx->ev[0], ctx->ev[1]);
    if (cudaEventElapsedTime(&ctx->last_ms[1], ctx->ev[2], ctx->ev[3]) != cudaSuccess) ctx->last_ms[1] = 0.f;
    cudaGetLastError();
    mark_collect(ctx);
    CKR(vm_collect(ctx, n));
    if (gt576) memcpy(gt576, gt, 576);
    if (fb == B3_FB_NONE) fb = -1;
    if (first_bad) *first_bad = fb;
    if (accept) *accept = (one && fb < 0) ? 1 : 0;
    return B3_OK;
}

struct partial_rec {
    fp12 f;
    long long first_bad;
    long long pad;
};
static_assert(sizeof(partial_rec) == B3_PARTIAL_BYTES, "partial record layout");

__global__ void k_pack_partial(const fp12* f, const long long* fb, partial_rec* out) {
    out->f = *f;
    out->first_bad = *fb;
    out->pad = 0;
}
// partial i is in[i * stride] (stride > 1: the records of one lane inside a gathered [rank][lane] array)
__global__ void k_unpack_partials(const partial_rec* in, size_t n, size_t stride, fp12* f, long long* fb) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    f[i] = in[i * stride].f;
    atomicMin(fb, in[i * stride].first_bad);
}
// this rank's partial -> partial_dev, one synchronise
static int vm_finish_partial(b3_ctx* ctx, size_t n, fp12* res, long long* d_fb, uint8_t* partial_dev) {
    CKR(vm_join_sig(ctx));
    LAUNCH(k_pack_partial, 1, 1, (const fp12*)res, (const long long*)d_fb, (partial_rec*)partial_dev);
    CK(cudaEventRecord(ctx->ev[1], ctx->stream));
    CKR(sync(ctx));
    mark_collect(ctx);
    cudaEventElapsedTime(&ctx->last_ms[0], ctx->ev[0], ctx->ev[1]);
    if (cudaEventElapsedTime(&ctx->last_ms[1], ctx->ev[2], ctx->ev[3]) != cudaSuccess) ctx->last_ms[1] = 0.f;
    cudaGetLastError();
    return vm_collect(ctx, n);
}
// stages the HOST inputs of a call (signatures, offsets, messages, scalars now; keys / indices later, on the aggregation
// stream) and fills `in`
// (n_msgs messages: n, or the message count of a grouped call)
static int vm_stage_host(b3_ctx* ctx, vm_in& in, const b3_keytable* tbl, const uint8_t* sigs192, const void* keys, const uint32_t* pk_off,
                         const uint8_t* msgs, const uint32_t* msg_off, const uint64_t* scalars, size_t n, long long index_base, size_t n_msgs) {
    if (n && (!keys || !msg_off || !scalars)) return B3_ERR_ARG;
    CKR(scalars_nonzero(ctx, scalars, n));
    in.n = n;
    in.n_hash = n_msgs;
    in.index_base = index_base;
    in.tbl = tbl;
    in.total_keys = pk_off ? pk_off[n] : n;
    in.prechecked = sigs192 == nullptr;
    if (n == 0) return B3_OK;
    if (sigs192) CKR(h2d(ctx, ctx->in_a, sigs192, 192 * n));
    CKR(ensure(ctx, ctx->in_b, (tbl ? 4 : 96) * in.total_keys + 16));   // copied inside the call, on the aggregation stream
    if (pk_off) CKR(h2d(ctx, ctx->in_e, pk_off, 4 * (n + 1)));
    CKR(h2d(ctx, ctx->in_c, msgs, msg_off[n_msgs]));
    CKR(h2d(ctx, ctx->in_d, msg_off, 4 * (n_msgs + 1)));
    CKR(h2d(ctx, ctx->in_f, scalars, 8 * n));
    in.d_sigs = (const uint8_t*)ctx->in_a.p;
    if (tbl) { in.d_idx = (const uint32_t*)ctx->in_b.p; in.h_idx = (const uint32_t*)keys; }
    else { in.d_pks = (const uint8_t*)ctx->in_b.p; in.h_pks = (const uint8_t*)keys; }
    in.d_pk_off = pk_off ? (const uint32_t*)ctx->in_e.p : nullptr;
    in.d_msgs = (const uint8_t*)ctx->in_c.p;
    in.d_msg_off = (const uint32_t*)ctx->in_d.p;
    in.d_scalars = (const uint64_t*)ctx->in_f.p;
    return B3_OK;
}
static int vm_fill_dev(b3_ctx* ctx, vm_in& in, const b3_keytable* tbl, const uint8_t* sigs_dev, const void* keys_dev, const uint32_t* pk_off_dev,
                       const uint8_t* msgs_dev, const uint32_t* msg_off_dev, const uint64_t* scalars_dev, size_t n, long long index_base,
                       size_t n_msgs) {
    if (n && (!sigs_dev || !keys_dev || !msg_off_dev || !scalars_dev)) return B3_ERR_ARG;
    CKR(dev_aligned(ctx, sigs_dev));
    if (!tbl) CKR(dev_aligned(ctx, keys_dev));
    in.n = n;
    in.n_hash = n_msgs;
    in.index_base = index_base;
    in.tbl = tbl;
    in.d_sigs = sigs_dev;
    if (tbl) in.d_idx = (const uint32_t*)keys_dev; else in.d_pks = (const uint8_t*)keys_dev;
    in.d_pk_off = pk_off_dev;
    in.d_msgs = msgs_dev;
    in.d_msg_off = msg_off_dev;
    in.d_scalars = scalars_dev;
    in.total_keys = n;
    if (pk_off_dev && n) {                               // only the lane-count heuristic of the aggregation needs it
        uint32_t t = 0;
        CK(cudaMemcpyAsync(&t, pk_off_dev + n, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CKR(sync(ctx));
        in.total_keys = t;
    }
    return B3_OK;
}
static int vm_begin(b3_ctx* ctx) {
    CKR(begin(ctx));
    CK(cudaEventRecord(ctx->ev[0], ctx->stream));
    mark_reset(ctx);
    return B3_OK;
}
static int vm_whole(b3_ctx* ctx, const vm_in& in0, int* accept, int64_t* first_bad, uint8_t* gt576) {
    call_guard guard(ctx, in0.n);
    vm_in in = in0;
    in.defer_sig = true;                       // the final exponentiation follows in the same call: checks beside the serial tail
    fp12* res;
    long long* d_fb;
    CKR(vm_enqueue(ctx, in, &res, &d_fb));
    int ok = 0;
    CKR(vm_finish_whole(ctx, in.n, res, d_fb, &ok, first_bad, gt576));
    if (accept) *accept = ok;
    ctx->loc_n = in.n;                         // the whole pipeline ran: its retained state serves b3_verify_multiple_locate
    ctx->loc_accept = ok != 0;
    ctx->loc_np = vm_pairs(in.n, in.n_hash);
    ctx->loc_idx = in.d_msg_idx;
    return B3_OK;
}
static int vm_partial(b3_ctx* ctx, const vm_in& in, uint8_t* partial_dev) {
    call_guard guard(ctx, in.n);
    fp12* res;
    long long* d_fb;
    CKR(vm_enqueue(ctx, in, &res, &d_fb));
    return vm_finish_partial(ctx, in.n, res, d_fb, partial_dev);
}

extern "C" int b3_verify_multiple(b3_ctx* ctx, const uint8_t* sigs192, const uint8_t* pks96, const uint32_t* pk_off, const uint8_t* msgs,
                                  const uint32_t* msg_off, const uint64_t* scalars, size_t n, int* accept, int64_t* first_bad, uint8_t* gt576) {
    if (accept) *accept = 0;
    if (first_bad) *first_bad = -1;
    CKR(vm_begin(ctx));
    if (n && !sigs192) return B3_ERR_ARG;
    vm_in in;
    CKR(vm_stage_host(ctx, in, nullptr, sigs192, pks96, pk_off, msgs, msg_off, scalars, n, 0, n));
    return vm_whole(ctx, in, accept, first_bad, gt576);
}
// The two-phase form that keeps the reference's RNG contract without doing anything twice (M/src/aggregates.rs:272-287: the
// scalar of set j is drawn only after the signatures 0..j passed subgroup_check_g2, and nothing is drawn for or after the
// first failing set):  b3_sig_precheck -> first_bad;  the caller draws min(first_bad, n) scalars and, if first_bad < 0, calls
// b3_verify_multiple_checked, which reuses the parsed + checked signatures left in the context.
extern "C" int b3_sig_precheck(b3_ctx* ctx, const uint8_t* sigs192, size_t n, int64_t* first_bad) {
    CKR(begin(ctx));
    if (first_bad) *first_bad = -1;
    ctx->pre_n = (size_t)-1;
    if (n == 0) { ctx->pre_n = 0; return B3_OK; }
    if (!sigs192) return B3_ERR_ARG;
    CKR(h2d(ctx, ctx->in_a, sigs192, 192 * n));
    CKR(ensure(ctx, ctx->g2a_sig, sizeof(g2_aff) * (n + 1)));
    CKR(ensure(ctx, ctx->status, 4 * (2 * n + 8)));
    CKR(ensure(ctx, ctx->ok, 4 * (n + 8)));
    CKR(ensure(ctx, ctx->misc, 64));
    long long* d_fb = (long long*)ctx->misc.p + 4;
    ctx->h_init[0] = B3_FB_NONE;
    CK(cudaMemcpyAsync(d_fb, ctx->h_init, 8, cudaMemcpyHostToDevice, ctx->stream));
    LAUNCH(k_g2_parse, nblk(n), B3_TPB, (const uint8_t*)ctx->in_a.p, n, (g2_aff*)ctx->g2a_sig.p, (int32_t*)ctx->status.p, 1);
    LAUNCH(k_g2_subgroup<lanes_pair>, nblk(2 * n), B3_TPB, (const g2_aff*)ctx->g2a_sig.p, (const int32_t*)ctx->status.p, n, (int32_t*)ctx->ok.p);
    LAUNCH(k_first_bad, nblk(n), B3_TPB, (const int32_t*)ctx->ok.p, n, 0LL, d_fb);
    CKR(first_status(ctx, (const int32_t*)ctx->status.p, n));          // malformed signature: the AmclError code
    long long fb = 0;
    CKR(d2h(ctx, &fb, d_fb, 8));
    CKR(sync(ctx));
    if (first_bad) *first_bad = fb == B3_FB_NONE ? -1 : fb;
    ctx->pre_n = n;
    return B3_OK;
}
extern "C" int b3_verify_multiple_checked(b3_ctx* ctx, const uint8_t* pks96, const uint32_t* pk_off, const uint8_t* msgs, const uint32_t* msg_off,
                                          const uint64_t* scalars, size_t n, int* accept, uint8_t* gt576) {
    if (accept) *accept = 0;
    CKR(vm_begin(ctx));
    vm_in in;
    CKR(vm_stage_host(ctx, in, nullptr, nullptr, pks96, pk_off, msgs, msg_off, scalars, n, 0, n));
    return vm_whole(ctx, in, accept, nullptr, gt576);
}
// verify_multiple over a key table: set j owns the table entries key_idx[pk_off[j] .. pk_off[j+1]) (pk_off == NULL: one entry per
// set).  sigs192 == NULL: the signatures of the preceding b3_sig_precheck.
extern "C" int b3_verify_multiple_indexed(b3_ctx* ctx, const b3_keytable* tbl, const uint8_t* sigs192, const uint32_t* key_idx,
                                          const uint32_t* pk_off, const uint8_t* msgs, const uint32_t* msg_off, const uint64_t* scalars, size_t n,
                                          int* accept, int64_t* first_bad, uint8_t* gt576) {
    if (accept) *accept = 0;
    if (first_bad) *first_bad = -1;
    CKR(vm_begin(ctx));
    if (!tbl) return B3_ERR_ARG;
    vm_in in;
    CKR(vm_stage_host(ctx, in, tbl, sigs192, key_idx, pk_off, msgs, msg_off, scalars, n, 0, n));
    return vm_whole(ctx, in, accept, first_bad, gt576);
}

// whole calls on inputs already resident in HBM (every pointer is device memory; results come back to the host)
extern "C" int b3_verify_multiple_dev(b3_ctx* ctx, const uint8_t* sigs192_dev, const uint8_t* pks96_dev, const uint32_t* pk_off_dev,
                                      const uint8_t* msgs_dev, const uint32_t* msg_off_dev, const uint64_t* scalars_dev, size_t n, int* accept,
                                      int64_t* first_bad, uint8_t* gt576) {
    if (accept) *accept = 0;
    if (first_bad) *first_bad = -1;
    CKR(vm_begin(ctx));
    vm_in in;
    CKR(vm_fill_dev(ctx, in, nullptr, sigs192_dev, pks96_dev, pk_off_dev, msgs_dev, msg_off_dev, scalars_dev, n, 0, n));
    return vm_whole(ctx, in, accept, first_bad, gt576);
}
extern "C" int b3_verify_multiple_indexed_dev(b3_ctx* ctx, const b3_keytable* tbl, const uint8_t* sigs192_dev, const uint32_t* key_idx_dev,
                                              const uint32_t* pk_off_dev, const uint8_t* msgs_dev, const uint32_t* msg_off_dev,
                                              const uint64_t* scalars_dev, size_t n, int* accept, int64_t* first_bad, uint8_t* gt576) {
    if (accept) *accept = 0;
    if (first_bad) *first_bad = -1;
    CKR(vm_begin(ctx));
    if (!tbl) return B3_ERR_ARG;
    vm_in in;
    CKR(vm_fill_dev(ctx, in, tbl, sigs192_dev, key_idx_dev, pk_off_dev, msgs_dev, msg_off_dev, scalars_dev, n, 0, n));
    return vm_whole(ctx, in, accept, first_bad, gt576);
}
// verify_multiple with the message of set j named by msg_idx[j] among n_msgs messages: one hash_to_G2 and one Miller pair per
// MESSAGE, whose G1 member is the sum of the scaled keys of the sets naming it (bilinearity).  The GT value is the one of the
// ungrouped call on the expanded inputs.  keys = pks96 (tbl == NULL) or u32 indices into tbl; device_pointers != 0: every
// input pointer is device memory (the range check of msg_idx is then a device flag read after the synchronise).
extern "C" int b3_verify_multiple_grouped(b3_ctx* ctx, const b3_keytable* tbl, const uint8_t* sigs192, const void* keys, const uint32_t* pk_off,
                                          const uint8_t* msgs, const uint32_t* msg_off, size_t n_msgs, const uint32_t* msg_idx,
                                          const uint64_t* scalars, size_t n, int device_pointers, int* accept, int64_t* first_bad, uint8_t* gt576) {
    if (accept) *accept = 0;
    if (first_bad) *first_bad = -1;
    CKR(vm_begin(ctx));
    if (n && (!msg_idx || n_msgs == 0 || n_msgs > 0xffffffffu)) {
        ctx->err = "b3_verify_multiple_grouped: n > 0 needs msg_idx and 0 < n_msgs < 2^32";
        return B3_ERR_ARG;
    }
    const size_t nm = n ? n_msgs : 0;
    vm_in in;
    if (device_pointers) {
        CKR(vm_fill_dev(ctx, in, tbl, sigs192, keys, pk_off, msgs, msg_off, scalars, n, 0, nm));
        CKR(ensure(ctx, ctx->in_g, 4 * n + 4));
        if (n) CK(cudaMemcpyAsync(ctx->in_g.p, msg_idx, 4 * n, cudaMemcpyDeviceToDevice, ctx->stream));   // locate reads it after the call
    } else {
        for (size_t j = 0; j < n; j++)
            if (msg_idx[j] >= n_msgs) { ctx->err = "b3_verify_multiple_grouped: msg_idx[j] >= n_msgs"; return B3_ERR_ARG; }
        CKR(vm_stage_host(ctx, in, tbl, sigs192, keys, pk_off, msgs, msg_off, scalars, n, 0, nm));
        CKR(h2d(ctx, ctx->in_g, msg_idx, 4 * n));
    }
    if (n) in.d_msg_idx = (const uint32_t*)ctx->in_g.p;
    return vm_whole(ctx, in, accept, first_bad, gt576);
}
// Per-set verdicts of the preceding whole call: set j is valid iff sig_j passed subgroup_check_g2 and e(sig_j, -G1) e(H_j, apk_j)
// == 1, which is verify_multiple over set j alone (c_j is invertible mod r, so the scalar drops out).  The call left in the
// context everything but the signatures' point chains: H_j's lines (pairs [0, n) of `lines` at stride loc_np -- after a grouped
// call pair msg_idx[j] of [0, n_msgs)), the
// unscaled apk_j (g1j), the parsed signatures (g2a_sig), their subgroup results (ok) and the input statuses (status).  Only
// the loc_* buffers, g2j and outb are written, so locate can be repeated and the next call starts from what it always does.
// The stage times stay those of the batch call.
extern "C" int b3_verify_multiple_locate(b3_ctx* ctx, size_t n, int32_t* valid, size_t* n_invalid) {
    if (!ctx) return B3_ERR_ARG;
    if (ctx->loc_n == (size_t)-1) {
        ctx->err = "b3_verify_multiple_locate: the preceding call on this context is not a whole verify_multiple call that returned B3_OK";
        return B3_ERR_ARG;
    }
    if (n != ctx->loc_n) {
        ctx->err = "b3_verify_multiple_locate: n differs from the n of the preceding verify_multiple call";
        return B3_ERR_ARG;
    }
    if (n && !valid) { ctx->err = "b3_verify_multiple_locate: valid is null"; return B3_ERR_ARG; }
    if (n_invalid) *n_invalid = 0;
    if (ctx->loc_accept) {                     // the batch accepted: so does every set
        for (size_t j = 0; j < n; j++) valid[j] = 1;
        return B3_OK;
    }
    CK(cudaSetDevice(ctx->device));
    call_guard guard(ctx, n);
    CKR(ensure(ctx, ctx->loc_pp, sizeof(g1_pp) * n));
    CKR(miller_reserve(ctx, n, ctx->loc_lines, ctx->loc_qinf));
    CKR(ensure(ctx, ctx->g2j, sizeof(g2_jac) * n));
    CKR(ensure(ctx, ctx->outb, 4 * n));
    int32_t* d_valid = (int32_t*)ctx->outb.p;
    const int32_t* d_st_sig = (const int32_t*)ctx->status.p;
    const int32_t* d_st_key = d_st_sig + n + 4;
    CK(cudaEventRecord(ctx->ev[0], ctx->stream));
    mark_reset(ctx);
    LAUNCH(k_g2_aff_to_jac, nblk(n), B3_TPB, (const g2_aff*)ctx->g2a_sig.p, n, (g2_jac*)ctx->g2j.p);
    CKR(miller_lines(ctx, ctx->stream, (const g2_jac*)ctx->g2j.p, n, 0, n, ctx->loc_lines, ctx->loc_qinf));
    LAUNCH(k_g1_jac_to_pp, nblk(n), B3_TPB, (const g1_jac*)ctx->g1j.p, n, (g1_pp*)ctx->loc_pp.p);
    CK(cudaEventRecord(ctx->ev[2], ctx->stream));
    items_finish(ctx, (const fp2*)ctx->loc_lines.p, (const uint32_t*)ctx->loc_qinf.p, n, 0, (const fp2*)ctx->lines.p, (const uint32_t*)ctx->qinf.p,
                 ctx->loc_np, 0, ctx->loc_idx, (const g1_pp*)ctx->loc_pp.p, n, d_st_sig, d_st_key, B3_KEY_BATCH, d_valid, nullptr, nullptr);
    CK(cudaEventRecord(ctx->ev[3], ctx->stream));
    CK(cudaEventRecord(ctx->ev[1], ctx->stream));
    CKR(d2h(ctx, valid, d_valid, 4 * n));
    CKR(sync(ctx));
    cudaEventElapsedTime(&ctx->last_ms[0], ctx->ev[0], ctx->ev[1]);
    if (cudaEventElapsedTime(&ctx->last_ms[1], ctx->ev[2], ctx->ev[3]) != cudaSuccess) ctx->last_ms[1] = 0.f;
    cudaGetLastError();
    if (n_invalid) for (size_t j = 0; j < n; j++) *n_invalid += valid[j] ? 0 : 1;
    return B3_OK;
}
extern "C" int b3_verify_multiple_partial_dev(b3_ctx* ctx, const uint8_t* sigs192_dev, const uint8_t* pks96_dev, const uint32_t* pk_off_dev,
                                              const uint8_t* msgs_dev, const uint32_t* msg_off_dev, const uint64_t* scalars_dev, size_t n,
                                              int64_t index_base, uint8_t* partial_dev) {
    CKR(vm_begin(ctx));
    if (!partial_dev) return B3_ERR_ARG;
    vm_in in;
    CKR(vm_fill_dev(ctx, in, nullptr, sigs192_dev, pks96_dev, pk_off_dev, msgs_dev, msg_off_dev, scalars_dev, n, index_base, n));
    return vm_partial(ctx, in, partial_dev);
}
extern "C" int b3_verify_multiple_indexed_partial_dev(b3_ctx* ctx, const b3_keytable* tbl, const uint8_t* sigs192_dev, const uint32_t* key_idx_dev,
                                                      const uint32_t* pk_off_dev, const uint8_t* msgs_dev, const uint32_t* msg_off_dev,
                                                      const uint64_t* scalars_dev, size_t n, int64_t index_base, uint8_t* partial_dev) {
    CKR(vm_begin(ctx));
    if (!partial_dev || !tbl) return B3_ERR_ARG;
    vm_in in;
    CKR(vm_fill_dev(ctx, in, tbl, sigs192_dev, key_idx_dev, pk_off_dev, msgs_dev, msg_off_dev, scalars_dev, n, index_base, n));
    return vm_partial(ctx, in, partial_dev);
}
// host-pointer form of the sharded call: this rank's shard comes from HOST memory (the keys are copied on the aggregation
// stream, overlapped with the other stages, as in b3_verify_multiple); the partial stays on the device for the all-gather
extern "C" int b3_verify_multiple_partial(b3_ctx* ctx, const uint8_t* sigs192, const uint8_t* pks96, const uint32_t* pk_off, const uint8_t* msgs,
                                          const uint32_t* msg_off, const uint64_t* scalars, size_t n, int64_t index_base, uint8_t* partial_dev) {
    CKR(vm_begin(ctx));
    if (!partial_dev || (n && !sigs192)) return B3_ERR_ARG;
    vm_in in;
    CKR(vm_stage_host(ctx, in, nullptr, sigs192, pks96, pk_off, msgs, msg_off, scalars, n, index_base, n));
    return vm_partial(ctx, in, partial_dev);
}
extern "C" int b3_verify_multiple_indexed_partial(b3_ctx* ctx, const b3_keytable* tbl, const uint8_t* sigs192, const uint32_t* key_idx,
                                                  const uint32_t* pk_off, const uint8_t* msgs, const uint32_t* msg_off, const uint64_t* scalars,
                                                  size_t n, int64_t index_base, uint8_t* partial_dev) {
    CKR(vm_begin(ctx));
    if (!partial_dev || !tbl || (n && !sigs192)) return B3_ERR_ARG;
    vm_in in;
    CKR(vm_stage_host(ctx, in, tbl, sigs192, key_idx, pk_off, msgs, msg_off, scalars, n, index_base, n));
    return vm_partial(ctx, in, partial_dev);
}
// product of partials [i * stride], i < n_partials -> final exponentiation -> accept / first_bad / GT
static int combine_strided(b3_ctx* ctx, const uint8_t* partials_dev, size_t n_partials, size_t stride, int* accept, int64_t* first_bad, uint8_t* gt576) {
    CK(cudaEventRecord(ctx->ev[2], ctx->stream));
    CK(cudaEventRecord(ctx->ev[3], ctx->stream));
    CKR(ensure(ctx, ctx->f12a, sizeof(fp12) * (n_partials + 1)));
    CKR(ensure(ctx, ctx->f12b, sizeof(fp12) * (n_partials / 2 + 2)));
    CKR(ensure(ctx, ctx->misc, 64));
    long long* d_fb = (long long*)ctx->misc.p;
    ctx->h_init[0] = B3_FB_NONE;
    CK(cudaMemcpyAsync(d_fb, ctx->h_init, 8, cudaMemcpyHostToDevice, ctx->stream));
    LAUNCH(k_unpack_partials, nblk(n_partials), B3_TPB, (const partial_rec*)partials_dev, n_partials, stride, (fp12*)ctx->f12a.p, d_fb);
    fp12* res;
    CKR(fp12_product(ctx, (fp12*)ctx->f12a.p, (fp12*)ctx->f12b.p, n_partials, &res));
    int ok = 0;
    CKR(finish(ctx, res, &ok, gt576));
    long long fb = 0;
    CKR(d2h(ctx, &fb, d_fb, 8));
    CKR(sync(ctx));
    if (fb == B3_FB_NONE) fb = -1;
    if (first_bad) *first_bad = fb;
    if (accept) *accept = (ok && fb < 0) ? 1 : 0;
    return B3_OK;
}
extern "C" int b3_combine_partials_dev(b3_ctx* ctx, const uint8_t* partials_dev, size_t n_partials, int* accept, int64_t* first_bad,
                                       uint8_t* gt576) {
    CKR(begin(ctx));
    if (accept) *accept = 0;
    if (first_bad) *first_bad = -1;
    if (!partials_dev || n_partials == 0) return B3_ERR_ARG;
    CK(cudaEventRecord(ctx->ev[0], ctx->stream));
    mark_reset(ctx);
    return combine_strided(ctx, partials_dev, n_partials, 1, accept, first_bad, gt576);
}

// ---------------------------------------------------------------------------------------------- multi-GPU: the collective
// Signature sets shard by rank (SURVEY.md 8e); each rank's 592-byte partial is combined with ONE ncclAllGather over
// NVLink / NVSwitch and one final exponentiation per rank.  NCCL is bound at run time (dlopen of the libnccl.so.2 that is
// already in the process -- e.g. torch's -- or the system one), so the library itself still links against libcudart only.
//
// A communicator serves `lanes` verification contexts of one process (one host thread + b3_ctx each, the reference's
// threading model).  Call k of lane t is STEP k; the all-gather of a step carries the partials of all its lanes
// (lanes x 592 B per rank) and is issued by whichever lane deposits last, on the communicator's own high-priority stream.
// begin() returns as soon as the partial is deposited; finish() combines once the step has been gathered -- so a lane can
// begin step k + 1 before finishing step k and the collective has a whole call time to complete behind the compute.
// Every rank must use the same `lanes` and make the same number of calls per lane.
struct nccl_api {
    void* h = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    std::string err;
};
static nccl_api* nccl() {
    static nccl_api api;
    static std::once_flag once;
    std::call_once(once, [] {
        const char* env = getenv("B3_NCCL_LIB");
        if (env) api.h = dlopen(env, RTLD_NOW | RTLD_GLOBAL);
        if (!api.h) api.h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);     // the copy already in the process
        if (!api.h) api.h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!api.h) api.h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!api.h) { api.err = "libnccl.so.2 not found (set B3_NCCL_LIB)"; return; }
        api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(api.h, "ncclGetUniqueId");
        api.CommInitRank = (decltype(api.CommInitRank))dlsym(api.h, "ncclCommInitRank");
        api.CommDestroy = (decltype(api.CommDestroy))dlsym(api.h, "ncclCommDestroy");
        api.AllGather = (decltype(api.AllGather))dlsym(api.h, "ncclAllGather");
        api.GetErrorString = (decltype(api.GetErrorString))dlsym(api.h, "ncclGetErrorString");
        if (!api.GetUniqueId || !api.CommInitRank || !api.CommDestroy || !api.AllGather) { api.err = "libnccl: missing symbols"; api.h = nullptr; }
    });
    return &api;
}
#define B3_COMM_DEPTH 4
struct b3_comm {
    int device = 0, nranks = 1, rank = 0, lanes = 1;
    ncclComm_t comm = nullptr;
    cudaStream_t stream = nullptr;
    uint8_t* d_send = nullptr;                         // [DEPTH][lanes][592]
    uint8_t* d_recv = nullptr;                         // [DEPTH][nranks][lanes][592]
    cudaEvent_t ev_dep[B3_COMM_DEPTH][64];             // partial of (slot, lane) is in d_send
    cudaEvent_t ev_done[B3_COMM_DEPTH];                // the all-gather of the slot has completed
    std::mutex mu;
    std::condition_variable cv;
    int deposited[B3_COMM_DEPTH] = {0, 0, 0, 0}, finished[B3_COMM_DEPTH] = {0, 0, 0, 0};
    long long gathered_step[B3_COMM_DEPTH] = {-1, -1, -1, -1};        // step whose all-gather has been issued into the slot
    long long free_from[B3_COMM_DEPTH] = {0, 0, 0, 0};                // first step that may deposit into the slot
    long long lane_next[64];                                          // next step of every lane
    uint64_t collectives = 0;
    std::string err;
};
extern "C" int b3_nccl_unique_id(uint8_t id128[128]) {
    nccl_api* a = nccl();
    if (!a->h || !id128) return B3_ERR_CUDA;
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId");
    ncclUniqueId id;
    if (a->GetUniqueId(&id) != ncclSuccess) return B3_ERR_CUDA;
    memcpy(id128, &id, 128);
    return B3_OK;
}
extern "C" void b3_comm_destroy(b3_comm* c);
extern "C" int b3_comm_create(int device, int nranks, int rank, const uint8_t id128[128], int lanes, b3_comm** out) {
    if (!out) return B3_ERR_ARG;
    *out = nullptr;
    if (nranks < 1 || rank < 0 || rank >= nranks || lanes < 1 || lanes > 64 || (nranks > 1 && !id128)) return B3_ERR_ARG;
    if (cudaSetDevice(device) != cudaSuccess) return B3_ERR_CUDA;
    b3_comm* c = new b3_comm();
    c->device = device; c->nranks = nranks; c->rank = rank; c->lanes = lanes;
    for (int l = 0; l < 64; l++) c->lane_next[l] = 0;
    for (int s = 0; s < B3_COMM_DEPTH; s++) c->free_from[s] = s;          // step k uses slot k % DEPTH
    for (int s = 0; s < B3_COMM_DEPTH; s++) { c->ev_done[s] = nullptr; for (int l = 0; l < 64; l++) c->ev_dep[s][l] = nullptr; }
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    bool ok = cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, prio_hi) == cudaSuccess;
    ok = ok && cudaMalloc((void**)&c->d_send, (size_t)B3_COMM_DEPTH * lanes * B3_PARTIAL_BYTES) == cudaSuccess;
    ok = ok && cudaMalloc((void**)&c->d_recv, (size_t)B3_COMM_DEPTH * nranks * lanes * B3_PARTIAL_BYTES) == cudaSuccess;
    for (int s = 0; ok && s < B3_COMM_DEPTH; s++) {
        ok = cudaEventCreateWithFlags(&c->ev_done[s], cudaEventDisableTiming) == cudaSuccess;
        for (int l = 0; ok && l < lanes; l++) ok = cudaEventCreateWithFlags(&c->ev_dep[s][l], cudaEventDisableTiming) == cudaSuccess;
    }
    if (ok && nranks > 1) {
        nccl_api* a = nccl();
        ncclUniqueId id;
        memcpy(&id, id128, 128);
        ok = a->h && a->CommInitRank(&c->comm, nranks, id, rank) == ncclSuccess;
    }
    if (!ok) { cudaGetLastError(); b3_comm_destroy(c); return B3_ERR_CUDA; }
    *out = c;
    return B3_OK;
}
extern "C" void b3_comm_destroy(b3_comm* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->comm) nccl()->CommDestroy(c->comm);
    if (c->d_send) cudaFree(c->d_send);
    if (c->d_recv) cudaFree(c->d_recv);
    for (int s = 0; s < B3_COMM_DEPTH; s++) {
        if (c->ev_done[s]) cudaEventDestroy(c->ev_done[s]);
        for (int l = 0; l < 64; l++) if (c->ev_dep[s][l]) cudaEventDestroy(c->ev_dep[s][l]);
    }
    if (c->stream) cudaStreamDestroy(c->stream);
    cudaGetLastError();
    delete c;
}
extern "C" uint64_t b3_comm_collective_count(b3_comm* c) { return c ? c->collectives : 0; }
extern "C" const char* b3_comm_last_error(b3_comm* c) { return c ? c->err.c_str() : "null communicator"; }
// deposit the partial at `d_partial` (on ctx->stream) as this lane's contribution to its next step; the last lane of a step
// issues the all-gather.  Returns the step (ticket) in *ticket.
static int comm_deposit(b3_ctx* ctx, b3_comm* c, int lane, const uint8_t* d_partial, long long* ticket) {
    if (lane < 0 || lane >= c->lanes || c->device != ctx->device) return B3_ERR_ARG;
    const long long step = c->lane_next[lane];
    const int slot = (int)(step % B3_COMM_DEPTH);
    {
        std::unique_lock<std::mutex> lk(c->mu);
        if (c->free_from[slot] > step) return B3_ERR_ARG;
        // the slot is reused every DEPTH steps: wait until every lane has finished the step that used it before
        c->cv.wait(lk, [&] { return c->free_from[slot] == step; });
    }
    uint8_t* dst = c->d_send + ((size_t)slot * c->lanes + lane) * B3_PARTIAL_BYTES;
    CK(cudaMemcpyAsync(dst, d_partial, B3_PARTIAL_BYTES, cudaMemcpyDeviceToDevice, ctx->stream));
    CK(cudaEventRecord(c->ev_dep[slot][lane], ctx->stream));
    {
        std::unique_lock<std::mutex> lk(c->mu);
        c->lane_next[lane] = step + 1;
        if (++c->deposited[slot] == c->lanes) {
            for (int l = 0; l < c->lanes; l++) CK(cudaStreamWaitEvent(c->stream, c->ev_dep[slot][l], 0));
            const uint8_t* send = c->d_send + (size_t)slot * c->lanes * B3_PARTIAL_BYTES;
            uint8_t* recv = c->d_recv + (size_t)slot * c->nranks * c->lanes * B3_PARTIAL_BYTES;
            const size_t bytes = (size_t)c->lanes * B3_PARTIAL_BYTES;
            if (c->nranks > 1) {
                // the ONLY collective of the path: nranks x lanes x 592 bytes
                ncclResult_t r = nccl()->AllGather(send, recv, bytes, ncclUint8, c->comm, c->stream);
                if (r != ncclSuccess) {
                    c->err = std::string("ncclAllGather: ") + (nccl()->GetErrorString ? nccl()->GetErrorString(r) : "error");
                    ctx->err = c->err;
                    return B3_ERR_CUDA;
                }
            } else {
                CK(cudaMemcpyAsync(recv, send, bytes, cudaMemcpyDeviceToDevice, c->stream));
            }
            c->collectives++;
            CK(cudaEventRecord(c->ev_done[slot], c->stream));
            c->gathered_step[slot] = step;
            c->cv.notify_all();
        }
    }
    *ticket = step;
    return B3_OK;
}
extern "C" int b3_sharded_finish(b3_ctx* ctx, b3_comm* c, int lane, int64_t ticket, int* accept, int64_t* first_bad, uint8_t* gt576) {
    CKR(begin(ctx));
    if (accept) *accept = 0;
    if (first_bad) *first_bad = -1;
    if (!c || lane < 0 || lane >= c->lanes || ticket < 0 || ticket >= c->lane_next[lane]) return B3_ERR_ARG;
    const int slot = (int)(ticket % B3_COMM_DEPTH);
    {
        std::unique_lock<std::mutex> lk(c->mu);
        c->cv.wait(lk, [&] { return c->gathered_step[slot] >= ticket; });
        if (c->gathered_step[slot] != ticket) return B3_ERR_ARG;         // finished too late: the slot was reused
    }
    CK(cudaStreamWaitEvent(ctx->stream, c->ev_done[slot], 0));
    CK(cudaEventRecord(ctx->ev[0], ctx->stream));
    mark_reset(ctx);
    const uint8_t* recv = c->d_recv + ((size_t)slot * c->nranks * c->lanes + lane) * B3_PARTIAL_BYTES;
    const int rc = combine_strided(ctx, recv, (size_t)c->nranks, (size_t)c->lanes, accept, first_bad, gt576);
    {
        std::unique_lock<std::mutex> lk(c->mu);
        if (++c->finished[slot] == c->lanes) {
            c->finished[slot] = 0;
            c->deposited[slot] = 0;
            c->free_from[slot] = ticket + B3_COMM_DEPTH;
            c->cv.notify_all();
        }
    }
    return rc;
}
// begin: this rank's shard -> partial -> deposited for the step's all-gather.  keys = pks96 (tbl == NULL) or u32 indices into
// tbl; device_pointers != 0: every input pointer is device memory.
extern "C" int b3_sharded_begin(b3_ctx* ctx, b3_comm* c, int lane, const b3_keytable* tbl, const uint8_t* sigs192, const void* keys,
                                const uint32_t* pk_off, const uint8_t* msgs, const uint32_t* msg_off, const uint64_t* scalars, size_t n,
                                int64_t index_base, int device_pointers, int64_t* ticket) {
    CKR(vm_begin(ctx));
    if (!c || !ticket || (n && !sigs192)) return B3_ERR_ARG;
    vm_in in;
    if (device_pointers) CKR(vm_fill_dev(ctx, in, tbl, sigs192, keys, pk_off, msgs, msg_off, scalars, n, index_base, n));
    else CKR(vm_stage_host(ctx, in, tbl, sigs192, keys, pk_off, msgs, msg_off, scalars, n, index_base, n));
    CKR(ensure(ctx, ctx->part, B3_PARTIAL_BYTES));
    CKR(vm_partial(ctx, in, (uint8_t*)ctx->part.p));
    long long t = 0;
    CKR(comm_deposit(ctx, c, lane, (const uint8_t*)ctx->part.p, &t));
    *ticket = t;
    return B3_OK;
}
// The sharded form of verify_multiple_aggregate_signatures (M/src/aggregates.rs:261-316 on sets [index_base, index_base + n) of
// the global batch) in one call: every rank gets the global accept bit, the global first_bad and the GT of the whole batch.
extern "C" int b3_verify_multiple_sharded(b3_ctx* ctx, b3_comm* c, int lane, const b3_keytable* tbl, const uint8_t* sigs192, const void* keys,
                                          const uint32_t* pk_off, const uint8_t* msgs, const uint32_t* msg_off, const uint64_t* scalars, size_t n,
                                          int64_t index_base, int device_pointers, int* accept, int64_t* first_bad, uint8_t* gt576) {
    int64_t t = 0;
    CKR(b3_sharded_begin(ctx, c, lane, tbl, sigs192, keys, pk_off, msgs, msg_off, scalars, n, index_base, device_pointers, &t));
    return b3_sharded_finish(ctx, c, lane, t, accept, first_bad, gt576);
}

// ---------------------------------------------------------------------------------------------- signing-side helpers
extern "C" int b3_g1_mul_gen(b3_ctx* ctx, const uint8_t* scalars32, size_t n, uint8_t* out96) {
    CKR(begin(ctx));
    if (n == 0) return B3_OK;
    if (!scalars32 || !out96) return B3_ERR_ARG;
    CKR(h2d(ctx, ctx->in_a, scalars32, 32 * n));
    CKR(ensure(ctx, ctx->outb, 96 * n));
    LAUNCH(k_g1_mul_gen_u256, nblk(n), B3_TPB, (const uint8_t*)ctx->in_a.p, n, (uint8_t*)ctx->outb.p);
    CKR(d2h(ctx, out96, ctx->outb.p, 96 * n));
    return sync(ctx);
}
extern "C" int b3_g2_mul(b3_ctx* ctx, const uint8_t* pts192, const uint8_t* scalars32, size_t n, uint8_t* out192) {
    CKR(begin(ctx));
    if (n == 0) return B3_OK;
    if (!pts192 || !scalars32 || !out192) return B3_ERR_ARG;
    CKR(h2d(ctx, ctx->in_a, pts192, 192 * n));
    CKR(h2d(ctx, ctx->in_b, scalars32, 32 * n));
    CKR(ensure(ctx, ctx->outb, 192 * n));
    LAUNCH(k_g2_mul_u256, nblk(n), B3_TPB, (const uint8_t*)ctx->in_a.p, (const uint8_t*)ctx->in_b.p, n, (uint8_t*)ctx->outb.p);
    CKR(d2h(ctx, out192, ctx->outb.p, 192 * n));
    return sync(ctx);
}

// ---------------------------------------------------------------------------------------------- roofline probe
extern "C" int b3_imad_peak(b3_ctx* ctx, int wide, double* ops_per_s) {
    CKR(begin(ctx));
    if (!ops_per_s) return B3_ERR_ARG;
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, ctx->device));
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    CKR(ensure(ctx, ctx->outb, (size_t)blocks * threads * 4));
    double best = 0;
    for (int rep = 0; rep < 5; rep++) {
        CK(cudaEventRecord(ctx->ev[0], ctx->stream));
    mark_reset(ctx);
        if (wide) LAUNCH(k_imad_wide_peak, blocks, threads, (uint32_t*)ctx->outb.p, iters, 12345u + rep);
        else LAUNCH(k_imad_peak, blocks, threads, (uint32_t*)ctx->outb.p, iters, 12345u + rep);
        CK(cudaEventRecord(ctx->ev[1], ctx->stream));
        CKR(sync(ctx));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]));
        // per thread per iteration: IMAD probe 64 IMADs; wide probe 4*8 = 32 mad.lo/madc.hi PAIRS (= 32 32x32->64 MACs)
        double ops = (double)blocks * threads * (double)iters * (wide ? 32.0 : 64.0);
        double rate = ops / (ms * 1e-3);
        if (rate > best) best = rate;
    }
    *ops_per_s = best;
    return B3_OK;
}
