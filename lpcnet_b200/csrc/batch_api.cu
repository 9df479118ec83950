// batch_api.cu — C-ABI of include/lpcnet_b200.h: batches of independent streams stepped in lockstep.
//
// Per call: [H2D features] -> (per chunk of <= CHUNK frames) frame network + LPC kernels -> persistent per-sample
// kernel -> [D2H PCM].  The per-stream state mirrors the resettable part of struct LPCNetState
// (reference src/lpcnet_private.h:28-48) in structure-of-arrays form (stream index fastest) so that lane==stream
// accesses coalesce.  Streams have their own lifecycle: each carries its own frame counter (silent warm-up frames after
// a reset, lpcnet.c:239-243), can be reset / exported / imported individually, and the whole batch can be snapshotted
// and rolled back on the device (what the reference's PLC does by copying LPCNetState by value, lpcnet_plc.c:216-230).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "engine.h"
#include "devmath.cuh"
#include "../../include/lpcnet_b200.h"

namespace lpcnet_b200 { const char *get_error(); }
using namespace lpcnet_b200;

#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { set_error("%s failed: %s", #call, cudaGetErrorString(e_)); return -1; } } while (0)

static const int CHUNK = FRAME_CHUNK;   // frames of conditioning buffered per sample-kernel launch
static const int DEFER_MAX = 4;     // MAX_FEATURE_BUFFER_SIZE (lpcnet_private.h:26): conv1.kernel_size + conv2.kernel_size - 2

// the sample-rate part of the per-stream state (resettable part of struct LPCNetState), structure of arrays
struct SampleState { float *hA, *hB, *last_sig, *deemph; int *last_exc; uint32_t *rng; };

struct LPCNetB200Batch {
    int device, n;
    DeviceModel model;
    FrameState fs;
    SampleState ss;
    SampleState shadow;                           // scratch copy for frames in which only SOME streams are still in their silent warm-up
    int *d_nsil;                                  // [n] silent frames of each stream in the segment being processed (mixed segments only)
    std::vector<int> *fc;                         // host mirror of fs.frame_count
    // work buffers
    float *condA, *condB, *lpc_raw;
    int cond_last;                                // chunk position of the most recent frame-network output (for the *_tail entry point), -1 = none
    float *d_features; size_t d_features_cap;     // staging for host-pointer calls / decoder output
    short *d_pcm; size_t d_pcm_cap;
    uint8_t *d_packets; size_t d_packets_cap;
    float *d_state; size_t d_state_cap;           // staging for export/import of one stream's state
    std::vector<float> *deferred; int deferred_fill;   // run_frame_network_deferred buffer: [DEFER_MAX][n][20] on the host
    cudaStream_t stream;
    // Ordering of the engine state across CUDA streams: every call that enqueues work records `order_ev` on the stream it
    // used; the next call makes ITS stream wait for that event first (and host-side readers synchronise on it).  A caller
    // may therefore pass a different cuda_stream to every `_device` call, or mix them with the host-pointer calls.
    cudaEvent_t order_ev; cudaStream_t last_stream; bool has_order;
    int env_spc;                                  // LPCNET_B200_STREAMS_PER_CTA (0: automatic)
    bool env_exact_cvt, env_float_lane_stream, env_two_halves;    // LPCNET_B200_EXACT_CVT / _FLOAT_LANE_STREAM / _TWO_HALVES, read once at create time (tests)
    cudaEvent_t ev0, ev1;                         // user timer (lpcnet_b200_batch_timer_*)
    std::vector<cudaEvent_t> *kev;                // event pairs around every per-sample kernel launch of the last call
    int kev_used;
    int last_launches;
    // PCM sink (multi-GPU gather): after every chunk the chunk's PCM block is also copied, on a copy stream that overlaps the next
    // chunk's kernels, to sink + row0*pitch (a buffer of another device / another process opened through CUDA IPC)
    short *sink; long long sink_pitch; long long sink_row0; cudaStream_t sink_stream; cudaEvent_t sink_ev, sink_done;
};

static int order_sync(LPCNetB200Batch *b);
// grow a staging buffer; work on any stream may still be using the old one, so wait for it before freeing
static int ensure(LPCNetB200Batch *b, void **p, size_t *cap, size_t bytes)
{
    if (*cap >= bytes) return 0;
    if (order_sync(b)) return -1;
    if (*p) cudaFree(*p);
    *p = nullptr; *cap = 0;
    CK(cudaMalloc(p, bytes));
    *cap = bytes;
    return 0;
}

// stream hand-over (see LPCNetB200Batch::order_ev)
static int order_enter(LPCNetB200Batch *b, cudaStream_t st)
{
    if (b->has_order && b->last_stream != st) CK(cudaStreamWaitEvent(st, b->order_ev, 0));
    return 0;
}
static int order_leave(LPCNetB200Batch *b, cudaStream_t st)
{
    CK(cudaEventRecord(b->order_ev, st));
    b->last_stream = st; b->has_order = true;
    return 0;
}
static int order_sync(LPCNetB200Batch *b)       // host-side readers / writers of the state: wait for whatever ran last
{
    if (b->has_order) CK(cudaEventSynchronize(b->order_ev));
    return 0;
}

// The RCPPS look-up of the per-sample kernel forms its table address as `table | index` (devmath.cuh), which needs the
// table 8 KB-aligned in the SHARED WINDOW; the image offsets assume dynamic shared memory starts at SMEM_RESERVED.
// Probed once per device at create time so that a driver with a different reservation fails here with a message,
// not with a trap inside the kernel.
__global__ void smem_base_probe_kernel(uint32_t *out)
{
    extern __shared__ __align__(128) uint8_t probe_smem[];
    *out = (uint32_t)__cvta_generic_to_shared(probe_smem);
}
static int probe_smem_base(uint32_t *base)
{
    uint32_t *d = nullptr;
    CK(cudaMalloc(&d, 4));
    CK(cudaFuncSetAttribute(smem_base_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    smem_base_probe_kernel<<<1, 32, 227 * 1024>>>(d);
    cudaError_t e = cudaMemcpy(base, d, 4, cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (e != cudaSuccess) { set_error("shared-memory probe failed: %s", cudaGetErrorString(e)); return -1; }
    return 0;
}

// Live streams per CTA: a batch smaller than 32 x SM count is spread over all SMs (one CTA per SM, fewer live slots each)
// instead of filling a few SMs completely: the time of a CTA-step barely depends on how many of its slots are live.
int lpcnet_b200::streams_per_cta_for(int n_streams, int override_spc)
{
    // (spc <= 16 additionally selects the half-A-only schedule)
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
    int spc = (n_streams + sms - 1) / sms;
    if (override_spc > 0) spc = override_spc;                    // LPCNET_B200_STREAMS_PER_CTA, read once per batch at create time (tests, tuning)
    return spc < 1 ? 1 : spc > STREAMS_PER_CTA ? STREAMS_PER_CTA : spc;
}
int lpcnet_b200::sample_kernel_smem_ok(uint32_t bytes) { return bytes <= 227u * 1024u; }

#ifdef LPCNET_TRACE
static long long *g_trace = nullptr;
extern "C" __attribute__((visibility("default"))) int lpcnet_b200_debug_read_trace(long long *out)
{
    if (!g_trace) return -1;
    cudaDeviceSynchronize();
    return cudaMemcpy(out, g_trace, (8 * 32 + 8 * 32 * 16) * 8, cudaMemcpyDeviceToHost) == cudaSuccess ? 0 : -1;   // + [8 samples][32 warps][16 events] per-warp stamps
}
#endif

// kiss99_srand(&rng, "LPCNet", 6): reference src/kiss99.c:32-57 called from lpcnet_reset (src/lpcnet.c:176-181).
static void kiss99_seed(uint32_t st[4])
{
    const unsigned char *d = (const unsigned char *)"LPCNet"; const int nd = 6;
    uint32_t z = 362436069u, w = 521288629u, jsr = 123456789u, jcong = 380116160u;
    int i;
    for (i = 3; i < nd; i += 4) {
        z ^= d[i - 3]; w ^= d[i - 2]; jsr ^= d[i - 1]; jcong ^= d[i];
        uint32_t znew = 36969u * (z & 0xFFFF) + (z >> 16), wnew = 18000u * (w & 0xFFFF) + (w >> 16);
        uint32_t shr3 = jsr ^ (jsr << 13); shr3 ^= shr3 >> 17; shr3 ^= shr3 << 5;
        z = znew; w = wnew; jsr = shr3; jcong = 69069u * jcong + 1234567u;
    }
    if (i - 3 < nd) z ^= d[i - 3];
    if (i - 2 < nd) w ^= d[i - 2];
    if (i - 1 < nd) jsr ^= d[i - 1];
    if (z == 0 || z == 0x9068FFFF) z++;
    if (w == 0 || w == 0x464FFFFF) w++;
    if (jsr == 0) jsr++;
    st[0] = z; st[1] = w; st[2] = jsr; st[3] = jcong;
}

// ------------------------------------------------------------------------------------------------------------------
// per-stream state kernels (rare paths: resets, export / import, mixed silent segments) — plain strided copies
struct StateView {
    int n, na;
    SampleState ss;
    FrameState fs;
};
// words of one stream's exported state: floats hA[na] hB[16] last_sig[16] deemph conv1[168] conv2[256] lpc_carry[2][16] vq_mem[18],
// then ints last_exc, frame_count, rng[4]
__host__ __device__ inline int state_words(int na) { return na + NB + LPC_ORDER + 1 + 2 * FRAME_IN + 2 * COND + 2 * LPC_ORDER + NB_BANDS + 6; }

// dir 0: state of stream s -> buf, dir 1: buf -> state of stream s
__global__ void state_pack_kernel(StateView v, int s, float *buf, int dir)
{
    const size_t n = v.n;
    int o = 0;
    auto mv = [&](float *base, size_t stride, int count, size_t off) {
        for (int i = threadIdx.x; i < count; i += blockDim.x) { float *p = base + off + (size_t)i * stride; if (dir) *p = buf[o + i]; else buf[o + i] = *p; }
        o += count;
    };
    mv(v.ss.hA, n, v.na, s); mv(v.ss.hB, n, NB, s); mv(v.ss.last_sig, n, LPC_ORDER, s); mv(v.ss.deemph, 1, 1, s);
    mv(v.fs.conv1_state, 1, 2 * FRAME_IN, (size_t)s * 2 * FRAME_IN); mv(v.fs.conv2_state, 1, 2 * COND, (size_t)s * 2 * COND);
    mv(v.fs.lpc_carry, 1, LPC_ORDER, (size_t)s * LPC_ORDER); mv(v.fs.lpc_carry, 1, LPC_ORDER, (n + s) * LPC_ORDER);
    mv(v.fs.vq_mem, 1, NB_BANDS, (size_t)s * NB_BANDS);
    mv(reinterpret_cast<float *>(v.ss.last_exc), 1, 1, s); mv(reinterpret_cast<float *>(v.fs.frame_count), 1, 1, s);
    mv(reinterpret_cast<float *>(v.ss.rng), n, 4, s);
}

// lpcnet_reset (lpcnet.c:174-182) for the listed streams (ids == NULL: all n streams); signal_only = lpcnet_reset_signal (lpcnet.c:226-233)
__global__ void reset_streams_kernel(StateView v, const int *ids, int count, uint4 seed, int signal_only)
{
    const int k = blockIdx.x;
    if (k >= count) return;
    const size_t n = v.n, s = ids ? ids[k] : k;
    for (int i = threadIdx.x; i < v.na; i += blockDim.x) v.ss.hA[i * n + s] = 0.f;
    for (int i = threadIdx.x; i < NB; i += blockDim.x) { v.ss.hB[i * n + s] = 0.f; v.ss.last_sig[i * n + s] = 0.f; }
    if (threadIdx.x == 0) { v.ss.deemph[s] = 0.f; v.ss.last_exc[s] = 128; }      // last_exc = lin2ulaw(0.f) = 128 (lpcnet.c:180)
    if (signal_only) return;
    for (int i = threadIdx.x; i < 2 * FRAME_IN; i += blockDim.x) v.fs.conv1_state[s * 2 * FRAME_IN + i] = 0.f;
    for (int i = threadIdx.x; i < 2 * COND; i += blockDim.x) v.fs.conv2_state[s * 2 * COND + i] = 0.f;
    for (int i = threadIdx.x; i < LPC_ORDER; i += blockDim.x) { v.fs.lpc_carry[s * LPC_ORDER + i] = 0.f; v.fs.lpc_carry[(n + s) * LPC_ORDER + i] = 0.f; }
    for (int i = threadIdx.x; i < NB_BANDS; i += blockDim.x) v.fs.vq_mem[s * NB_BANDS + i] = 0.f;
    if (threadIdx.x == 0) {
        v.fs.frame_count[s] = 0;
        v.ss.rng[s] = seed.x; v.ss.rng[n + s] = seed.y; v.ss.rng[2 * n + s] = seed.z; v.ss.rng[3 * n + s] = seed.w;
    }
}

// after a one-frame launch over a MIXED segment: streams still in their silent warm-up (f < nsil[s]) get their sample-rate
// state back from the shadow copy and zeros as output (lpcnet.c:239-243: RNN_CLEAR(output), return — nothing advances)
__global__ void restore_silent_kernel(SampleState cur, SampleState old, const int *nsil, int f, int n, int na, short *pcm, long long pcm_stride, int spf)
{
    const int s = blockIdx.x;
    if (s >= n || f >= nsil[s]) return;
    const size_t nn = n;
    for (int i = threadIdx.x; i < na; i += blockDim.x) cur.hA[i * nn + s] = old.hA[i * nn + s];
    for (int i = threadIdx.x; i < NB; i += blockDim.x) { cur.hB[i * nn + s] = old.hB[i * nn + s]; cur.last_sig[i * nn + s] = old.last_sig[i * nn + s]; }
    if (threadIdx.x < 4) cur.rng[threadIdx.x * nn + s] = old.rng[threadIdx.x * nn + s];
    if (threadIdx.x == 0) { cur.deemph[s] = old.deemph[s]; cur.last_exc[s] = old.last_exc[s]; }
    for (int i = threadIdx.x; i < spf; i += blockDim.x) pcm[(size_t)s * pcm_stride + i] = 0;
}

static StateView view_of(LPCNetB200Batch *b) { return StateView{b->n, b->model.na, b->ss, b->fs}; }

static int alloc_sample_state(SampleState *ss, size_t n, int na)
{
    CK(cudaMalloc((void **)&ss->hA, sizeof(float) * na * n)); CK(cudaMalloc((void **)&ss->hB, sizeof(float) * NB * n));
    CK(cudaMalloc((void **)&ss->last_sig, sizeof(float) * LPC_ORDER * n)); CK(cudaMalloc((void **)&ss->deemph, sizeof(float) * n));
    CK(cudaMalloc((void **)&ss->last_exc, sizeof(int) * n)); CK(cudaMalloc((void **)&ss->rng, sizeof(uint32_t) * 4 * n));
    return 0;
}
static void free_sample_state(SampleState *ss)
{
    void *p[] = {ss->hA, ss->hB, ss->last_sig, ss->deemph, ss->last_exc, ss->rng};
    for (void *q : p) if (q) cudaFree(q);
    memset(ss, 0, sizeof(*ss));
}
static int copy_sample_state(const SampleState &dst, const SampleState &src, size_t n, int na, cudaStream_t st)
{
    CK(cudaMemcpyAsync(dst.hA, src.hA, sizeof(float) * na * n, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(dst.hB, src.hB, sizeof(float) * NB * n, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(dst.last_sig, src.last_sig, sizeof(float) * LPC_ORDER * n, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(dst.deemph, src.deemph, sizeof(float) * n, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(dst.last_exc, src.last_exc, sizeof(int) * n, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(dst.rng, src.rng, sizeof(uint32_t) * 4 * n, cudaMemcpyDeviceToDevice, st));
    return 0;
}

extern "C" {

int lpcnet_b200_version(void) { return 200; }
const char *lpcnet_b200_last_error(void) { return get_error(); }

int lpcnet_b200_device_count(void)
{
    int c = 0;
    if (cudaGetDeviceCount(&c) != cudaSuccess) { cudaGetLastError(); return 0; }
    return c;
}

static int reset_impl(LPCNetB200Batch *b, const int *ids, int count, int signal_only)
{
    CK(cudaSetDevice(b->device));
    if (order_enter(b, b->stream)) return -1;
    uint32_t seed[4];
    kiss99_seed(seed);
    int *d_ids = nullptr;
    if (ids) {
        for (int k = 0; k < count; k++) if (ids[k] < 0 || ids[k] >= b->n) { set_error("reset_streams: stream %d out of range", ids[k]); return -1; }
        CK(cudaMalloc((void **)&d_ids, sizeof(int) * count));
        CK(cudaMemcpyAsync(d_ids, ids, sizeof(int) * count, cudaMemcpyHostToDevice, b->stream));
    }
    reset_streams_kernel<<<count, 128, 0, b->stream>>>(view_of(b), d_ids, count, make_uint4(seed[0], seed[1], seed[2], seed[3]), signal_only);
    if (order_leave(b, b->stream)) return -1;
    CK(cudaStreamSynchronize(b->stream));
    if (d_ids) cudaFree(d_ids);
    if (!signal_only) {
        if (ids) for (int k = 0; k < count; k++) (*b->fc)[ids[k]] = 0;
        else std::fill(b->fc->begin(), b->fc->end(), 0);
        if (!ids) { b->cond_last = -1; b->deferred_fill = 0; }
    }
    return 0;
}

int lpcnet_b200_batch_reset(LPCNetB200Batch *b)
{
    if (!b) { set_error("null batch"); return -1; }
    return reset_impl(b, nullptr, b->n, 0);
}
int lpcnet_b200_batch_reset_streams(LPCNetB200Batch *b, const int *streams, int count)
{
    if (!b || !streams || count < 0) { set_error("reset_streams: bad arguments"); return -1; }
    return count ? reset_impl(b, streams, count, 0) : 0;
}
int lpcnet_b200_batch_reset_signal(LPCNetB200Batch *b)
{
    if (!b) { set_error("null batch"); return -1; }
    return reset_impl(b, nullptr, b->n, 1);
}

LPCNetB200Batch *lpcnet_b200_batch_create_ex(int n_streams, const unsigned char *blob, int blob_len, const LPCNetB200Config *cfg, int device)
{
    if (n_streams <= 0) { set_error("n_streams must be positive"); return nullptr; }
    int cnt = lpcnet_b200_device_count();
    if (cnt <= 0) { set_error("no CUDA device available (this engine has no CPU fallback)"); return nullptr; }
    if (device < 0 || device >= cnt) { set_error("device %d out of range (%d devices)", device, cnt); return nullptr; }
    if (cudaSetDevice(device) != cudaSuccess) { set_error("cudaSetDevice(%d) failed", device); return nullptr; }
    LPCNetB200Batch *b = (LPCNetB200Batch *)calloc(1, sizeof(*b));
    b->device = device; b->n = n_streams; b->cond_last = -1;
    b->kev = new std::vector<cudaEvent_t>();
    b->fc = new std::vector<int>(n_streams, 0);
    b->deferred = new std::vector<float>();
    ModelConfig mc{-1.f, -1, -1};
    if (cfg) { mc.lpc_gamma = cfg->lpc_gamma; mc.features_delay = cfg->features_delay; mc.end2end = cfg->end2end; }
    if (model_load(&b->model, blob, blob_len, &mc) != 0) { delete b->kev; delete b->fc; delete b->deferred; free(b); return nullptr; }
    const size_t n = n_streams;
    const int na = b->model.na;
    bool ok = alloc_sample_state(&b->ss, n, na) == 0;
    auto al = [&](void **p, size_t bytes) { if (ok && cudaMalloc(p, bytes) != cudaSuccess) ok = false; };
    al((void **)&b->fs.conv1_state, sizeof(float) * 2 * FRAME_IN * n); al((void **)&b->fs.conv2_state, sizeof(float) * 2 * COND * n);
    al((void **)&b->fs.lpc_carry, sizeof(float) * 2 * LPC_ORDER * n); al((void **)&b->fs.vq_mem, sizeof(float) * NB_BANDS * n);
    al((void **)&b->fs.frame_count, sizeof(int) * n);
    al((void **)&b->fs.work, sizeof(float) * frame_work_floats(n));
    al((void **)&b->condA, sizeof(float) * (size_t)CHUNK * condA_frame_floats(b->model.is_float != 0, n, na)); al((void **)&b->condB, sizeof(float) * (size_t)CHUNK * n * 3 * NB);
    al((void **)&b->lpc_raw, sizeof(float) * (size_t)(CHUNK + 2) * n * LPC_ORDER);
    if (ok && cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking) != cudaSuccess) ok = false;
    if (ok && (cudaStreamCreateWithFlags(&b->fs.side, cudaStreamNonBlocking) != cudaSuccess || cudaEventCreateWithFlags(&b->fs.ev_fork, cudaEventDisableTiming) != cudaSuccess ||
               cudaEventCreateWithFlags(&b->fs.ev_join, cudaEventDisableTiming) != cudaSuccess)) ok = false;
    if (ok && (cudaEventCreate(&b->ev0) != cudaSuccess || cudaEventCreate(&b->ev1) != cudaSuccess)) ok = false;
    if (ok && cudaEventCreateWithFlags(&b->order_ev, cudaEventDisableTiming) != cudaSuccess) ok = false;
    { const char *e = getenv("LPCNET_B200_STREAMS_PER_CTA"); b->env_spc = e ? atoi(e) : 0; }
    b->env_exact_cvt = getenv("LPCNET_B200_EXACT_CVT") != nullptr;
    b->env_float_lane_stream = getenv("LPCNET_B200_FLOAT_LANE_STREAM") != nullptr;
    b->env_two_halves = getenv("LPCNET_B200_TWO_HALVES") != nullptr;
    if (!ok) { set_error("device allocation failed: %s", cudaGetErrorString(cudaGetLastError())); lpcnet_b200_batch_destroy(b); return nullptr; }
    if (!b->model.is_float) {
        uint32_t base = 0;
        const Geom G = make_geom(na);
        if (probe_smem_base(&base)) { lpcnet_b200_batch_destroy(b); return nullptr; }
        if ((base + G.sm_image + G.im_rcp) % 8192u != 0) {
            set_error("dynamic shared memory starts at window offset %u on this driver, the image layout assumes %u (engine.h SMEM_RESERVED)", base, SMEM_RESERVED);
            lpcnet_b200_batch_destroy(b); return nullptr;
        }
    }
    if (lpcnet_b200_batch_reset(b) != 0) { lpcnet_b200_batch_destroy(b); return nullptr; }
    return b;
}

LPCNetB200Batch *lpcnet_b200_batch_create(int n_streams, const unsigned char *blob, int blob_len, float lpc_gamma, int device)
{
    LPCNetB200Config c = {lpc_gamma, -1, -1};       // FEATURES_DELAY / END2END: the blob's metadata record if it has one, else 2 / 0
    return lpcnet_b200_batch_create_ex(n_streams, blob, blob_len, &c, device);
}

void lpcnet_b200_batch_destroy(LPCNetB200Batch *b)
{
    if (!b) return;
    cudaSetDevice(b->device);
    if (b->stream) cudaStreamSynchronize(b->stream);
    if (b->fs.side) { cudaStreamSynchronize(b->fs.side); cudaStreamDestroy(b->fs.side); }
    if (b->fs.ev_fork) cudaEventDestroy(b->fs.ev_fork);
    if (b->fs.ev_join) cudaEventDestroy(b->fs.ev_join);
    if (b->sink_stream) { cudaStreamSynchronize(b->sink_stream); cudaStreamDestroy(b->sink_stream); }
    if (b->sink_ev) cudaEventDestroy(b->sink_ev);
    if (b->sink_done) cudaEventDestroy(b->sink_done);
    free_sample_state(&b->ss); free_sample_state(&b->shadow);
    void *ptrs[] = {b->fs.conv1_state, b->fs.conv2_state, b->fs.lpc_carry, b->fs.vq_mem, b->fs.frame_count, b->fs.work, b->condA, b->condB, b->lpc_raw,
                    b->d_features, b->d_pcm, b->d_packets, b->d_state, b->d_nsil};
    for (void *p : ptrs) if (p) cudaFree(p);
    if (b->kev) { for (cudaEvent_t e : *b->kev) cudaEventDestroy(e); delete b->kev; }
    delete b->fc; delete b->deferred;
    model_free(&b->model);
    if (b->ev0) cudaEventDestroy(b->ev0);
    if (b->ev1) cudaEventDestroy(b->ev1);
    if (b->order_ev) { if (b->has_order) cudaEventSynchronize(b->order_ev); cudaEventDestroy(b->order_ev); }
    if (b->stream) cudaStreamDestroy(b->stream);
    free(b);
}

int lpcnet_b200_batch_streams(const LPCNetB200Batch *b) { return b ? b->n : 0; }
int lpcnet_b200_batch_is_float(const LPCNetB200Batch *b) { return b ? b->model.is_float : -1; }
int lpcnet_b200_batch_model_info(const LPCNetB200Batch *b, int *gru_a_units, LPCNetB200Config *cfg)
{
    if (!b) { set_error("null batch"); return -1; }
    if (gru_a_units) *gru_a_units = b->model.na;
    if (cfg) { cfg->lpc_gamma = b->model.cfg.lpc_gamma; cfg->features_delay = b->model.cfg.features_delay; cfg->end2end = b->model.cfg.end2end; }
    return 0;
}

int lpcnet_b200_batch_set_codebooks(LPCNetB200Batch *b, const float *cb, size_t n_floats)
{
    if (!b) { set_error("null batch"); return -1; }
    const size_t want = 3 * 1024 * 17 + 4096 * 18;
    if (!cb || n_floats != want) { set_error("codebooks: expected %zu floats", want); return -1; }
    CK(cudaSetDevice(b->device));
    if (!b->model.codebooks) CK(cudaMalloc((void **)&b->model.codebooks, want * sizeof(float)));
    CK(cudaMemcpy(b->model.codebooks, cb, want * sizeof(float), cudaMemcpyHostToDevice));
    return 0;
}

// launch the per-sample kernel for `nf` frames whose conditioning sits at chunk position `pos`
static int launch_sample(LPCNetB200Batch *b, int pos, int nf, int spf, short *pcm, long long pcm_stride, int preload, cudaStream_t st, bool time_it)
{
    const int n = b->n, na = b->model.na;
    SampleParams p = {};
    p.L = b->model.L; p.image = b->model.image;
    p.emb_sig = b->model.emb_sig; p.emb_pred = b->model.emb_pred; p.emb_exc = b->model.emb_exc; p.fcw = b->model.fcw;
    p.spc = streams_per_cta_for(n, b->env_spc);
    p.one_half = p.spc <= HALF && !b->env_two_halves;
    p.fast_cvt = ((b->model.fast_cvt && !b->env_exact_cvt) ? 1 : 0) | (preload << 8);   // env LPCNET_B200_EXACT_CVT: force the conversion-unit path (tests)
#ifdef LPCNET_TRACE
    { static long long *d_trace = nullptr; if (!d_trace) { CK(cudaMalloc(&d_trace, (8 * 32 + 8 * 32 * 16) * 8)); CK(cudaMemset(d_trace, 0, (8 * 32 + 8 * 32 * 16) * 8)); } p.trace = d_trace; g_trace = d_trace; }
#endif
    const int d = b->model.cfg.end2end ? 0 : b->model.cfg.features_delay;   // frame f uses lpc_raw entry f + 2 - d (frame_kernels.cu)
    p.condA = b->condA + (size_t)pos * condA_frame_floats(b->model.is_float != 0, n, na);
    p.condB = b->condB + (size_t)pos * n * 3 * NB;
    p.lpc_raw = b->lpc_raw + (size_t)(pos + 2 - d) * n * LPC_ORDER;
    p.gamma_pow = b->model.gamma_pow;
    p.hA = b->ss.hA; p.hB = b->ss.hB; p.last_sig = b->ss.last_sig; p.deemph = b->ss.deemph; p.last_exc = b->ss.last_exc; p.rng = b->ss.rng;
    p.pcm = pcm;
    p.pcm_stream_stride = pcm_stride;
    p.n_streams = n; p.nframes = nf; p.spf = spf;
    if (time_it) {      // event pair around the launch, resolved lazily by lpcnet_b200_batch_last_sample_kernel_ms (no sync here)
        while ((int)b->kev->size() < b->kev_used + 2) { cudaEvent_t e; CK(cudaEventCreate(&e)); b->kev->push_back(e); }
        CK(cudaEventRecord((*b->kev)[b->kev_used], st));
    }
    const bool small_float = b->model.is_float && p.spc <= FN_S && !b->env_float_lane_stream;
    if (small_float) { p.L = b->model.Ln; p.image = b->model.image_n; }       // small batch: neuron-per-lane float kernel
    cudaError_t e;
#define LPCNET_DISPATCH(ns) (small_float ? ns::launch_sample_kernel_f32n(p, st) : b->model.is_float ? ns::launch_sample_kernel_f32(p, st) : ns::launch_sample_kernel(p, st))
    switch (na) {
    case 128: e = LPCNET_DISPATCH(na128); break;
    case 256: e = LPCNET_DISPATCH(na256); break;
    default:  e = LPCNET_DISPATCH(na384); break;
    }
#undef LPCNET_DISPATCH
    if (e != cudaSuccess) { set_error("per-sample kernel launch failed: %s", cudaGetErrorString(e)); return -1; }
    if (time_it) { CK(cudaEventRecord((*b->kev)[b->kev_used + 1], st)); b->kev_used += 2; }
    return 0;
}

// The sample loops of the frames at chunk positions [pos0, pos0 + nf): per stream, frames whose post-increment frame
// counter is <= FEATURES_DELAY are silent and do not advance the sample state (lpcnet.c:239-243).  b->fc = the streams'
// counters before frame pos0 (host mirror), advanced here.  Returns the number of engine kernels launched, < 0 on error.
static int sample_frames(LPCNetB200Batch *b, int pos0, int nf, int spf, short *pcm, long long pcm_stride, int preload, cudaStream_t st)
{
    const int n = b->n, delay = b->model.cfg.features_delay;
    int fc_min = 1 << 30, fc_max = 0;
    for (int v : *b->fc) { fc_min = std::min(fc_min, v); fc_max = std::max(fc_max, v); }
    const int sil_all = std::min(nf, std::max(0, delay - fc_max));     // frames silent for EVERY stream
    const int sil_any = std::min(nf, std::max(0, delay - fc_min));     // frames silent for at least one stream
    int launches = 0;
    if (sil_all > 0) CK(cudaMemset2DAsync(pcm, pcm_stride * sizeof(short), 0, (size_t)sil_all * spf * sizeof(short), n, st));
    if (sil_any > sil_all) {
        // mixed segment (some streams were reset later than others): one launch per frame over all streams, then the streams
        // that are still silent get their state back and zeros as output
        if (!b->shadow.hA && alloc_sample_state(&b->shadow, n, b->model.na)) return -1;
        if (!b->d_nsil) CK(cudaMalloc((void **)&b->d_nsil, sizeof(int) * n));
        std::vector<int> nsil(n);
        for (int s = 0; s < n; s++) nsil[s] = std::min(nf, std::max(0, delay - (*b->fc)[s]));
        CK(cudaMemcpyAsync(b->d_nsil, nsil.data(), sizeof(int) * n, cudaMemcpyHostToDevice, st));
        CK(cudaStreamSynchronize(st));                              // (nsil is a stack vector; this path runs at most FEATURES_DELAY times per reset)
        for (int f = sil_all; f < sil_any; f++) {
            if (copy_sample_state(b->shadow, b->ss, n, b->model.na, st)) return -1;
            if (launch_sample(b, pos0 + f, 1, spf, pcm + (size_t)f * spf, pcm_stride, f == 0 ? preload : 0, st, true)) return -1;
            restore_silent_kernel<<<n, 128, 0, st>>>(b->ss, b->shadow, b->d_nsil, f, n, b->model.na, pcm + (size_t)f * spf, pcm_stride, spf);
            launches += 2;
        }
    }
    if (nf > sil_any) {
        if (launch_sample(b, pos0 + sil_any, nf - sil_any, spf, pcm + (size_t)sil_any * spf, pcm_stride, sil_any == 0 ? preload : 0, st, true)) return -1;
        launches += 1;
    }
    for (int &v : *b->fc) v = std::min(1000, v + nf);
    return launches;
}

// chunk [c0, c0+nf) of a call is complete on `st`: forward its PCM block to the sink (if one is set) on the copy stream
static int forward_to_sink(LPCNetB200Batch *b, const short *d_pcm, long long pcm_stride, int c0, int nf, int spf, cudaStream_t st)
{
    if (!b->sink) return 0;
    CK(cudaEventRecord(b->sink_ev, st));
    CK(cudaStreamWaitEvent(b->sink_stream, b->sink_ev, 0));
    short *dst = b->sink + b->sink_row0 * b->sink_pitch + (size_t)c0 * spf;
    if (c0 == 0 && (long long)nf * spf == pcm_stride && b->sink_pitch == pcm_stride)      // whole rows, same pitch: one contiguous block (one DMA descriptor
        CK(cudaMemcpyAsync(dst, d_pcm, (size_t)b->n * pcm_stride * sizeof(short), cudaMemcpyDefault, b->sink_stream));   // instead of n row copies)
    else
        CK(cudaMemcpy2DAsync(dst, b->sink_pitch * sizeof(short), d_pcm + (size_t)c0 * spf, pcm_stride * sizeof(short), (size_t)nf * spf * sizeof(short), b->n,
                             cudaMemcpyDefault, b->sink_stream));       // (the sink may live on another device: UVA infers the route)
    return 0;
}

// Core: features and pcm are device pointers. `st` is the stream all work is enqueued on.
static int synth_device(LPCNetB200Batch *b, const float *d_feat, long long stream_stride, int frame_stride, int nframes,
                        int spf, short *d_pcm, int preload, cudaStream_t st)
{
    if (!b) { set_error("null batch"); return -1; }
    if (nframes <= 0) return 0;
    if (spf < 1 || spf > 65536) { set_error("samples_per_frame must be in 1..65536"); return -1; }
    if (preload < 0 || preload > spf) { set_error("preload must be in 0..samples_per_frame"); return -1; }
    if (frame_stride < NB_FEAT) { set_error("feature_stride must be >= 20"); return -1; }
    const int n = b->n;
    const long long pcm_stride = (long long)nframes * spf;
    if (b->sink && b->sink_pitch < pcm_stride) { set_error("PCM sink pitch %lld smaller than the call's %lld samples per stream", b->sink_pitch, pcm_stride); return -1; }
    int launches = 0;
    b->kev_used = 0;
    if (order_enter(b, st)) return -1;
    for (int c0 = 0; c0 < nframes; c0 += CHUNK) {
        const int nf = nframes - c0 < CHUNK ? nframes - c0 : CHUNK;
        launch_frame_network(b->model, b->fs, d_feat + (size_t)c0 * frame_stride, stream_stride, frame_stride, n, nf, b->condA, b->condB, b->lpc_raw, st);
        launches += frame_network_launches(b->model);
        b->cond_last = nf - 1;
        const int r = sample_frames(b, 0, nf, spf, d_pcm + (size_t)c0 * spf, pcm_stride, c0 == 0 ? preload : 0, st);
        if (r < 0) return -1;
        launches += r;
        if (forward_to_sink(b, d_pcm, pcm_stride, c0, nf, spf, st)) return -1;
    }
    CK(cudaGetLastError());
    if (b->sink) {       // the call's stream also waits for the forwarded copies: "call complete" includes "PCM at the sink"
        CK(cudaEventRecord(b->sink_done, b->sink_stream));
        CK(cudaStreamWaitEvent(st, b->sink_done, 0));
    }
    if (order_leave(b, st)) return -1;
    b->last_launches = launches;
    return 0;
}

int lpcnet_b200_batch_synthesize_device_ex(LPCNetB200Batch *b, const float *d_features, int nframes, int feature_stride,
                                           int samples_per_frame, short *d_pcm, int preload, void *cuda_stream)
{
    if (!b) { set_error("null batch"); return -1; }
    CK(cudaSetDevice(b->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : b->stream;
    int r = synth_device(b, d_features, (long long)nframes * feature_stride, feature_stride, nframes, samples_per_frame, d_pcm, preload, st);
    if (r == 0 && !cuda_stream) CK(cudaStreamSynchronize(st));
    return r;
}
int lpcnet_b200_batch_synthesize_device(LPCNetB200Batch *b, const float *d_features, int nframes, int feature_stride,
                                        int samples_per_frame, short *d_pcm, void *cuda_stream)
{
    return lpcnet_b200_batch_synthesize_device_ex(b, d_features, nframes, feature_stride, samples_per_frame, d_pcm, 0, cuda_stream);
}

int lpcnet_b200_batch_synthesize_ex(LPCNetB200Batch *b, const float *features, int nframes, int feature_stride,
                                    int samples_per_frame, short *pcm, int preload)
{
    if (!b) { set_error("null batch"); return -1; }
    if (nframes <= 0) return 0;
    if (!features || !pcm) { set_error("null buffer"); return -1; }
    CK(cudaSetDevice(b->device));
    const size_t fbytes = sizeof(float) * (size_t)b->n * nframes * feature_stride;
    const size_t pbytes = sizeof(short) * (size_t)b->n * nframes * samples_per_frame;
    if (ensure(b, (void **)&b->d_features, &b->d_features_cap, fbytes)) return -1;
    if (ensure(b, (void **)&b->d_pcm, &b->d_pcm_cap, pbytes)) return -1;
    if (order_enter(b, b->stream)) return -1;       // the staging buffers may still be read by work on another stream
    CK(cudaMemcpyAsync(b->d_features, features, fbytes, cudaMemcpyHostToDevice, b->stream));
    if (preload > 0)                                // teacher forcing reads the caller's signal from the output buffer (lpcnet.c:257)
        CK(cudaMemcpy2DAsync(b->d_pcm, (size_t)nframes * samples_per_frame * sizeof(short), pcm, (size_t)nframes * samples_per_frame * sizeof(short),
                             (size_t)std::min(preload, samples_per_frame) * sizeof(short), b->n, cudaMemcpyHostToDevice, b->stream));
    if (order_leave(b, b->stream)) return -1;
    if (synth_device(b, b->d_features, (long long)nframes * feature_stride, feature_stride, nframes, samples_per_frame, b->d_pcm, preload, b->stream)) return -1;
    CK(cudaMemcpyAsync(pcm, b->d_pcm, pbytes, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    return 0;
}
int lpcnet_b200_batch_synthesize(LPCNetB200Batch *b, const float *features, int nframes, int feature_stride,
                                 int samples_per_frame, short *pcm)
{
    return lpcnet_b200_batch_synthesize_ex(b, features, nframes, feature_stride, samples_per_frame, pcm, 0);
}

// ---- the reference's internal entry points around the same kernels (lpcnet_private.h:125-133), batched ----
// run_frame_network only (lpcnet.c:82-120): advances the 100 Hz state and the frame counters, keeps the conditioning of the LAST
// frame for lpcnet_b200_batch_synthesize_tail
int lpcnet_b200_batch_run_frame_network(LPCNetB200Batch *b, const float *features, int nframes, int feature_stride)
{
    if (!b) { set_error("null batch"); return -1; }
    if (nframes <= 0) return 0;
    if (!features || feature_stride < NB_FEAT) { set_error("run_frame_network: bad arguments"); return -1; }
    CK(cudaSetDevice(b->device));
    const size_t fbytes = sizeof(float) * (size_t)b->n * nframes * feature_stride;
    if (ensure(b, (void **)&b->d_features, &b->d_features_cap, fbytes)) return -1;
    if (order_enter(b, b->stream)) return -1;
    CK(cudaMemcpyAsync(b->d_features, features, fbytes, cudaMemcpyHostToDevice, b->stream));
    for (int c0 = 0; c0 < nframes; c0 += CHUNK) {
        const int nf = std::min(CHUNK, nframes - c0);
        launch_frame_network(b->model, b->fs, b->d_features + (size_t)c0 * feature_stride, (long long)nframes * feature_stride, feature_stride, b->n, nf,
                             b->condA, b->condB, b->lpc_raw, b->stream);
        b->cond_last = nf - 1;
        for (int &v : *b->fc) v = std::min(1000, v + nf);
    }
    if (order_leave(b, b->stream)) return -1;
    CK(cudaStreamSynchronize(b->stream));
    return 0;
}

// lpcnet_synthesize_tail_impl (lpcnet.c:235-271): `samples` more samples with the conditioning of the last frame-network run
int lpcnet_b200_batch_synthesize_tail(LPCNetB200Batch *b, int samples, short *pcm, int preload)
{
    if (!b || !pcm || samples < 1 || samples > 65536) { set_error("synthesize_tail: bad arguments"); return -1; }
    if (preload < 0 || preload > samples) { set_error("preload must be in 0..samples"); return -1; }
    if (b->cond_last < 0) { set_error("synthesize_tail: no frame network output yet"); return -1; }
    CK(cudaSetDevice(b->device));
    const size_t pbytes = sizeof(short) * (size_t)b->n * samples;
    if (ensure(b, (void **)&b->d_pcm, &b->d_pcm_cap, pbytes)) return -1;
    if (order_enter(b, b->stream)) return -1;
    if (preload > 0) CK(cudaMemcpyAsync(b->d_pcm, pcm, pbytes, cudaMemcpyHostToDevice, b->stream));
    b->kev_used = 0;
    // the frame counters were already advanced by the frame network run; the silent test of lpcnet.c:239 looks at the CURRENT
    // count, sample_frames() at the count before the frame: step back by one for the duration of the call
    std::vector<int> saved = *b->fc;
    for (int &v : *b->fc) v = v - 1;
    const int r = sample_frames(b, b->cond_last, 1, samples, b->d_pcm, samples, preload, b->stream);
    *b->fc = saved;
    if (r < 0) return -1;
    b->last_launches = r;
    if (order_leave(b, b->stream)) return -1;
    CK(cudaMemcpyAsync(pcm, b->d_pcm, pbytes, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    return 0;
}

// run_frame_network_deferred / _flush (lpcnet.c:122-144): queue up to 4 feature frames without evaluating the network; the
// flush runs the frame network over them (outputs discarded, state and frame counters advance)
int lpcnet_b200_batch_frame_network_deferred(LPCNetB200Batch *b, const float *features, int feature_stride)
{
    if (!b || !features || feature_stride < NB_FEAT) { set_error("frame_network_deferred: bad arguments"); return -1; }
    const size_t fr = (size_t)b->n * NB_FEAT;
    b->deferred->resize(fr * DEFER_MAX);
    float *q = b->deferred->data();
    if (b->deferred_fill == DEFER_MAX) memmove(q, q + fr, sizeof(float) * fr * (DEFER_MAX - 1));
    else b->deferred_fill++;
    float *dst = q + fr * (b->deferred_fill - 1);
    for (int s = 0; s < b->n; s++) memcpy(dst + (size_t)s * NB_FEAT, features + (size_t)s * feature_stride, sizeof(float) * NB_FEAT);
    return 0;
}
int lpcnet_b200_batch_frame_network_flush(LPCNetB200Batch *b)
{
    if (!b) { set_error("null batch"); return -1; }
    const int fill = b->deferred_fill;
    if (fill == 0) return 0;
    const size_t fr = (size_t)b->n * NB_FEAT;
    std::vector<float> f((size_t)b->n * fill * NB_FEAT);             // [n][fill][20]
    for (int k = 0; k < fill; k++) for (int s = 0; s < b->n; s++)
        memcpy(&f[((size_t)s * fill + k) * NB_FEAT], b->deferred->data() + fr * k + (size_t)s * NB_FEAT, sizeof(float) * NB_FEAT);
    b->deferred_fill = 0;
    return lpcnet_b200_batch_run_frame_network(b, f.data(), fill, NB_FEAT);
}

static int decode_device(LPCNetB200Batch *b, const uint8_t *d_packets, int npackets, short *d_pcm, cudaStream_t st)
{
    if (!b->model.codebooks) { set_error("decode: no VQ codebooks loaded (lpcnet_b200_batch_set_codebooks)"); return -1; }
    const size_t fbytes = sizeof(float) * (size_t)b->n * npackets * 4 * NB_FEAT;
    if (ensure(b, (void **)&b->d_features, &b->d_features_cap, fbytes)) return -1;
    if (order_enter(b, st)) return -1;
    launch_decode_packets(b->model, b->fs, d_packets, b->n, npackets, b->d_features, st);
    if (order_leave(b, st)) return -1;
    int r = synth_device(b, b->d_features, (long long)npackets * 4 * NB_FEAT, NB_FEAT, npackets * 4, FRAME_SIZE, d_pcm, 0, st);
    b->last_launches += 1;
    return r;
}

int lpcnet_b200_batch_decode_device(LPCNetB200Batch *b, const unsigned char *d_packets, int npackets, short *d_pcm, void *cuda_stream)
{
    if (!b) { set_error("null batch"); return -1; }
    if (npackets <= 0) return 0;
    CK(cudaSetDevice(b->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : b->stream;
    int r = decode_device(b, d_packets, npackets, d_pcm, st);
    if (r == 0 && !cuda_stream) CK(cudaStreamSynchronize(st));
    return r;
}

int lpcnet_b200_batch_decode(LPCNetB200Batch *b, const unsigned char *packets, int npackets, short *pcm)
{
    if (!b) { set_error("null batch"); return -1; }
    if (npackets <= 0) return 0;
    if (!packets || !pcm) { set_error("null buffer"); return -1; }
    CK(cudaSetDevice(b->device));
    const size_t kbytes = (size_t)b->n * npackets * 8, pbytes = sizeof(short) * (size_t)b->n * npackets * 640;
    if (ensure(b, (void **)&b->d_packets, &b->d_packets_cap, kbytes)) return -1;
    if (ensure(b, (void **)&b->d_pcm, &b->d_pcm_cap, pbytes)) return -1;
    if (order_enter(b, b->stream)) return -1;
    CK(cudaMemcpyAsync(b->d_packets, packets, kbytes, cudaMemcpyHostToDevice, b->stream));
    if (order_leave(b, b->stream)) return -1;
    if (decode_device(b, b->d_packets, npackets, b->d_pcm, b->stream)) return -1;
    CK(cudaMemcpyAsync(pcm, b->d_pcm, pbytes, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    return 0;
}

float lpcnet_b200_batch_last_sample_kernel_ms(const LPCNetB200Batch *b, int *launches)
{
    if (!b) return 0.f;
    if (launches) *launches = b->last_launches;
    float total = 0.f;
    for (int i = 0; i + 1 < b->kev_used; i += 2) {
        float ms = 0.f;
        if (cudaEventSynchronize((*b->kev)[i + 1]) != cudaSuccess) return -1.f;
        if (cudaEventElapsedTime(&ms, (*b->kev)[i], (*b->kev)[i + 1]) != cudaSuccess) return -1.f;
        total += ms;
    }
    return total;
}

// ---- PCM sink: the multi-GPU gather as part of the call (SURVEY 8e: the only exchange of the path) ----
int lpcnet_b200_batch_set_pcm_sink(LPCNetB200Batch *b, short *sink, long long pitch_samples, long long first_row)
{
    if (!b) { set_error("null batch"); return -1; }
    CK(cudaSetDevice(b->device));
    if (order_sync(b)) return -1;
    if (sink && !b->sink_stream) {
        CK(cudaStreamCreateWithFlags(&b->sink_stream, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&b->sink_ev, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&b->sink_done, cudaEventDisableTiming));
    }
    if (b->sink_stream) CK(cudaStreamSynchronize(b->sink_stream));
    b->sink = sink; b->sink_pitch = pitch_samples; b->sink_row0 = first_row;
    return 0;
}
int lpcnet_b200_ipc_export(void *d_ptr, unsigned char handle[64])
{
    cudaIpcMemHandle_t h;
    static_assert(sizeof(h) == 64, "CUDA IPC handle size");
    CK(cudaIpcGetMemHandle(&h, d_ptr));
    memcpy(handle, &h, 64);
    return 0;
}
void *lpcnet_b200_ipc_open(const unsigned char handle[64])
{
    cudaIpcMemHandle_t h; memcpy(&h, handle, 64);
    void *p = nullptr;
    if (cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { set_error("cudaIpcOpenMemHandle: %s", cudaGetErrorString(cudaGetLastError())); return nullptr; }
    return p;
}
int lpcnet_b200_ipc_close(void *p) { CK(cudaIpcCloseMemHandle(p)); return 0; }

// CUDA-event stopwatch on the engine's own stream (the stream every engine kernel is launched on when the caller
// passes cuda_stream == NULL): start records an event, stop records another, synchronises and returns the ms between.
int lpcnet_b200_batch_timer_start(LPCNetB200Batch *b)
{
    if (!b) { set_error("null batch"); return -1; }
    CK(cudaSetDevice(b->device));
    CK(cudaEventRecord(b->ev0, b->stream));
    return 0;
}
float lpcnet_b200_batch_timer_stop(LPCNetB200Batch *b)
{
    if (!b) return -1.f;
    float ms = 0.f;
    if (cudaEventRecord(b->ev1, b->stream) != cudaSuccess || cudaEventSynchronize(b->ev1) != cudaSuccess ||
        cudaEventElapsedTime(&ms, b->ev0, b->ev1) != cudaSuccess) { set_error("timer: %s", cudaGetErrorString(cudaGetLastError())); return -1.f; }
    return ms;
}
// Evict L2 between timed iterations: overwrite a scratch buffer larger than the 126 MB L2 on the engine's stream.
int lpcnet_b200_batch_flush_l2(LPCNetB200Batch *b)
{
    if (!b) { set_error("null batch"); return -1; }
    static void *scratch[64] = {nullptr};
    const size_t bytes = 256u << 20;
    CK(cudaSetDevice(b->device));
    if (b->device < 0 || b->device >= 64) { set_error("flush_l2: device index"); return -1; }
    if (!scratch[b->device]) CK(cudaMalloc(&scratch[b->device], bytes));
    CK(cudaMemsetAsync(scratch[b->device], 0x5a, bytes, b->stream));
    return 0;
}
int lpcnet_b200_batch_sync(LPCNetB200Batch *b)
{
    if (!b) { set_error("null batch"); return -1; }
    CK(cudaSetDevice(b->device));
    if (order_sync(b)) return -1;
    CK(cudaStreamSynchronize(b->stream));
    return 0;
}
// Device memory helpers so that a plain-C / ctypes caller can keep inputs resident in HBM (no torch needed).
void *lpcnet_b200_device_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaMalloc(&p, bytes) != cudaSuccess) { set_error("cudaMalloc(%zu) failed", bytes); return nullptr; }
    return p;
}
void lpcnet_b200_device_free(void *p) { if (p) cudaFree(p); }
int lpcnet_b200_memcpy_h2d(void *dst, const void *src, size_t bytes) { CK(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice)); return 0; }
int lpcnet_b200_memcpy_d2h(void *dst, const void *src, size_t bytes) { CK(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost)); return 0; }
int lpcnet_b200_set_device(int device) { CK(cudaSetDevice(device)); return 0; }
// CUDA streams for callers without their own CUDA binding (the `cuda_stream` argument of the `_device` entry points)
void *lpcnet_b200_stream_create(void)
{
    cudaStream_t s = nullptr;
    if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess) { set_error("cudaStreamCreate failed"); return nullptr; }
    return s;
}
void lpcnet_b200_stream_destroy(void *s) { if (s) cudaStreamDestroy((cudaStream_t)s); }
int lpcnet_b200_stream_sync(void *s) { CK(cudaStreamSynchronize((cudaStream_t)s)); return 0; }

int lpcnet_b200_batch_algorithmic_bytes(const LPCNetB200Batch *b, long *total, long *sparse_gemv)
{
    if (!b) { set_error("null batch"); return -1; }
    if (total) *total = b->model.algo_bytes_total;
    if (sparse_gemv) *sparse_gemv = b->model.algo_bytes_sparse;
    return 0;
}

int lpcnet_b200_batch_get_state(LPCNetB200Batch *b, int s, float *gru_a, float *gru_b, float *last_sig, int *misc, uint32_t *rng)
{
    if (!b || s < 0 || s >= b->n) { set_error("bad stream index"); return -1; }
    CK(cudaSetDevice(b->device));
    if (order_sync(b)) return -1;
    const size_t n = b->n;
    if (gru_a) CK(cudaMemcpy2D(gru_a, sizeof(float), b->ss.hA + s, n * sizeof(float), sizeof(float), b->model.na, cudaMemcpyDeviceToHost));
    if (gru_b) CK(cudaMemcpy2D(gru_b, sizeof(float), b->ss.hB + s, n * sizeof(float), sizeof(float), NB, cudaMemcpyDeviceToHost));
    if (last_sig) CK(cudaMemcpy2D(last_sig, sizeof(float), b->ss.last_sig + s, n * sizeof(float), sizeof(float), LPC_ORDER, cudaMemcpyDeviceToHost));
    if (misc) { CK(cudaMemcpy(&misc[0], b->ss.last_exc + s, sizeof(int), cudaMemcpyDeviceToHost)); misc[1] = (*b->fc)[s]; }
    if (rng) CK(cudaMemcpy2D(rng, sizeof(uint32_t), b->ss.rng + s, n * sizeof(uint32_t), sizeof(uint32_t), 4, cudaMemcpyDeviceToHost));
    return 0;
}

// ---- state by value (what the PLC does with `LPCNetState copy = *st`, lpcnet_plc.c:216-230): one stream <-> host blob ----
int lpcnet_b200_batch_state_size(const LPCNetB200Batch *b)
{
    return b ? state_words(b->model.na) * 4 : -1;
}
static int state_move(LPCNetB200Batch *b, int s, void *buf, int dir)
{
    if (!b || !buf || s < 0 || s >= b->n) { set_error("state export/import: bad arguments"); return -1; }
    CK(cudaSetDevice(b->device));
    const size_t bytes = (size_t)state_words(b->model.na) * 4;
    if (ensure(b, (void **)&b->d_state, &b->d_state_cap, bytes)) return -1;
    if (order_enter(b, b->stream)) return -1;
    if (dir) CK(cudaMemcpyAsync(b->d_state, buf, bytes, cudaMemcpyHostToDevice, b->stream));
    state_pack_kernel<<<1, 128, 0, b->stream>>>(view_of(b), s, b->d_state, dir);
    if (!dir) CK(cudaMemcpyAsync(buf, b->d_state, bytes, cudaMemcpyDeviceToHost, b->stream));
    if (order_leave(b, b->stream)) return -1;
    CK(cudaStreamSynchronize(b->stream));
    if (dir) {
        int fcv; memcpy(&fcv, (const char *)buf + (size_t)(state_words(b->model.na) - 5) * 4, 4);
        (*b->fc)[s] = fcv;
    }
    return 0;
}
int lpcnet_b200_batch_export_state(LPCNetB200Batch *b, int s, void *buf) { return state_move(b, s, buf, 0); }
int lpcnet_b200_batch_import_state(LPCNetB200Batch *b, int s, const void *buf) { return state_move(b, s, const_cast<void *>(buf), 1); }

// ---- whole-batch snapshot on the device (roll-back after speculative synthesis) ----
struct LPCNetB200Snapshot {
    int n, na, device;
    SampleState ss; FrameState fs;
    std::vector<int> *fc; int cond_last; int deferred_fill; std::vector<float> *deferred;
};
void lpcnet_b200_batch_snapshot_destroy(LPCNetB200Snapshot *s)
{
    if (!s) return;
    cudaSetDevice(s->device);
    free_sample_state(&s->ss);
    void *ptrs[] = {s->fs.conv1_state, s->fs.conv2_state, s->fs.lpc_carry, s->fs.vq_mem, s->fs.frame_count};
    for (void *p : ptrs) if (p) cudaFree(p);
    delete s->fc; delete s->deferred;
    free(s);
}
LPCNetB200Snapshot *lpcnet_b200_batch_snapshot_create(LPCNetB200Batch *b)
{
    if (!b) { set_error("null batch"); return nullptr; }
    if (cudaSetDevice(b->device) != cudaSuccess) return nullptr;
    LPCNetB200Snapshot *s = (LPCNetB200Snapshot *)calloc(1, sizeof(*s));
    s->n = b->n; s->na = b->model.na; s->device = b->device;
    s->fc = new std::vector<int>(b->n, 0); s->deferred = new std::vector<float>();
    const size_t n = b->n;
    bool ok = alloc_sample_state(&s->ss, n, s->na) == 0;
    auto al = [&](void **p, size_t bytes) { if (ok && cudaMalloc(p, bytes) != cudaSuccess) ok = false; };
    al((void **)&s->fs.conv1_state, sizeof(float) * 2 * FRAME_IN * n); al((void **)&s->fs.conv2_state, sizeof(float) * 2 * COND * n);
    al((void **)&s->fs.lpc_carry, sizeof(float) * 2 * LPC_ORDER * n); al((void **)&s->fs.vq_mem, sizeof(float) * NB_BANDS * n);
    al((void **)&s->fs.frame_count, sizeof(int) * n);
    if (!ok) { set_error("snapshot: device allocation failed"); lpcnet_b200_batch_snapshot_destroy(s); return nullptr; }
    return s;
}
static int copy_frame_state(const FrameState &dst, const FrameState &src, size_t n, cudaStream_t st)
{
    CK(cudaMemcpyAsync(dst.conv1_state, src.conv1_state, sizeof(float) * 2 * FRAME_IN * n, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(dst.conv2_state, src.conv2_state, sizeof(float) * 2 * COND * n, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(dst.lpc_carry, src.lpc_carry, sizeof(float) * 2 * LPC_ORDER * n, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(dst.vq_mem, src.vq_mem, sizeof(float) * NB_BANDS * n, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(dst.frame_count, src.frame_count, sizeof(int) * n, cudaMemcpyDeviceToDevice, st));
    return 0;
}
int lpcnet_b200_batch_snapshot_save(LPCNetB200Batch *b, LPCNetB200Snapshot *s)
{
    if (!b || !s || s->n != b->n || s->na != b->model.na || s->device != b->device) { set_error("snapshot does not belong to this batch"); return -1; }
    CK(cudaSetDevice(b->device));
    if (order_enter(b, b->stream)) return -1;
    if (copy_sample_state(s->ss, b->ss, b->n, s->na, b->stream) || copy_frame_state(s->fs, b->fs, b->n, b->stream)) return -1;
    if (order_leave(b, b->stream)) return -1;
    *s->fc = *b->fc; s->cond_last = b->cond_last; s->deferred_fill = b->deferred_fill; *s->deferred = *b->deferred;
    return 0;
}
int lpcnet_b200_batch_snapshot_restore(LPCNetB200Batch *b, const LPCNetB200Snapshot *s)
{
    if (!b || !s || s->n != b->n || s->na != b->model.na || s->device != b->device) { set_error("snapshot does not belong to this batch"); return -1; }
    CK(cudaSetDevice(b->device));
    if (order_enter(b, b->stream)) return -1;
    if (copy_sample_state(b->ss, s->ss, b->n, s->na, b->stream) || copy_frame_state(b->fs, s->fs, b->n, b->stream)) return -1;
    if (order_leave(b, b->stream)) return -1;
    *b->fc = *s->fc; b->deferred_fill = s->deferred_fill; *b->deferred = *s->deferred;
    b->cond_last = -1;            // the conditioning buffers are not part of the snapshot: a tail call needs a fresh frame-network run
    return 0;
}

// Test hook: run ONLY the frame-rate kernels on host features for a fresh batch state and return all taps.
// ga [n][nframes][3*na], gb [n][nframes][48], lpc [n][nframes][16] (gamma-weighted, i.e. what the sample loop uses)
int lpcnet_b200_debug_frame_network(LPCNetB200Batch *b, const float *features, int nframes, int feature_stride,
                                                  float *ga, float *gb, float *lpc)
{
    if (!b) { set_error("null batch"); return -1; }
    if (nframes > CHUNK) { set_error("debug_frame_network: at most %d frames", CHUNK); return -1; }
    CK(cudaSetDevice(b->device));
    const int n = b->n, na = b->model.na;
    const size_t fbytes = sizeof(float) * (size_t)n * nframes * feature_stride;
    if (order_sync(b)) return -1;
    if (ensure(b, (void **)&b->d_features, &b->d_features_cap, fbytes)) return -1;
    CK(cudaMemcpyAsync(b->d_features, features, fbytes, cudaMemcpyHostToDevice, b->stream));
    launch_frame_network(b->model, b->fs, b->d_features, (long long)nframes * feature_stride, feature_stride, n, nframes,
                         b->condA, b->condB, b->lpc_raw, b->stream);
    for (int &v : *b->fc) v = std::min(1000, v + nframes);
    b->cond_last = nframes - 1;
    const bool isf = b->model.is_float != 0;
    const size_t fA = condA_frame_floats(isf, n, na);
    std::vector<float> hA((size_t)nframes * fA), hB((size_t)nframes * n * 3 * NB), hl((size_t)(nframes + 2) * n * LPC_ORDER), gp(LPC_ORDER);
    CK(cudaMemcpyAsync(hA.data(), b->condA, hA.size() * 4, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaMemcpyAsync(hB.data(), b->condB, hB.size() * 4, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaMemcpyAsync(hl.data(), b->lpc_raw, hl.size() * 4, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaMemcpyAsync(gp.data(), b->model.gamma_pow, LPC_ORDER * 4, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    const int d = b->model.cfg.end2end ? 0 : b->model.cfg.features_delay;
    for (int s = 0; s < n; s++) for (int f = 0; f < nframes; f++) {
        if (isf) memcpy(ga + ((size_t)s * nframes + f) * 3 * na, &hA[((size_t)f * n + s) * 3 * na], sizeof(float) * 3 * na);
        else for (int g = 0; g < 3; g++) memcpy(ga + ((size_t)s * nframes + f) * 3 * na + (size_t)g * na, &hA[(size_t)f * fA + ((size_t)g * n + s) * (na + 8)], sizeof(float) * na);
        memcpy(gb + ((size_t)s * nframes + f) * 3 * NB, &hB[((size_t)f * n + s) * 3 * NB], sizeof(float) * 3 * NB);
        for (int i = 0; i < LPC_ORDER; i++) lpc[((size_t)s * nframes + f) * LPC_ORDER + i] = hl[((size_t)(f + 2 - d) * n + s) * LPC_ORDER + i] * gp[i];
    }
    return 0;
}

// Test hook (host only, no CUDA): the shared-memory image and its run-time layout words
// layout = {wA, metaA, wB, metaB, image_bytes, total_bytes, nblkA_padded, nblkB_padded, sm_image, para, dira, grpa, dirb,
// wbrec, parb, fcw, compute warps, groups per compute warp, dual_fc rows in shared memory, K parts of GRU_B, na, fast_cvt, is_float}.
// Offsets 9..15 are relative to sm_image and belong to the kernel that reads the image: the int8 kernel, or for float blobs the
// lane==stream float kernel (which keeps no dual_fc rows in shared memory: fcw = ~0, rows = 0).
int lpcnet_b200_debug_image(const unsigned char *blob, int len, unsigned char *out, size_t cap, uint32_t *layout)
{
    SmemLayout L; Geom G; int fast_cvt = 0, is_float = 0;
    int r = debug_build_image(blob, len, out, cap, &L, &G, &fast_cvt, &is_float);
    if (r < 0) return r;
    layout[0] = L.wA; layout[1] = L.metaA; layout[2] = L.wB; layout[3] = L.metaB; layout[4] = L.image_bytes; layout[5] = L.total_bytes;
    layout[6] = L.nblkA_padded; layout[7] = L.nblkB_padded; layout[8] = L.sm_image;
    if (is_float) {
        layout[9] = G.fi_para; layout[10] = G.fi_dira; layout[11] = G.fi_grpa; layout[12] = G.fi_dirb; layout[13] = L.wBrecF - L.sm_image; layout[14] = G.fi_parb;
        layout[15] = 0xFFFFFFFFu; layout[16] = F_NWC; layout[17] = G.f_gpw; layout[18] = 0; layout[19] = F_KPARTS;
    } else {
        layout[9] = G.im_para; layout[10] = G.im_dira; layout[11] = G.im_grpa; layout[12] = G.im_dirb; layout[13] = G.im_wbrec; layout[14] = G.im_parb;
        layout[15] = G.im_fcw; layout[16] = NWC; layout[17] = G.gpw; layout[18] = *reinterpret_cast<const uint32_t *>(out + G.im_fcwn); layout[19] = KPARTS;
    }
    layout[20] = G.na; layout[21] = (uint32_t)fast_cvt; layout[22] = (uint32_t)is_float;
    return r;
}

// Test hook: the two device implementations of the reference's _mm256_rcp_ps (table in memory / table-free arithmetic)
// on n host floats.
__global__ void debug_rcp_kernel(const float *x, float *out_table, float *out_arith, int n, const uint16_t *tab16)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out_table[i] = rcp_emul(x[i], tab16);
    out_arith[i] = rcp_emul(x[i], RcpArith());
}
int lpcnet_b200_debug_rcp(LPCNetB200Batch *b, const float *x, float *out_table, float *out_arith, int n)
{
    if (!b || n <= 0) { set_error("debug_rcp: bad arguments"); return -1; }
    CK(cudaSetDevice(b->device));
    float *d = nullptr;
    CK(cudaMalloc(&d, (size_t)3 * n * sizeof(float)));
    CK(cudaMemcpy(d, x, (size_t)n * sizeof(float), cudaMemcpyHostToDevice));
    debug_rcp_kernel<<<(n + 255) / 256, 256, 0, b->stream>>>(d, d + n, d + 2 * n, n, b->model.rcp16);
    CK(cudaStreamSynchronize(b->stream));
    CK(cudaMemcpy(out_table, d + n, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(out_arith, d + 2 * n, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
    cudaFree(d);
    return 0;
}

// Test hook (host only): image of the neuron-per-lane float kernel.  layout = {wA, metaA, wB, metaB, image_bytes, total_bytes,
// nblkA, nblkB, fn_image, fni_neur, fni_dira, fni_para, fni_dirb, fni_parb, fni_wbrec, fni_fcw, dense flag, na}
int lpcnet_b200_debug_image_n(const unsigned char *blob, int len, unsigned char *out, size_t cap, uint32_t *layout)
{
    SmemLayout L; Geom G;
    int r = debug_build_image_n(blob, len, out, cap, &L, &G);
    if (r < 0) return r;
    layout[0] = L.wA; layout[1] = L.metaA; layout[2] = L.wB; layout[3] = L.metaB; layout[4] = L.image_bytes; layout[5] = L.total_bytes;
    layout[6] = L.nblkA_padded; layout[7] = L.nblkB_padded; layout[8] = G.fn_image; layout[9] = G.fni_neur; layout[10] = G.fni_dira; layout[11] = G.fni_para;
    layout[12] = G.fni_dirb; layout[13] = G.fni_parb; layout[14] = G.fni_wbrec; layout[15] = G.fni_fcw; layout[16] = L.wBrecF; layout[17] = G.na;
    return r;
}

// Pinned host memory helpers for callers that want true async H2D/D2H (the benchmark's e2e leg).
void *lpcnet_b200_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) { set_error("cudaHostAlloc(%zu) failed", bytes); return nullptr; }
    return p;
}
void lpcnet_b200_host_free(void *p) { if (p) cudaFreeHost(p); }

}  // extern "C"
