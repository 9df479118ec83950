// sample_kernel.cu — the 16 kHz autoregressive loop as ONE persistent, warp-specialised sm_100a kernel.
//
// Replaces (reference file:line):
//   lpcnet_synthesize_tail_impl  src/lpcnet.c:235-271   (LPC prediction, u-law, de-emphasis, clamp/round)
//   run_sample_network           src/lpcnet.c:146-167
//   compute_gru_a_input          src/nnet.c:484-491     (cond + 3 embedding rows, left to right)
//   compute_sparse_gru           src/nnet.c:410-448  +  sparse_sgemv_accum8x4 (int8) src/vec_avx.h:790-858
//   compute_gruB                 src/nnet.c:326-372  +  sgemv_accum8x4 src/vec_avx.h:690-755
//   sample_mdense                src/nnet.c:163-214  +  kiss99_rand src/kiss99.c:59-81
//   lin2ulaw / ulaw2lin          src/common.h:37-58
//
// One CTA = 32 independent streams on one SM, stepped as two HALVES of 16 streams that run half a sample apart:
// a GRU step cannot start before the previous sample of the same stream has been drawn and its embedding rows gathered,
// so while that serial tail (sampler -> indices -> gather) runs for one half, the compute warps work on the other half.
// NWC + NWP + 1 warps:
//
//   NWC compute warps own 48/NWC neuron groups (8 neurons x {z,r,h}) of GRU_A each.  The integer GEMVs S = W.q(h) of a
//                     half are small GEMMs and run on the tensor cores: mma.sync m16n8k16 (u8 x s8 -> s32, exact, so the
//                     summation order is free): M = the 16 streams of the half, N = the 8 neurons of a row group, K = four
//                     8x4 weight blocks ("quad") whose column blocks may be anywhere (block-sparse): the A fragment of lane
//                     (gid, t) is gathered from the quantised state with ONE LDS.64 (the words of streams gid, gid+8 for
//                     the column block of slot t); the B fragment (the lane's word of the quad's weights) and the slot's column
//                     offset are lane-private constants of the model and live in TENSOR MEMORY (tcgen05.st once per launch,
//                     tcgen05.ld.x4 = the operands of two quads, one pipeline step ahead).  The accumulator layout makes lane
//                     (gid, t) own neurons 2t, 2t+1 of the group for streams gid, gid+8 of each half: the fp32 state of those
//                     (stream, neuron) pairs is private to the lane for the whole launch (parked in tensor memory between the
//                     half's activations) and the activations are evaluated there.  The sums do not depend on the sampled
//                     excitation, so they are computed before the gathered input term is waited for:
//                     acc = rne((bias + diag*h + gin)*16256) + S  is the same integer the reference gets.
//                     Order of a step: GRU_B(B, previous sample) | GEMV r,h (A) | activations A | GRU_B(A) | GEMV r,h (B) |
//                     activations B  (GRU_B right behind its activations: its state is what the half's sampler waits for).
//   NWP producer warps gather the GRU_A input term cond + E_sig[a] + E_pred[b] + E_exc[c] (compute_gru_a_input), one gate of
//                     one half at a time, with 512-byte contiguous LDG.128 into a ring of four [16][392] fp32 tiles
//                     (full/empty mbarriers) that the compute lanes read conflict-free.
//    2 sampler warps  (one per half; lanes 0-15 = the streams, lanes 16-31 shadow them and evaluate the second dual_fc channel)
//                     run the strictly serial tail (two KISS99 draws, 8-level sigmoid tree with sequential fp32 dot
//                     products, ulaw2lin, order-16 LPC filter, de-emphasis, lin2ulaw).
//
// Weights, su-biases, the upper dual_fc levels and the sampler tables are staged into shared memory once per launch
// by TMA bulk copies (cp.async.bulk + mbarrier).  Roles hand data over with mbarriers; the compute warps synchronise
// among themselves with two named barriers.
#include <cstdint>
#include <cstdlib>
#ifndef LPCNET_NA
#define LPCNET_NA 384          // GRU_A units this translation unit is compiled for (lpcnet_b200/build.py compiles one per supported size)
#endif
#include "engine.h"
#include "devmath.cuh"

// tuning builds (-DLPCNET_TRACE): clock64 stamps of CTA 0 for samples 200..207 of a launch
#ifdef LPCNET_TRACE
#define TRACE(P_, step_, ev_, lane_) do { if (blockIdx.x == 0 && (lane_) == 0 && (step_) >= 200 && (step_) < 208) (P_).trace[((step_) - 200) * 32 + (ev_)] = clock64(); } while (0)
#ifdef LPCNET_TRACE_W0
#define TRACEC TRACE         // the detailed stamps of compute warp 0 (they cost that warp ~12 extra clock reads + stores per sample)
#else
#define TRACEC(P_, step_, ev_, lane_) do { } while (0)
#endif
// the same stamp for every warp: [8 samples][32 warps][16 events] behind the first table
#define TRACEW(P_, step_, ev_) do { if (blockIdx.x == 0 && (threadIdx.x & 31) == 0 && (step_) >= 200 && (step_) < 208) (P_).trace[256 + (((step_) - 200) * 32 + (threadIdx.x >> 5)) * 16 + (ev_)] = clock64(); } while (0)
#else
#define TRACE(P_, step_, ev_, lane_) do { } while (0)
#define TRACEC(P_, step_, ev_, lane_) do { } while (0)
#define TRACEW(P_, step_, ev_) do { } while (0)
#endif

namespace lpcnet_b200 {
namespace LPCNET_KNS {

namespace {

// named barriers of the compute warps
enum {
    BAR_X = 1,       // restored state visible (kernel start only)
    BAR_HB = 3       // (+ half) finishing warps arrive, sampler waits: GRU_B state of the half's sample is in hBs
};
constexpr int CNT_C = NWC * 32, CNT_HB = NFIN * 32 + 32;
__device__ __forceinline__ void bar_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }

__device__ __forceinline__ void bar_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- TMA bulk copy global -> shared, completion on an mbarrier ----
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// one arrival per warp: the lanes' shared-memory accesses are ordered before it by the fence + warp barrier.
// -DLPCNET_ARRIVE_ALL (checking builds): every lane arrives itself, so that compute-sanitizer's racecheck, which does not
// chain a warp barrier with an mbarrier, can follow the hand-over.
#ifdef LPCNET_ARRIVE_ALL
constexpr int ARRIVALS_PER_WARP = 32;
__device__ __forceinline__ void warp_arrive(uint32_t bar, int lane) { (void)lane; mbar_arrive(bar); }
#else
constexpr int ARRIVALS_PER_WARP = 1;
__device__ __forceinline__ void warp_arrive(uint32_t bar, int lane)
{
    __threadfence_block();
    __syncwarp();
    if (lane == 0) mbar_arrive(bar);
}
#endif
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}

__device__ __forceinline__ uint32_t lds32(uint32_t addr)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds16(uint32_t addr)
{
    uint32_t v;
    asm volatile("{ .reg .u16 t; ld.shared.u16 t, [%1]; cvt.u32.u16 %0, t; }" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ int2 lds64(uint32_t addr)
{
    int2 v;
    asm volatile("ld.shared.v2.s32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
    return v;
}
// D[16 streams][8 neurons] += A[16 streams][16 inputs] (u8) . B[16 inputs][8 neurons] (s8): exact int32.
// Pinned in program order (volatile) for the hand-scheduled quad pipeline below
__device__ __forceinline__ void imma16816_v(int (&c)[4], const int2 &a, uint32_t b0)
{
    asm volatile("mma.sync.aligned.m16n8k16.row.col.s32.u8.s8.s32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
                 : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3]) : "r"(a.x), "r"(a.y), "r"(b0));
}
// ---- tensor memory as the operand store of the B side ----
// Per quad a lane needs three things: its A fragment (gathered from the quantised state: shared memory, it changes every sample),
// its B fragment word (weights) and its slot's column offset (meta).  The last two are constants of the model and are private to
// one lane of one warp, so they do not have to travel through the L1/shared-memory data pipe — the unit that bounds this kernel
// (DESIGN.md 4.1): at kernel start every compute warp copies its own quads from the shared-memory image into TENSOR MEMORY
// (tcgen05.st, two 32-bit columns per quad: {weights word, meta}), and the GEMV pipeline reads them back with tcgen05.ld
// (SASS LDTM), which has its own datapath (12-cycle latency, 64 B/clk) and leaves the LSU pipe to the state gather, the
// activations' table look-ups and the conditioning tiles.  A warp can only address the 32 TMEM lanes of its quarter
// (warp id mod 4); the four compute warps of a quarter get 128 columns each (TMEM_COLS_PER_WARP; model.cu checks the budget).
constexpr uint32_t TMEM_COLS = 512, TMEM_COLS_PER_WARP = 128;
// Behind the end of a stream the pipeline has fetched four more quads and formed shared-memory addresses from the meta of the first
// two (never multiplied).  The GRU_A stream is followed by the warp's GRU_B stream (valid metas of the same state layout), the last
// stream by QUAD_TAIL copies of a valid quad; what is fetched beyond those is the parked state below (fetched only, never used).
constexpr uint32_t QUAD_TAIL = 2;
constexpr uint32_t TMEM_H_COL = TMEM_COLS_PER_WARP - 8 * (uint32_t)GPW;         // last columns of a warp's range: the lane's fp32 GRU_A state, [half][group][4]
__device__ __forceinline__ void tmem_st2(uint32_t taddr, uint32_t a, uint32_t b)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(taddr), "r"(a), "r"(b) : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// {weights word, meta} of the quad at column `taddr` (asynchronous: valid after tmem_wait_ld on the same registers)
__device__ __forceinline__ void tmem_ld2(uint32_t &w, uint32_t &m, uint32_t taddr)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(w), "=r"(m) : "r"(taddr));
}
// the {weights word, meta} pairs of two consecutive quads with one instruction (four columns)
__device__ __forceinline__ void tmem_ld22(uint32_t &w0, uint32_t &m0, uint32_t &w1, uint32_t &m1, uint32_t taddr)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(w0), "=r"(m0), "=r"(w1), "=r"(m1) : "r"(taddr));
}
// four consecutive columns <-> four floats (the fp32 GRU_A state of a lane parks in tensor memory between its activations, see below)
__device__ __forceinline__ void tmem_ld4f(float (&v)[4], uint32_t taddr)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(taddr));
}
__device__ __forceinline__ void tmem_st4f(uint32_t taddr, const float (&v)[4])
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld4f(float (&v)[4])
{
    asm volatile("tcgen05.wait::ld.sync.aligned;" : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]) :: "memory");
}
// completes every tcgen05.ld this thread has issued; the registers are operands so that no use can be scheduled above the wait
__device__ __forceinline__ void tmem_wait_ld(uint32_t &a, uint32_t &b, uint32_t &c, uint32_t &d)
{
    asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(a), "+r"(b), "+r"(c), "+r"(d) :: "memory");
}

// A stream of quads (several lists back to back) walked with a two-deep operand pipeline:
// set 0 / set 1 hold the A fragment (x) and B fragment (w) of the next two quads, nW* / nM* the {weights, meta} of the two quads
// after those, fetched from tensor memory one pipeline step ahead.  Right after a quad is multiplied its registers are reloaded
// with the quad two positions ahead, so every LDS has two multiplications (and their bookkeeping) to complete, also across list
// boundaries.  QUAD_SLACK readable quads follow every stream; what is loaded past the end of a stream is never used.
//   col : tensor-memory address (lane quarter | column) of the quad in set 0
//   xs  : shared address of the state buffer; the lane's 8-byte vector of slot t is at xs + (meta ^ lc), lc = (half << 6) | (gid << 3)
struct QuadPipe {
    uint32_t col, xs, lc;
    int2 x0, x1;
    uint32_t w0, w1, nW0, nM0, nW1, nM1;
    __device__ __forceinline__ void start(uint32_t col_, uint32_t xs_, uint32_t lc_)
    {
        col = col_; xs = xs_; lc = lc_;
        uint32_t m0, m1;
        tmem_ld2(w0, m0, col); tmem_ld2(w1, m1, col + 2);
        tmem_wait_ld(w0, m0, w1, m1);
        tmem_ld22(nW0, nM0, nW1, nM1, col + 4);
        x0 = lds64(xs + (m0 ^ lc)); x1 = lds64(xs + (m1 ^ lc));
    }
    // acc[2jj+i] += sum over the next `nq` quads of the stream, for stream gid+8jj (of one half) and neuron 2t+i of the row group
    __device__ __forceinline__ void list(int (&acc)[4], int nq)
    {
#pragma unroll 1
        for (; nq >= 2; nq -= 2) {
            imma16816_v(acc, x0, w0);
            tmem_wait_ld(nW0, nM0, nW1, nM1);                     // issued one step ago
            x0 = lds64(xs + (nM0 ^ lc)); w0 = nW0;
            imma16816_v(acc, x1, w1);
            x1 = lds64(xs + (nM1 ^ lc)); w1 = nW1;
            col += 4;
            tmem_ld22(nW0, nM0, nW1, nM1, col + 4);
        }
        if (nq) {                                                // odd tail: multiply set 0, and let the sets trade places
            imma16816_v(acc, x0, w0);
            tmem_wait_ld(nW0, nM0, nW1, nM1);
            x0 = x1; w0 = w1;
            x1 = lds64(xs + (nM0 ^ lc)); w1 = nW0;
            col += 2;
            tmem_ld22(nW0, nM0, nW1, nM1, col + 4);
        }
    }
    // The look-ahead loads of the last step are still in flight when a stream ends: they must land before the registers they
    // write are given to anything else (tcgen05.ld completes asynchronously, outside the register scoreboard).
    __device__ __forceinline__ void finish() { tmem_wait_ld(nW0, nM0, nW1, nM1); }
};

// Stream slots of a CTA: the CTA's spc streams are split between the halves, half A takes the first ceil(spc/2): slot (half hh, row si)
// holds stream  cta_s0 + hh*ceil(spc/2) + si  — the rows of a half are CONSECUTIVE streams, so their conditioning rows are one
// contiguous piece of condA (engine.h, condA_frame_floats); in the half-A-only schedule (ONE, spc <= 16) slot (0, si) holds stream
// cta_s0 + si and half B is dead.  Dead slots shadow the batch's last stream: loads valid, stores masked.
template <bool ONE>
__device__ __forceinline__ int slot_stream(int cta_s0, int hh, int si, int spc, int n, bool &live)
{
    if (ONE) {
        const int g = cta_s0 + si;
        live = hh == 0 && si < spc && g < n;
        return min(g, n - 1);
    }
    const int na_ = (spc + 1) >> 1, c = hh * na_ + si, g = cta_s0 + c;
    live = si < (hh ? spc - na_ : na_) && g < n;
    return min(g, n - 1);
}
// the conditioning row (gate, stream) of a frame: condA_frame_floats (engine.h)
__device__ __forceinline__ const float *cond_row(const float *cond_f, int n, int gate, int sg) { return cond_f + ((size_t)gate * n + sg) * GIN_ROW; }

// Producer warps: ONE gate's input term for the 16 streams of a half,
//   G[si][k] = ((cond[s][k] + E_sig[a_s][k]) + E_pred[b_s][k]) + E_exc[c_s][k]        (nnet.c:484-491, left to right)
// Producer p serves tile rows si = p, p+NWP, ...: per stream the four row pointers are formed once and the NA columns
// of the gate are covered by NA/128 512-byte LDG.128 per row (4 L1 lines per request), i.e. 4*NA/128 (12 for the default
// 384 units) independent loads in flight per lane, then as many fp32 adds and NA/128 512-byte conflict-free STS.128 into
// the [16][NA + 8] tile.
template <bool ONE>
__device__ __forceinline__ void gather_half(float *__restrict__ G, const float *__restrict__ cond_f, int n, int cta_s0, int hh, int spc,
                                            const float *__restrict__ emb_sig, const float *__restrict__ emb_pred,
                                            const float *__restrict__ emb_exc, const int *__restrict__ idx_h,
                                            int gate, int p, int lane)
{
    const int col = gate * NA + lane * 4;
#pragma unroll 1
    for (int si = p; si < HALF; si += NWP) {
        bool live;
        const int sg = slot_stream<ONE>(cta_s0, hh, si, spc, n, live);
        if (!live) continue;                                     // dead slot: its tile row is never used for anything that is stored
        const float *c = cond_row(cond_f, n, gate, sg) + lane * 4;
        const float *e0 = emb_sig + idx_h[si] * (3 * NA) + col;
        const float *e1 = emb_pred + idx_h[HALF + si] * (3 * NA) + col;
        const float *e2 = emb_exc + idx_h[2 * HALF + si] * (3 * NA) + col;
        constexpr int NCH = NA / 128;
        float4 a[NCH], b[NCH], d[NCH], e[NCH];
#pragma unroll
        for (int j = 0; j < NCH; j++) { a[j] = ldg4(c + 128 * j); b[j] = ldg4(e0 + 128 * j); d[j] = ldg4(e1 + 128 * j); e[j] = ldg4(e2 + 128 * j); }
        float *g = G + si * GIN_ROW + lane * 4;
#pragma unroll
        for (int j = 0; j < NCH; j++) {
            float4 r;
            r.x = __fadd_rn(__fadd_rn(__fadd_rn(a[j].x, b[j].x), d[j].x), e[j].x);
            r.y = __fadd_rn(__fadd_rn(__fadd_rn(a[j].y, b[j].y), d[j].y), e[j].y);
            r.z = __fadd_rn(__fadd_rn(__fadd_rn(a[j].z, b[j].z), d[j].z), e[j].z);
            r.w = __fadd_rn(__fadd_rn(__fadd_rn(a[j].w, b[j].w), d[j].w), e[j].w);
            *reinterpret_cast<float4 *>(g + 128 * j) = r;
        }
    }
}

// ---- per-lane constants of a compute warp ----
struct ComputeCtx {
    uint32_t gid8;              // (lane >> 2) * 8
    int gid, t;
    int warp, lane;
    uint32_t tmA, tmB;                  // tensor-memory address (lane quarter | column) of the warp's first GRU_A / GRU_B quad
    uint32_t tmH;                       // ... of the lane's parked fp32 GRU_A state: [half][GPW][4] columns
    uint32_t qA0;                       // global index of the warp's first GRU_A quad (the directory holds global indices)
    uint32_t xs0;                       // shared address of state buffer 0
    const uint32_t *dirA, *dirB;
    const float *parA;                  // + 2t folded in
    const float *parB;
    const uint8_t *wBrec;
    RcpShared rcp;
    f32x2 one2;                         // {1.f, 1.f} read from shared memory (opaque to the compiler: oadd2, devmath.cuh)
    uint8_t *smem;
    int gcol[GPW];                      // neuron index of this lane's first neuron of each group: 8*g + 2t
    uint32_t xoff[GPW];                 // byte offset (in a state buffer) of this lane's two quantised neurons, stream gid of half 0 (half 1: ^ 64, stream gid+8: + 4)
};

// One GRU_A + GRU_B step of half H (16 streams).  k0 = index of the half-step's first tile fill (gate r; z and h follow).
// A half-step of the compute warps is three pieces:  gemv_rh<H>  |  activations<H> (ends by ARRIVING on MB_X[H])  |  grub<H> (WAITS on MB_X[H]).
// grub<H> runs right behind the activations, before the other half's gemv_rh, although it then waits on a CTA-wide barrier right after
// it was armed: the GRU_B state is what the half's sampler waits for, i.e. it is on the serial chain of a sample, while a warp that waits
// at the barrier only gives its issue slots to the others (-2.9 % per step against the other order, profiles/r02r_sweep.txt).

// GEMVs of the candidate and reset gates of half H (need only the previous state)
template <int H>
__device__ __forceinline__ void gemv_rh(const ComputeCtx &C, int (&Sh)[GPW][4], int (&Sg)[GPW][4], int cur)
{
    QuadPipe Q;
    Q.start(C.tmA + 2 * (C.dirA[2] - C.qA0), C.xs0 + cur * XS_BYTES, C.gid8 | (H << 6));
#pragma unroll
    for (int sl = 0; sl < GPW; sl++) {
        const uint32_t *dir = C.dirA + sl * 3 * 2;
#pragma unroll
        for (int i = 0; i < 4; i++) { Sh[sl][i] = 0; Sg[sl][i] = 0; }
        Q.list(Sg[sl], (int)dir[3]);                              // the warp's lists are stored r0 h0 r1 h1 ... (model.cu)
        Q.list(Sh[sl], (int)dir[5]);
    }
    Q.finish();
}

// gates r, z, candidate and state update of half H; Sh / Sg = GEMV sums of the candidate / reset gate
template <int H, bool FAST>
__device__ __forceinline__ void activations(const ComputeCtx &C, int (&Sh)[GPW][4], int (&Sg)[GPW][4], uint32_t k0, int cur)
{
    // The fp32 state of the lane's (stream, neuron) pairs of this half is only needed here: between its activations it is parked in
    // tensor memory (12-cycle private storage) instead of holding GPW*4 registers per half through the GEMV phases — at the 80-register
    // cap of a 768-thread CTA those registers were what spilled to local memory (through the LSU pipe this kernel is bound by).
    float h[GPW][4];
    tmem_wait_st();                                              // the state stored one sample ago has landed
#pragma unroll
    for (int sl = 0; sl < GPW; sl++) tmem_ld4f(h[sl], C.tmH + (H * GPW + sl) * 4);
    uint8_t *smem = C.smem;
    const int gid = C.gid, lane = C.lane;
    const RcpShared rcp = C.rcp;
    const int nxt = cur ^ 1;
    const uint32_t xs_cur = C.xs0 + cur * XS_BYTES, lc = C.gid8 | (H << 6);
    uint8_t *xs_nxt = smem + SM_XS + nxt * XS_BYTES;
    const uint32_t kr = k0, kz = k0 + 1, kh = k0 + 2;
    const float *tile_r = reinterpret_cast<const float *>(smem + SM_TILES + (kr & 3) * TILE_BYTES) + gid * GIN_ROW;
    const float *tile_z = reinterpret_cast<const float *>(smem + SM_TILES + (kz & 3) * TILE_BYTES) + gid * GIN_ROW;
    uint8_t *tile_hb = smem + SM_TILES + (kh & 3) * TILE_BYTES;
    const float *tile_h = reinterpret_cast<const float *>(tile_hb) + gid * GIN_ROW;
    const uint32_t mb_full = smem_u32(smem + MB_FULL), mb_empty = smem_u32(smem + MB_EMPTY);
    // ---- reset gate r (nnet.c:431-435) with the gathered input term; keep rec_h * r (nnet.c:436-440) ----
    mbar_wait(mb_full + 8 * (kr & 3), (kr >> 2) & 1);
#pragma unroll
    for (int sl = 0; sl < GPW; sl++) tmem_wait_ld4f(h[sl]);
#pragma unroll
    for (int sl = 0; sl < GPW; sl++) {
        const float *par = C.parA + sl * 3 * 16;
        const float2 br = *reinterpret_cast<const float2 *>(par + 16), dr = *reinterpret_cast<const float2 *>(par + 24);
        const float2 bh = *reinterpret_cast<const float2 *>(par + 32), dh = *reinterpret_cast<const float2 *>(par + 40);
        const float bri[2] = {br.x, br.y}, dri[2] = {dr.x, dr.y}, bhi[2] = {bh.x, bh.y}, dhi[2] = {dh.x, dh.y};
#pragma unroll
        for (int jj = 0; jj < 2; jj++) {
            const float2 gv = *reinterpret_cast<const float2 *>(tile_r + 8 * jj * GIN_ROW + C.gcol[sl]);
            const float gin[2] = {gv.x, gv.y};
            if constexpr (FAST) {
                int a[2], ah[2];
                {   // both neurons of the lane at a time; every mul -> add of the reference goes through oadd2
                    const f32x2 hv2 = pk2(h[sl][2 * jj], h[sl][2 * jj + 1]), ONE = C.one2;
                    float a0, a1, b0, b1;
                    upk2(oadd2(mul2(add2(oadd2(mul2(pk2(dr.x, dr.y), hv2), ONE, pk2(br.x, br.y)), pk2(gv.x, gv.y)), k2(LPCNET_SCALE)), ONE, k2(LPCNET_CVT_MAGIC)), a0, a1);
                    upk2(oadd2(mul2(oadd2(mul2(pk2(dh.x, dh.y), hv2), ONE, pk2(bh.x, bh.y)), k2(LPCNET_SCALE)), ONE, k2(LPCNET_CVT_MAGIC)), b0, b1);
                    a[0] = __float_as_int(a0) + Sg[sl][2 * jj]; a[1] = __float_as_int(a1) + Sg[sl][2 * jj + 1];
                    ah[0] = __float_as_int(b0) + Sh[sl][2 * jj]; ah[1] = __float_as_int(b1) + Sh[sl][2 * jj + 1];
                }
                f32x2 num, den;
                rational2(acc_finish2(a[0], a[1]), LPCNET_SIGMOID_COEF, num, den);
                float n0, n1, d0, d1, rh0, rh1;
                upk2(num, n0, n1); upk2(den, d0, d1);
                const float r0 = fmaxf(0.f, fminf(1.f, __fmaf_rn(n0, rcp_emul(d0, rcp), 0.5f)));
                const float r1 = fmaxf(0.f, fminf(1.f, __fmaf_rn(n1, rcp_emul(d1, rcp), 0.5f)));
                upk2(mul2(acc_finish2(ah[0], ah[1]), pk2(r0, r1)), rh0, rh1);
                Sh[sl][2 * jj] = __float_as_int(rh0);
                Sh[sl][2 * jj + 1] = __float_as_int(rh1);
            } else {
#pragma unroll
                for (int i = 0; i < 2; i++) {
                    const float hv = h[sl][2 * jj + i];
                    const int acc = acc_init_t<FAST>(__fadd_rn(__fadd_rn(bri[i], __fmul_rn(dri[i], hv)), gin[i])) + Sg[sl][2 * jj + i];
                    const float r = sigmoid_approx(acc_finish_t<FAST>(acc), rcp);
                    const int acch = acc_init_t<FAST>(__fadd_rn(bhi[i], __fmul_rn(dhi[i], hv))) + Sh[sl][2 * jj + i];
                    Sh[sl][2 * jj + i] = __float_as_int(__fmul_rn(acc_finish_t<FAST>(acch), r));
                }
            }
        }
    }
    warp_arrive(mb_empty + 8 * (kr & 3), lane);                  // gate-r tile consumed
    // ---- update gate z (nnet.c:426-430) ----
    {
        QuadPipe Q;
        Q.start(C.tmA + 2 * (C.dirA[0] - C.qA0), xs_cur, lc);
#pragma unroll
        for (int sl = 0; sl < GPW; sl++) {
#pragma unroll
            for (int i = 0; i < 4; i++) Sg[sl][i] = 0;
            Q.list(Sg[sl], (int)C.dirA[sl * 3 * 2 + 1]);          // z0 z1 z2 are contiguous too
        }
        Q.finish();
    }
    mbar_wait(mb_full + 8 * (kz & 3), (kz >> 2) & 1);
#pragma unroll
    for (int sl = 0; sl < GPW; sl++) {
        const float *par = C.parA + sl * 3 * 16;
        const float2 bz = *reinterpret_cast<const float2 *>(par), dz = *reinterpret_cast<const float2 *>(par + 8);
        const float bzi[2] = {bz.x, bz.y}, dzi[2] = {dz.x, dz.y};
#pragma unroll
        for (int jj = 0; jj < 2; jj++) {
            const float2 gv = *reinterpret_cast<const float2 *>(tile_z + 8 * jj * GIN_ROW + C.gcol[sl]);
            const float gin[2] = {gv.x, gv.y};
            if constexpr (FAST) {
                int a[2];
                {
                    const f32x2 ONE = C.one2;
                    float a0, a1;
                    upk2(oadd2(mul2(add2(oadd2(mul2(pk2(dz.x, dz.y), pk2(h[sl][2 * jj], h[sl][2 * jj + 1])), ONE, pk2(bz.x, bz.y)), pk2(gv.x, gv.y)), k2(LPCNET_SCALE)), ONE, k2(LPCNET_CVT_MAGIC)), a0, a1);
                    a[0] = __float_as_int(a0) + Sg[sl][2 * jj]; a[1] = __float_as_int(a1) + Sg[sl][2 * jj + 1];
                }
                f32x2 num, den;
                rational2(acc_finish2(a[0], a[1]), LPCNET_SIGMOID_COEF, num, den);
                float n0, n1, d0, d1;
                upk2(num, n0, n1); upk2(den, d0, d1);
                Sg[sl][2 * jj] = __float_as_int(fmaxf(0.f, fminf(1.f, __fmaf_rn(n0, rcp_emul(d0, rcp), 0.5f))));
                Sg[sl][2 * jj + 1] = __float_as_int(fmaxf(0.f, fminf(1.f, __fmaf_rn(n1, rcp_emul(d1, rcp), 0.5f))));
            } else {
#pragma unroll
                for (int i = 0; i < 2; i++) {
                    const int acc = acc_init_t<FAST>(__fadd_rn(__fadd_rn(bzi[i], __fmul_rn(dzi[i], h[sl][2 * jj + i])), gin[i])) + Sg[sl][2 * jj + i];
                    Sg[sl][2 * jj + i] = __float_as_int(sigmoid_approx(acc_finish_t<FAST>(acc), rcp));
                }
            }
        }
    }
    warp_arrive(mb_empty + 8 * (kz & 3), lane);                  // gate-z tile consumed
    // ---- h~ = tanh(rec_h*r + gin_h) (nnet.c:443-445), h <- z*h + (1-z)*h~ (nnet.c:446-447), new quantised state ----
    mbar_wait(mb_full + 8 * (kh & 3), (kh >> 2) & 1);
#pragma unroll
    for (int sl = 0; sl < GPW; sl++)
#pragma unroll
        for (int jj = 0; jj < 2; jj++) {
            const float2 gv = *reinterpret_cast<const float2 *>(tile_h + 8 * jj * GIN_ROW + C.gcol[sl]);
            const float gin[2] = {gv.x, gv.y};
            uint32_t q[2];
            if constexpr (FAST) {
                f32x2 num, den;
                rational2(add2(pk2(__int_as_float(Sh[sl][2 * jj]), __int_as_float(Sh[sl][2 * jj + 1])), pk2(gin[0], gin[1])), LPCNET_TANH_COEF, num, den);
                float d0, d1, t0, t1;
                upk2(den, d0, d1);
                upk2(mul2(num, pk2(rcp_emul(d0, rcp), rcp_emul(d1, rcp))), t0, t1);
                const float hh[2] = {fmaxf(-1.f, fminf(1.f, t0)), fmaxf(-1.f, fminf(1.f, t1))};
                float hn[2];
                {
                    const f32x2 z2 = pk2(__int_as_float(Sg[sl][2 * jj]), __int_as_float(Sg[sl][2 * jj + 1]));
                    upk2(oadd2(mul2(z2, pk2(h[sl][2 * jj], h[sl][2 * jj + 1])), C.one2, mul2(one_minus2(z2), pk2(hh[0], hh[1]))), hn[0], hn[1]);
                    h[sl][2 * jj] = hn[0]; h[sl][2 * jj + 1] = hn[1];
                }
                // quantised bytes in the low bytes of the biased patterns: fma -> add, safe to pack
                float q0, q1;
                upk2(add2(fma2(pk2(hn[0], hn[1]), k2(127.f), k2(127.f)), k2(LPCNET_CVT_MAGIC)), q0, q1);
                q[0] = __float_as_uint(q0); q[1] = __float_as_uint(q1);
            } else {
#pragma unroll
                for (int i = 0; i < 2; i++) {
                    const float hh = tanh_approx(__fadd_rn(__int_as_float(Sh[sl][2 * jj + i]), gin[i]), rcp);
                    const float z = __int_as_float(Sg[sl][2 * jj + i]);
                    const float hn = __fadd_rn(__fmul_rn(z, h[sl][2 * jj + i]), __fmul_rn(__fsub_rn(1.f, z), hh));
                    h[sl][2 * jj + i] = hn;
                    q[i] = quant_u8_t<FAST>(hn);
                }
            }
            // other buffer: readers of the old state are unaffected
            *reinterpret_cast<uint16_t *>(xs_nxt + (C.xoff[sl] ^ (H << 6)) + 4 * jj) = (uint16_t)__byte_perm(q[0], q[1], 0x0040);
        }
#pragma unroll
    for (int sl = 0; sl < GPW; sl++) tmem_st4f(C.tmH + (H * GPW + sl) * 4, h[sl]);
    warp_arrive(smem_u32(smem + MB_X) + 8 * H, lane);            // this warp's part of the new quantised state is written, candidate-gate tile consumed
}

// GRU_B of half H for the half-step whose activations were issued before; par = parity of that sample
template <int H, bool FAST>
__device__ __forceinline__ void grub(const ComputeCtx &C, const SampleParams &P, float &hb, uint32_t k0, int cur, int f, int s_fin, uint32_t par, int trstep = -1)
{
    uint8_t *smem = C.smem;
    const int gid = C.gid, t = C.t, lane = C.lane, warp = C.warp;
    const RcpShared rcp = C.rcp;
    const int nxt = cur ^ 1;
    const uint32_t lc = C.gid8 | (H << 6);
    const uint32_t kh = k0 + 2;
    uint8_t *tile_hb = smem + SM_TILES + (kh & 3) * TILE_BYTES;
    const uint32_t mb_empty = smem_u32(smem + MB_EMPTY);
    mbar_wait(smem_u32(smem + MB_X) + 8 * H, par);               // new quantised GRU_A state complete; candidate-gate tile dead: GRU_B scratch may use it
    TRACEC(P, trstep, 27, warp == 0 ? lane : 1);
    // ---------------- GRU_B input GEMV (48 x 384 int8, dense): warp = (row group, K part) ----------------
    int *accB = reinterpret_cast<int *>(tile_hb + T_ACCB);
    float *hBs = reinterpret_cast<float *>(tile_hb + T_HBS);
    if (warp < NWB) {
        int acc[4] = {0, 0, 0, 0};
        const uint32_t nq = C.dirB[warp * 2 + 1];
        QuadPipe Q;
        Q.start(C.tmB, C.xs0 + nxt * XS_BYTES, lc);
        Q.list(acc, (int)nq);
        Q.finish();
        const int rgp = warp / KPARTS, part = warp % KPARTS;
        int *dst = accB + (part * 3 * NB + rgp * 8 + 2 * t) * ACCB_ROW + gid;
        dst[0] = acc[0]; dst[ACCB_ROW] = acc[1]; dst[8] = acc[2]; dst[ACCB_ROW + 8] = acc[3];
        warp_arrive(smem_u32(smem + MB_ACCB) + 8 * H, lane);
    }
    TRACEC(P, trstep, 28, warp == 0 ? lane : 1);
    // ---------------- GRU_B finish (nnet.c:346-371): warps FIN0 .. FIN0+NFIN-1, lane = (neuron parity, stream of the half) ----------------
    uint32_t *xb = reinterpret_cast<uint32_t *>(smem + SM_XB) + H * (2 * 4 * HALF);
    if (warp >= FIN0 && warp < FIN0 + NFIN) {
        const int jb = 2 * (warp - FIN0) + (lane >> 4), si = lane & 15;
        const float *condBp = P.condB + ((size_t)f * P.n_streams + s_fin) * (3 * NB);
        const float cbz = __ldg(condBp + jb), cbr = __ldg(condBp + NB + jb), cbh = __ldg(condBp + 2 * NB + jb);
        const uint32_t *xbc = xb + cur * 4 * HALF;
        // recurrent side first: it only needs the previous GRU_B state, so it runs while other warps finish their partial sums
        int rz = acc_init(C.parB[3 * NB + jb]), rr = acc_init(C.parB[4 * NB + jb]), rh = acc_init(C.parB[5 * NB + jb]);
#pragma unroll
        for (int k = 0; k < 4; k++) {    // W_rec layout [out/8][in/4][8][4] (dump_lpcnet.py:58-59)
            const uint32_t xw = xbc[k * HALF + si];
            rz = dp4a_us(xw, *reinterpret_cast<const int *>(C.wBrec + (((jb >> 3) * 4 + k) * 8 + (jb & 7)) * 4), rz);
            rr = dp4a_us(xw, *reinterpret_cast<const int *>(C.wBrec + ((((NB + jb) >> 3) * 4 + k) * 8 + ((NB + jb) & 7)) * 4), rr);
            rh = dp4a_us(xw, *reinterpret_cast<const int *>(C.wBrec + ((((2 * NB + jb) >> 3) * 4 + k) * 8 + ((2 * NB + jb) & 7)) * 4), rh);
        }
        mbar_wait(smem_u32(smem + MB_ACCB) + 8 * H, par);      // all K-part partial sums are in accB
        TRACEC(P, trstep, 29, warp == 0 ? lane : 1);
        int az = acc_init(__fadd_rn(C.parB[jb], cbz)), ar = acc_init(__fadd_rn(C.parB[NB + jb], cbr)), ah = acc_init(__fadd_rn(C.parB[2 * NB + jb], cbh));
#pragma unroll
        for (int kp = 0; kp < KPARTS; kp++) {
            az += accB[(kp * 3 * NB + jb) * ACCB_ROW + si];
            ar += accB[(kp * 3 * NB + NB + jb) * ACCB_ROW + si];
            ah += accB[(kp * 3 * NB + 2 * NB + jb) * ACCB_ROW + si];
        }
        const float zz = sigmoid_approx(__fadd_rn(acc_finish(az), acc_finish(rz)), rcp);
        const float rrr = sigmoid_approx(__fadd_rn(acc_finish(ar), acc_finish(rr)), rcp);
        const float hh = tanh_approx(__fadd_rn(acc_finish(ah), __fmul_rn(acc_finish(rh), rrr)), rcp);
        hb = __fadd_rn(__fmul_rn(zz, hb), __fmul_rn(__fsub_rn(1.f, zz), hh));
        hBs[jb * HALF + si] = hb;
        reinterpret_cast<uint8_t *>(xb + nxt * 4 * HALF)[((jb >> 2) * HALF + si) * 4 + (jb & 3)] = (uint8_t)quant_u8(hb);
        __threadfence_block();
        bar_arrive(BAR_HB + H, CNT_HB);                          // GRU_B state of this sample is in hBs
    }
    warp_arrive(mb_empty + 8 * (kh & 3), lane);                  // (its refill is additionally gated by the half's next indices)
}

}  // namespace

template <bool FAST, bool ONE>
__global__ void __launch_bounds__(SAMPLE_THREADS, 1) lpcnet_sample_kernel(const __grid_constant__ SampleParams P)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const SmemLayout &L = P.L;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n = P.n_streams;
    constexpr bool one = ONE;                                     // spc <= 16: half-A-only schedule (SampleParams::one_half)
    const int spc = P.spc;
    const int cta_s0 = blockIdx.x * spc;
    const int spf = P.spf;

    // ---- mbarriers; stage the constant image with TMA bulk copies ----
    const uint32_t bar = smem_u32(smem + MB_IMAGE);
    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        for (int b = 0; b < NTILE; b++) { mbar_init(smem_u32(smem + MB_FULL) + 8 * b, NWP * ARRIVALS_PER_WARP); mbar_init(smem_u32(smem + MB_EMPTY) + 8 * b, NWC * ARRIVALS_PER_WARP); }
        for (int hh = 0; hh < 2; hh++) { mbar_init(smem_u32(smem + MB_IDX) + 8 * hh, ARRIVALS_PER_WARP); mbar_init(smem_u32(smem + MB_X) + 8 * hh, NWC * ARRIVALS_PER_WARP); mbar_init(smem_u32(smem + MB_ACCB) + 8 * hh, NWB * ARRIVALS_PER_WARP); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (threadIdx.x == 32) *reinterpret_cast<float *>(smem + SM_MBAR + 124) = 1.f;     // ComputeCtx::one2 (last free word of the mbarrier block)
    // tensor memory for the GEMV operands: warp 0 allocates all 512 columns (one CTA per SM), the base address travels through shared memory
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + SM_MBAR + 120);
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (threadIdx.x == 0) {
        mbar_expect_tx(bar, L.image_bytes);
        const uint32_t CH = 16384;
        for (uint32_t o = 0; o < L.image_bytes; o += CH) {
            const uint32_t nbytes = min(CH, L.image_bytes - o);
            bulk_g2s(smem_u32(smem + SM_IMAGE + o), P.image + o, nbytes, bar);
        }
    }
    const RcpShared rcp = {smem_u32(smem + SM_IMAGE + IM_RCP)};
    if (threadIdx.x == 0 && (rcp.addr & 0x1FFFu) != 0) __trap();      // the table-address trick of rcp_emul needs the 8 KB alignment
    int *idx_s = reinterpret_cast<int *>(smem + SM_IDX);

    if (warp < NWC) {
        // =====================================================  compute warps  =====================================================
        mbar_wait(bar, 0);
        ComputeCtx C;
        C.gid = lane >> 2; C.t = lane & 3; C.gid8 = C.gid * 8; C.warp = warp; C.lane = lane; C.smem = smem; C.rcp = rcp;
        { const float one = *reinterpret_cast<const volatile float *>(smem + SM_MBAR + 124); C.one2 = pk2(one, one); }
        const uint32_t *grpA = reinterpret_cast<const uint32_t *>(smem + SM_IMAGE + IM_GRPA);
        C.dirA = reinterpret_cast<const uint32_t *>(smem + SM_IMAGE + IM_DIRA) + warp * GPW * 3 * 2;
        C.parA = reinterpret_cast<const float *>(smem + SM_IMAGE + IM_PARA) + warp * GPW * 3 * 16 + 2 * C.t;
        C.dirB = reinterpret_cast<const uint32_t *>(smem + SM_IMAGE + IM_DIRB);
        const uint32_t tbase_w = *tmem_slot + ((uint32_t)(32 * (warp & 3)) << 16) + (uint32_t)(warp >> 2) * TMEM_COLS_PER_WARP;
        {   // this warp's quads: shared-memory image -> tensor memory, {weights word of the lane, meta of the lane's slot} per quad, GRU_A stream
            // (r0 h0 r1 h1 ... z0 z1 ...: contiguous in the image), then the warp's GRU_B stream, then QUAD_TAIL copies of the first quad
            const uint32_t tbase = tbase_w;
            const uint32_t zl = ((GPW - 1) * 3 + 0) * 2;                                   // directory entry of the warp's last list (z of its last slot)
            C.qA0 = C.dirA[2];
            const uint32_t nqa = C.dirA[zl] + C.dirA[zl + 1] - C.qA0;
            const uint32_t wsrc = smem_u32(smem + L.wA) + lane * 4, msrc = smem_u32(smem + L.metaA) + C.t * 2;
            for (uint32_t q = 0; q < nqa; q++) tmem_st2(tbase + 2 * q, lds32(wsrc + (C.qA0 + q) * QUAD_BYTES), lds16(msrc + (C.qA0 + q) * QUAD_META_BYTES));
            C.tmA = tbase; C.tmB = tbase + 2 * nqa;
            uint32_t tail = C.tmB;
            if (warp < NWB) {
                const uint32_t q0 = C.dirB[warp * 2], nqb = C.dirB[warp * 2 + 1];
                const uint32_t wsb = smem_u32(smem + L.wB) + lane * 4, msb = smem_u32(smem + L.metaB) + C.t * 2;
                for (uint32_t q = 0; q < nqb; q++) tmem_st2(C.tmB + 2 * q, lds32(wsb + (q0 + q) * QUAD_BYTES), lds16(msb + (q0 + q) * QUAD_META_BYTES));
                tail += 2 * nqb;
            }
            for (uint32_t q = 0; q < QUAD_TAIL; q++) tmem_st2(tail + 2 * q, lds32(wsrc + C.qA0 * QUAD_BYTES), lds16(msrc + C.qA0 * QUAD_META_BYTES));
            tmem_wait_st();
        }
        C.parB = reinterpret_cast<const float *>(smem + SM_IMAGE + IM_PARB);
        C.wBrec = smem + SM_IMAGE + IM_WBREC;
        C.xs0 = smem_u32(smem + SM_XS);
        // the stream slots of this lane: half j>>1, row gid + 8*(j&1)
        int sj[4]; bool livej[4];
#pragma unroll
        for (int j = 0; j < 4; j++) sj[j] = slot_stream<ONE>(cta_s0, j >> 1, C.gid + 8 * (j & 1), spc, n, livej[j]);

        // restored fp32 state: [half][group][stream jj][neuron i] at 2jj+i -> the lane's tensor-memory columns, quantised copy -> xs buffer 0
        C.tmH = tbase_w + TMEM_H_COL;
#pragma unroll
        for (int sl = 0; sl < GPW; sl++) {
            const int g = (int)grpA[warp * GPW + sl];
            C.gcol[sl] = 8 * g + 2 * C.t;
            C.xoff[sl] = xs_offset(2 * g + (C.t >> 1), C.gid) + (C.t & 1) * 2;
#pragma unroll
            for (int hh2 = 0; hh2 < 2; hh2++) {
                float hv[4];
#pragma unroll
                for (int jj = 0; jj < 2; jj++)
#pragma unroll
                    for (int i = 0; i < 2; i++) hv[2 * jj + i] = P.hA[(size_t)(C.gcol[sl] + i) * n + sj[2 * hh2 + jj]];
                tmem_st4f(C.tmH + (hh2 * GPW + sl) * 4, hv);
#pragma unroll
                for (int jj = 0; jj < 2; jj++)
                    *reinterpret_cast<uint16_t *>(smem + SM_XS + (C.xoff[sl] ^ (hh2 << 6)) + 4 * jj) = (uint16_t)(quant_u8(hv[2 * jj]) | (quant_u8(hv[2 * jj + 1]) << 8));
            }
        }
        // GRU_B neuron finished by this lane (warps FIN0 .. FIN0+NFIN-1): neuron 2*(warp - FIN0) + (lane >> 4), stream lane & 15 of each half
        const bool fin_warp = warp >= FIN0 && warp < FIN0 + NFIN;
        const int jb_fin = min(max(2 * (warp - FIN0), 0) + (lane >> 4), NB - 1);
        int s_fin[2]; bool live_fin[2];
        float hb[2];
#pragma unroll
        for (int hh = 0; hh < 2; hh++) {
            s_fin[hh] = slot_stream<ONE>(cta_s0, hh, lane & 15, spc, n, live_fin[hh]);
            hb[hh] = P.hB[(size_t)jb_fin * n + s_fin[hh]];
        }
        // quantised copy of the restored GRU_B state: xb[half][0] <- q(hB)
        if (fin_warp) {
#pragma unroll
            for (int hh = 0; hh < 2; hh++)
                reinterpret_cast<uint8_t *>(smem + SM_XB)[(((hh * 2 + 0) * 4 + (jb_fin >> 2)) * HALF + (lane & 15)) * 4 + (jb_fin & 3)] = (uint8_t)quant_u8(hb[hh]);
        }
        bar_sync(BAR_X, CNT_C);                                          // restored quantised state visible to all compute warps

        uint32_t k = 0; int step = 0, f_prev = 0;
        if constexpr (ONE) {
            // small batch: half A alone, strictly in program order (nothing to overlap with)
            for (int f = 0; f < P.nframes; f++)
                for (int t_ = 0; t_ < spf; t_++, step++, k += 3) {
                    int Sh[GPW][4], Sg[GPW][4];
                    gemv_rh<0>(C, Sh, Sg, step & 1);
                    activations<0, FAST>(C, Sh, Sg, k, step & 1);
                    grub<0, FAST>(C, P, hb[0], k, step & 1, f, s_fin[0], step & 1, step);
                }
        } else {
        for (int f = 0; f < P.nframes; f++)
            for (int t_ = 0; t_ < spf; t_++, step++, k += 6) {
                int Sh[GPW][4], Sg[GPW][4];                              // candidate-gate sums (later rec_h * r) / r-gate, then z-gate sums (later z)
                const int tl = warp == 0 ? lane : 1; (void)tl;    // (lane selector of the TRACE stamps)
                TRACEC(P, step, 0, tl); TRACEW(P, step, 0);
                if (step > 0) grub<1, FAST>(C, P, hb[1], k - 3, (step - 1) & 1, f_prev, s_fin[1], (step - 1) & 1);
                TRACEC(P, step, 1, tl); TRACEW(P, step, 1);
                gemv_rh<0>(C, Sh, Sg, step & 1);
                TRACEC(P, step, 2, tl); TRACEW(P, step, 2);       // = HB of half B (previous sample) signalled
                mbar_wait(smem_u32(smem + MB_FULL) + 8 * (k & 3), (k >> 2) & 1);
                TRACEC(P, step, 3, tl); TRACEW(P, step, 3);       // r tile of half A present
                activations<0, FAST>(C, Sh, Sg, k, step & 1);
                TRACEC(P, step, 4, tl); TRACEW(P, step, 4);
                grub<0, FAST>(C, P, hb[0], k, step & 1, f, s_fin[0], step & 1, step);
                TRACEC(P, step, 5, tl); TRACEW(P, step, 5);
                gemv_rh<1>(C, Sh, Sg, step & 1);
                TRACEC(P, step, 6, tl); TRACEW(P, step, 6);       // = HB of half A signalled
                mbar_wait(smem_u32(smem + MB_FULL) + 8 * ((k + 3) & 3), ((k + 3) >> 2) & 1);
                TRACEC(P, step, 7, tl); TRACEW(P, step, 7);       // r tile of half B present
                activations<1, FAST>(C, Sh, Sg, k + 3, step & 1);
                TRACEC(P, step, 8, tl); TRACEW(P, step, 8);
                f_prev = f;
            }
        if (step > 0) grub<1, FAST>(C, P, hb[1], k - 3, (step - 1) & 1, f_prev, s_fin[1], (step - 1) & 1);
        }
        // ---- save the recurrent state ----
        tmem_wait_st();
#pragma unroll
        for (int sl = 0; sl < GPW; sl++)
#pragma unroll
            for (int hh2 = 0; hh2 < 2; hh2++) {
                float hv[4];
                tmem_ld4f(hv, C.tmH + (hh2 * GPW + sl) * 4);
                tmem_wait_ld4f(hv);
#pragma unroll
                for (int jj = 0; jj < 2; jj++)
                    if (livej[2 * hh2 + jj]) {
                        P.hA[(size_t)C.gcol[sl] * n + sj[2 * hh2 + jj]] = hv[2 * jj];
                        P.hA[(size_t)(C.gcol[sl] + 1) * n + sj[2 * hh2 + jj]] = hv[2 * jj + 1];
                    }
            }
        if (fin_warp) {
#pragma unroll
            for (int hh = 0; hh < 2; hh++) if (live_fin[hh]) P.hB[(size_t)jb_fin * n + s_fin[hh]] = hb[hh];
        }
        // every compute warp is done with its tensor-memory columns: warp 0 returns the allocation
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        bar_sync(BAR_X, CNT_C);
        if (warp == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(*tmem_slot), "n"(TMEM_COLS) : "memory");
        }
    } else if (warp < NWC + NWP) {
        // =====================================================  producer warps  =====================================================
        const int p = warp - NWC;
        const uint32_t mb_full = smem_u32(smem + MB_FULL), mb_empty = smem_u32(smem + MB_EMPTY), mb_idx = smem_u32(smem + MB_IDX);
        uint32_t k = 0, it = 0;
        for (int f = 0; f < P.nframes; f++) {
            const float *condA_f = P.condA + (size_t)f * n * (3 * GIN_ROW);
            for (int t_ = 0; t_ < spf; t_++, it++)
#pragma unroll 1
                for (int hh = 0; hh < (one ? 1 : 2); hh++) {
                    mbar_wait(mb_idx + 8 * hh, it & 1);                  // indices of this sample of the half are in idx_s
                    TRACE(P, (int)it, 10 + 4 * hh, p == 0 ? lane : 1);
#pragma unroll 1
                    for (int gi = 0; gi < 3; gi++, k++) {
                        const int gate = gi == 0 ? 1 : (gi == 1 ? 0 : 2);    // fill order r, z, h
                        mbar_wait(mb_empty + 8 * (k & 3), ((k >> 2) & 1) ^ 1);  // previous contents of the tile consumed
                        gather_half<ONE>(reinterpret_cast<float *>(smem + SM_TILES + (k & 3) * TILE_BYTES), condA_f, n, cta_s0, hh, spc,
                                    P.emb_sig, P.emb_pred, P.emb_exc, idx_s + hh * 3 * HALF, gate, p, lane);
                        warp_arrive(mb_full + 8 * (k & 3), lane);
                        TRACE(P, (int)it, 11 + 4 * hh + gi, p == 0 ? lane : 1);
                    }
                }
        }
    } else {
        // =====================================================  sampler warps  =====================================================
        // warp NWC+NWP+hh serves half hh.  Lane = (channel, stream): both lanes of a stream run the same serial code on the
        // same state (so they take the same decisions); they differ only in the dual_fc channel they evaluate, and the
        // channel-1 lane issues no stores.
        mbar_wait(bar, 0);
        const int hh = warp - NWC - NWP, ch = lane >> 4, si = lane & 15;
        if (one && hh) return;                                           // small batch: half B is not stepped
        bool live;
        const int s = slot_stream<ONE>(cta_s0, hh, si, spc, n, live);
        live = live && ch == 0;
        const float *logit = reinterpret_cast<const float *>(smem + SM_IMAGE + IM_LOGIT);
        const float *u2l = reinterpret_cast<const float *>(smem + SM_IMAGE + IM_U2L);
        const float *fcw = reinterpret_cast<const float *>(smem + SM_IMAGE + IM_FCW) + ch * NB;
        const float *fcw_g = P.fcw + ch * NB;
        const int fcw_nodes = *reinterpret_cast<const int *>(smem + SM_IMAGE + IM_FCWN);    // dual_fc rows kept in shared memory (64 unless the model needed the room)
        const uint32_t mb_idx = smem_u32(smem + MB_IDX) + 8 * hh;
        int *idx_h = idx_s + hh * 3 * HALF;

        float ls[LPC_ORDER], lpc[LPC_ORDER];
#pragma unroll
        for (int j = 0; j < LPC_ORDER; j++) ls[j] = P.last_sig[(size_t)j * n + s];
        float deemph = P.deemph[s];
        int last_exc = P.last_exc[s];
        Kiss99 rng;
        rng.z = P.rng[s]; rng.w = P.rng[(size_t)n + s]; rng.jsr = P.rng[2 * (size_t)n + s]; rng.jcong = P.rng[3 * (size_t)n + s];
        short *pcm_out = P.pcm + (size_t)s * P.pcm_stream_stride;
        float pred = 0.f;
        const int preload = P.fast_cvt >> 8;                             // teacher-forced samples at the start of the call's first frame (lpcnet.c:256-259)

        // publish the conditioning indices of the half's next sample (lpcnet.c:251-254)
        auto publish = [&]() {
            pred = 0.f;
#pragma unroll
            for (int j = 0; j < LPC_ORDER; j++) pred = __fsub_rn(pred, __fmul_rn(ls[j], lpc[j]));
            if (ch == 0) {
                idx_h[si] = lin2ulaw(ls[0]);
                idx_h[HALF + si] = lin2ulaw(pred);
                idx_h[2 * HALF + si] = last_exc;
            }
            warp_arrive(mb_idx, lane);
        };
        auto load_lpc = [&](int f) {   // frame f uses the LPC computed from the features of frame f-2 (lpcnet.c:110-112), weighted by gamma^i (freq.c:299-308)
            const float *lp = P.lpc_raw + ((size_t)f * n + s) * LPC_ORDER;
            const float4 a = ldg4(lp), b = ldg4(lp + 4), c = ldg4(lp + 8), d = ldg4(lp + 12);
            const float raw[16] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w, d.x, d.y, d.z, d.w};
#pragma unroll
            for (int j = 0; j < LPC_ORDER; j++) lpc[j] = __fmul_rn(raw[j], __ldg(&P.gamma_pow[j]));
        };
        load_lpc(0);
        publish();
        uint32_t k = 0;
        for (int f = 0; f < P.nframes; f++) {
            for (int t_ = 0; t_ < spf; t_++, k += one ? 3 : 6) {
                const bool last_t = t_ == spf - 1, last = last_t && f == P.nframes - 1;
                // thresholds (nnet.c:178-184): two RNG words -> 8 logits; does not depend on the network
                float thr[8];
                {
                    uint32_t r0 = kiss99_rand(rng), r1 = kiss99_rand(rng);
                    thr[0] = logit[r0 & 0xFF]; thr[1] = logit[(r0 >> 8) & 0xFF]; thr[2] = logit[(r0 >> 16) & 0xFF]; thr[3] = logit[r0 >> 24];
                    thr[4] = logit[r1 & 0xFF]; thr[5] = logit[(r1 >> 8) & 0xFF]; thr[6] = logit[(r1 >> 16) & 0xFF]; thr[7] = logit[r1 >> 24];
                }
                bar_sync(BAR_HB + hh, CNT_HB);                           // GRU_B state of the half is in hBs (inside the half's candidate-gate tile)
                TRACE(P, (int)(k / 6), 20 + 4 * hh, lane);
                const float *hBs = reinterpret_cast<const float *>(smem + SM_TILES + ((k + 3 * hh + 2) & 3) * TILE_BYTES + T_HBS);
                float hbv[NB];
#pragma unroll
                for (int j = 0; j < NB; j++) hbv[j] = hBs[j * HALF + si];
                int val = 0;
#pragma unroll
                for (int b = 0; b < 8; b++) {                            // sample_mdense, nnet.c:186-211
                    const int i = (1 << b) | val;
                    // this lane's channel: a sequential 16-term chain
                    float w16[16], sum, fac;
                    if (b < 3 || (b < 6 && i < fcw_nodes)) {             // upper levels: rows in shared memory (8 nodes always, up to 64: model.cu)
                        const float *wr = fcw + i * FCW_ROW;
                        const float4 a0 = *reinterpret_cast<const float4 *>(wr), a1 = *reinterpret_cast<const float4 *>(wr + 4);
                        const float4 a2 = *reinterpret_cast<const float4 *>(wr + 8), a3 = *reinterpret_cast<const float4 *>(wr + 12);
                        w16[0] = a0.x; w16[1] = a0.y; w16[2] = a0.z; w16[3] = a0.w; w16[4] = a1.x; w16[5] = a1.y; w16[6] = a1.z; w16[7] = a1.w;
                        w16[8] = a2.x; w16[9] = a2.y; w16[10] = a2.z; w16[11] = a2.w; w16[12] = a3.x; w16[13] = a3.y; w16[14] = a3.z; w16[15] = a3.w;
                        sum = wr[2 * NB - ch * NB + ch]; fac = wr[2 * NB - ch * NB + 2 + ch];
                    } else {                                             // lower levels: the row comes from global memory (L2/L1-resident)
                        const float *wr = fcw_g + i * FCW_ROW;
                        const float4 a0 = ldg4(wr), a1 = ldg4(wr + 4), a2 = ldg4(wr + 8), a3 = ldg4(wr + 12);
                        w16[0] = a0.x; w16[1] = a0.y; w16[2] = a0.z; w16[3] = a0.w; w16[4] = a1.x; w16[5] = a1.y; w16[6] = a1.z; w16[7] = a1.w;
                        w16[8] = a2.x; w16[9] = a2.y; w16[10] = a2.z; w16[11] = a2.w; w16[12] = a3.x; w16[13] = a3.y; w16[14] = a3.z; w16[15] = a3.w;
                        sum = __ldg(wr + 2 * NB - ch * NB + ch); fac = __ldg(wr + 2 * NB - ch * NB + 2 + ch);
                    }
#pragma unroll
                    for (int j = 0; j < NB; j++) sum = __fadd_rn(sum, __fmul_rn(w16[j], hbv[j]));
                    const float mine = __fmul_rn(fac, tanh_approx(sum, rcp));
                    const float other = __shfl_xor_sync(0xffffffffu, mine, 16);
                    const float tot = __fadd_rn(mine, other);            // channel 0 + channel 1 (commutative: both lanes get the same bits)
                    val = (val << 1) | (thr[b] < tot ? 1 : 0);
                }
                int exc = val;
                float pcm;
                const bool forced = f == 0 && t_ < preload;
                if (forced) {                                            // lpcnet.c:256-259: the network ran (state, RNG advanced) but the excitation
                    const float o = (float)pcm_out[t_];                  // is derived from the signal the caller supplied in the output buffer
                    pcm = __fsub_rn(o, __fmul_rn(0.85f, deemph));
                    exc = lin2ulaw(__fsub_rn(pcm, pred));
                } else pcm = __fadd_rn(pred, u2l[exc]);                  // lpcnet.c:260
#pragma unroll
                for (int j = LPC_ORDER - 1; j > 0; j--) ls[j] = ls[j - 1];
                ls[0] = pcm;
                last_exc = exc;
                pcm = __fadd_rn(pcm, __fmul_rn(0.85f, deemph));          // PREEMPH, lpcnet.c:265
                deemph = pcm;
                if (pcm < -32767) pcm = -32767;
                if (pcm > 32767) pcm = 32767;
                if (live && !forced) pcm_out[(size_t)f * spf + t_] = (short)__double2int_rd(0.5 + (double)pcm);   // (int)floor(.5 + pcm); lpcnet.c:269
                TRACE(P, (int)(k / 6), 21 + 4 * hh, lane);
                if (last_t && !last) load_lpc(f + 1);
                if (!last) publish();                                    // indices of the half's next sample
                TRACE(P, (int)(k / 6), 22 + 4 * hh, lane);
            }
        }
        if (live) {
#pragma unroll
            for (int j = 0; j < LPC_ORDER; j++) P.last_sig[(size_t)j * n + s] = ls[j];
            P.deemph[s] = deemph;
            P.last_exc[s] = last_exc;
            P.rng[s] = rng.z; P.rng[(size_t)n + s] = rng.w; P.rng[2 * (size_t)n + s] = rng.jsr; P.rng[3 * (size_t)n + s] = rng.jcong;
        }
    }
}

cudaError_t launch_sample_kernel(const SampleParams &p, cudaStream_t st)
{
    // per-device attribute; cheap enough to set on every launch (one launch covers >= 160 x n_streams samples)
    const bool one = p.one_half != 0;                             // (decided by the caller: spc <= 16, batch_api.cu)
    auto kern = (p.fast_cvt & 1) ? (one ? lpcnet_sample_kernel<true, true> : lpcnet_sample_kernel<true, false>)
                           : (one ? lpcnet_sample_kernel<false, true> : lpcnet_sample_kernel<false, false>);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return e;
    const int ctas = (p.n_streams + p.spc - 1) / p.spc;
    kern<<<ctas, SAMPLE_THREADS, p.L.total_bytes, st>>>(p);
    return cudaGetLastError();
}

}  // namespace LPCNET_KNS
}  // namespace lpcnet_b200
