// engine.h — internal structures shared by the host-side model loader and the sm_100a kernels.
// Not part of the C ABI (include/*.h is).
//
// Model shapes (SURVEY 8f N1): the number of GRU_A units is a property of the loaded blob (training_tf2/train_lpcnet.py
// --grua-size; default 384).  Everything that depends on it — warp->neuron-group mapping, tile strides, the whole
// shared-memory map — is a constexpr function of `na` (make_geom below).  The per-sample kernels are compiled once per
// supported size (lpcnet_b200/build.py passes -DLPCNET_NA=<na>; the kernels of a size live in namespace na<na>) so that
// every offset stays a compile-time constant in the hot loop; the host code (model.cu, batch_api.cu) evaluates the same
// function at run time for the size found in the blob.  GRU_B (16 units), the conditioning width (128) and the feature
// layout are fixed (training_tf2/lpcnet.py:234 defaults).
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

namespace lpcnet_b200 {

// ---- fixed model dimensions (default LPCNet: training_tf2/lpcnet.py:234; generated nnet_data.h) ----
constexpr int NB = 16;             // GRU_B units
constexpr int COND = 128;          // conditioning width
constexpr int PITCH_EMBED = 64;
constexpr int NB_FEAT = 20;
constexpr int FRAME_IN = NB_FEAT + PITCH_EMBED;   // 84
constexpr int LPC_ORDER = 16;
constexpr int NB_BANDS = 18;
constexpr int FRAME_SIZE = 160;
constexpr int MAX_FEATURES_DELAY = 2;             // FEATURES_DELAY of the reference (dump_lpcnet.py:323-329) is a per-model value 0..2
constexpr int WINDOW_SIZE = 320;
constexpr int FREQ_SIZE = 161;
constexpr int FRAME_CHUNK = 16;                   // frames of conditioning evaluated (and buffered) per per-sample kernel launch
constexpr int NA_SUPPORTED[] = {128, 256, 384};   // GRU_A sizes with a compiled per-sample kernel (multiples of 128: 16 neuron groups per compute-warp slot)
constexpr int NA_MAX = 384;

// ---- per-sample kernel geometry (warp-specialised CTA) ----
constexpr int STREAMS_PER_CTA = 32;          // stream slots of a CTA; the launcher may leave some dead (SampleParams::spc) to spread a small batch over all SMs
#ifndef LPCNET_NWC
#define LPCNET_NWC 16
#endif
constexpr int NWC = LPCNET_NWC;              // compute warps (12, 16 or 24): each owns NGRP/NWC neuron groups of GRU_A, a (row group, K part) of the
                                             // GRU_B input GEMV and up to ceil(16/NWC) GRU_B neurons.  24 warps x 2 groups keeps the per-thread
                                             // working set small (h, S_h, S_z = 48 registers) so that 7 warps per scheduler hide the LDS latency
#ifndef LPCNET_NWP
#define LPCNET_NWP 6
#endif
constexpr int NWP = LPCNET_NWP;              // producer warps: cooperative gather of the GRU_A input rows.  The gather is latency-bound (L2 hits, ~1k cycles
                                             // under load), so what matters is loads in flight: NWP warps x (registers/4) LDG.128 each
constexpr int SAMPLE_THREADS = (NWC + NWP + 2) * 32;   // + 2 sampler warps, one per half (tree sampler, LPC filter, u-law, de-emphasis)
constexpr int FCW_ROW = 36;                  // dual_fc row: 32 weights (16 per channel) + {bias0, bias1, factor0, factor1}; 144 B stride = 16 mod 128, so the
                                             // per-lane LDS.128 row reads of lanes on different nodes mostly land in different 4-bank groups
constexpr int FCW_SMEM_NODES = 64;           // at most the tree levels 0..5 (nodes 1..63) live in shared memory, the rest is read from global (L2);
                                             // a model whose block lists need the room keeps fewer (32, 16, 8: model.cu), the count travels in the image
constexpr int KPARTS = (NWC >= 24) ? 4 : 2;  // K split of the GRU_B input GEMV
constexpr int NWB = 6 * KPARTS;              // warps used by the GRU_B input GEMV: (row group 0..5) x (K part)
static_assert(NWB <= NWC, "one (row group, K part) of GRU_B per compute warp");
constexpr int HALF = 16;                     // the 32 streams of a CTA are stepped as two halves of 16 (= the M of one MMA), half a sample apart:
                                             // while the sampler / gather of one half run, the compute warps work on the other half
constexpr int NFIN = NB * HALF / 32;         // compute warps that finish GRU_B for a half: lane = (neuron parity, stream in half)
static_assert(NFIN <= NWC, "GRU_B finishing warps");
constexpr int ACCB_ROW = 20;                 // int32 per output row of the GRU_B partial sums (16 streams + 4 pad: the MMA accumulator stores of a warp
                                             // (rows 2t, columns gid) then fall into 32 different banks)
constexpr int NTILE = 4;                     // ring of gather tiles, filled in the order (half A: r, z, h), (half B: r, z, h), ...

// ---- int8 flavour: the integer GEMVs run on the tensor cores (mma.sync m16n8k16, u8 x s8 -> s32, exact) ----
// A "quad" is four 8x4 weight blocks of one 8-row group = one MMA: 16 streams x (4 blocks x 4 inputs) x 8 outputs.
//   weights: 128 B per quad, word [gid][t] = the 4 int8 weights of output row gid for the block in slot t   (B fragment of lane gid*4+t)
//   meta   : 4 x u16 per quad, one per slot: xs_offset(column block of the slot, stream 0)
// Quantised state xs: column block c (inputs 4c..4c+3) is a 128-byte row = 2 halves x 8 streams x 2 words; the word of
// stream s = 16*H + 8*jj + gid sits at
//   c*128 + (((H << 6) | (gid << 3)) ^ (((c & 1) << 6) | ((c & 2) << 4))) + jj*4
// i.e. the two streams {gid, gid+8} of a half that lane (gid, t) feeds to its MMA are one 8-byte vector, and the XOR
// spreads the four slots of a quad (whose column blocks are ordered to have distinct c & 3 where possible) over the
// four 32-byte bank groups that a half-warp (gid 0..3 or 4..7) does not already separate: conflict-free LDS.64.
constexpr uint32_t QUAD_BYTES = 128, QUAD_META_BYTES = 8;
#ifdef __CUDACC__
__host__ __device__
#endif
constexpr uint32_t xs_offset(uint32_t c, uint32_t s)
{
    return c * 128u + (((((s >> 4) & 1u) << 6) | ((s & 7u) << 3)) ^ (((c & 1u) << 6) | ((c & 2u) << 4))) + ((s >> 3) & 1u) * 4u;
}

constexpr uint32_t al128(uint32_t x) { return (x + 127u) & ~127u; }
constexpr uint32_t SMEM_RESERVED = 1024;     // shared-window address of dynamic shared memory on sm_100 (probed at batch_create, batch_api.cu)
constexpr uint32_t T_ACCB = 0;               // the tile that held a half's candidate gate is dead once h~ is computed; until the half's next indices are out
                                             // it carries  int32 [KPARTS][48][ACCB_ROW] partial sums of the GRU_B input GEMV  and
constexpr uint32_t T_ACCB_BYTES = KPARTS * 3 * NB * ACCB_ROW * 4;      //   float [16 neurons][16 streams] GRU_B state for the sampler in the LAST 1 KB of the tile (Geom::t_hbs):
                                             // that is inside the tile's last row(s), the only rows whose conditioning vector may not be
                                             // prefetched into the r tile that takes the slot next (the sampler is still reading; Geom::late_row0)

// float flavour geometry that does not depend on the GRU_A size
constexpr int F_NWC = 16, F_KPARTS = 2, F_NWB = 6 * F_KPARTS;
constexpr int FN_S = 4;                      // neuron-per-lane float kernel: streams per CTA (live slots: SampleParams::spc <= FN_S)

// ---- everything that depends on the number of GRU_A units ----
struct Geom {
    int na;                  // GRU_A units
    int ngrp;                // groups of 8 neurons (one 8-row block group per gate)
    int gpw;                 // neuron groups per compute warp (int8 kernel)
    uint32_t xs_bytes;       // quantised GRU_A state of 32 streams: [na/4 column blocks][32 words], see xs_offset()
    uint32_t gin_row;        // floats per stream in a gather tile: na + 8 pad => row stride = 8 words mod 32: the LDS.64 of lanes (gid, t) = row gid,
                             // column 2t hit 32 different banks per half-warp
    uint32_t tile_bytes;     // one gate of one half: float [16 streams][gin_row]
    uint32_t t_hbs;          // offset of the GRU_B state scratch inside a (dead) candidate-gate tile
    int late_row0;           // first tile row that overlaps it
    // shared-memory map of the int8 per-sample kernel.  Everything whose size does not depend on the model's sparsity pattern
    // sits at a COMPILE-TIME offset (keeps the addresses out of registers); only the four block-sparse arrays are placed at
    // run-time offsets behind them.  [sm_image, sm_image + image_bytes) is copied verbatim from the global "SMEM image" built
    // at model-load time (TMA bulk copies); [0, sm_image) is the mutable working set.
    uint32_t sm_xs;          // 2 x quantised GRU_A state (double-buffered), both halves interleaved (xs_offset)
    uint32_t sm_xb;          // u32 [2 halves][2 buffers][4 words][16 streams]: quantised GRU_B state
    uint32_t sm_tiles;
    uint32_t sm_idx;         // int32 [2 halves][3][16]: last_sig_ulaw, pred_ulaw, last_exc
    uint32_t sm_mbar;        // mbarriers: image | full[NTILE] | empty[NTILE] | idx[2] | x[2] | accb[2]
    uint32_t mb_image, mb_full, mb_empty, mb_idx, mb_x, mb_accb;
    uint32_t mb_cond;        // [NTILE]: the conditioning rows of a tile have landed (TMA, complete_tx)
    uint32_t sm_image;
    // image, fixed part (offsets relative to sm_image)
    uint32_t im_logit;       // float [256] sampling_logit_table
    uint32_t im_u2l;         // float [256] ulaw2lin
    uint32_t im_dira;        // uint32 [NWC][gpw][3][2] = {first quad, quad count}
    uint32_t im_grpa;        // uint32 [NWC][gpw] neuron-group id
    uint32_t im_dirb;        // uint32 [NWB][2]
    uint32_t im_pre_end;
    uint32_t im_rcp;         // u32 [2048] RCPPS table, pre-biased: T[k] + 0x3f800000 (one IADD rebuilds the result); its absolute shared address
                             // is 8 KB-aligned so that the entry address is table | index (no add)
    uint32_t im_fcwn;        // u32: number of dual_fc rows present at im_fcw (lives in the alignment gap in front of the table)
    uint32_t im_para;        // float [NWC][gpw][3 gates][16] = recurrent su-bias[8], diag[8]
    uint32_t im_wbrec;       // int8 [6][4][8][4] GRU_B recurrent blocks
    uint32_t im_parb;        // float [96]: input-side su-bias[48], recurrent-side su-bias[48]
    uint32_t im_fcw;         // float [<= FCW_SMEM_NODES][FCW_ROW] dual_fc rows of the upper tree levels
    uint32_t im_var;         // start of the variable-size arrays when all FCW_SMEM_NODES rows are kept
    // ---- FLOAT flavour, lane == stream kernel (sample_kernel_f32.cu): fp32 GRU_A state tile instead of the u8 one, no gather
    // tiles (per-lane gather), fp16 weights (64 B per block), the whole dual_fc table read from global memory
    int f_gpw;
    uint32_t f_xs;           // float [na][32]: GRU_A state of the 32 streams (single buffer)
    uint32_t f_hb;           // float [2][16][32]: GRU_B state (double-buffered)
    uint32_t f_accb;         // float [48][32]: GRU_B input-side pre-activations
    uint32_t f_idx;          // int32 [3][32]
    uint32_t f_mbar, f_image;
    uint32_t fi_rcp, fi_logit, fi_u2l, fi_fcb, fi_fcf;
    uint32_t fi_para;        // float [F_NWC][f_gpw][3][16] = recurrent bias[8], diag[8]
    uint32_t fi_dira, fi_grpa;
    uint32_t fi_dirb;        // uint32 [6*F_KPARTS][2] (only part 0 of each row group is non-empty)
    uint32_t fi_parb;        // float [96]: input-side bias[48], recurrent-side bias[48]
    uint32_t fi_var;
    // ---- FLOAT flavour, small batches: neuron-per-lane kernel (sample_kernel_f32n.cu).  With only a few streams per SM the
    // lane==stream mapping leaves the lanes idle and every lane walks all chains of its warp's neurons.  Here a compute lane owns
    // ONE GRU_A neuron (its z, r and h rows: three sequential fp32 FMA chains in the reference's block order) for up to FN_S
    // streams of the CTA; the latency of a sample is then set by the longest chain (the na-term rows of GRU_B)
    int fn_nwc;              // na / 32 compute warps: na lanes = na neurons
    int fn_threads;          // + sampler warp (lane == stream)
    uint32_t fn_x;           // float [2][FN_S][na]: GRU_A state (double-buffered)
    uint32_t fn_hb;          // float [2][NB][FN_S]: GRU_B state (double-buffered)
    uint32_t fn_accb;        // float [48][FN_S]: GRU_B input-side pre-activations
    uint32_t fn_idx;         // int32 [3][FN_S]
    uint32_t fn_mbar, fn_image;
    uint32_t fni_rcp, fni_logit, fni_u2l;
    uint32_t fni_fcw;        // float [256][FCW_ROW]: all dual_fc rows (weights, biases, factors)
    uint32_t fni_neur;       // u16 [na]: neuron of compute lane (warp*32 + lane); groups sorted by list length
    uint32_t fni_dira;       // u32 [ngrp groups][3 gates][2] = {first block, block count}
    uint32_t fni_para;       // float [3 gates][2][na]: recurrent bias, diag per neuron
    uint32_t fni_dirb;       // u32 [6][2]
    uint32_t fni_parb;       // float [96]
    uint32_t fni_wbrec;      // float [16 in][48 out]
    uint32_t fni_var;        // blocks: fp16 [8 rows][4 cols] (64 B), u16 meta = 4 * pos
};

constexpr bool na_supported(int na) { for (int v : NA_SUPPORTED) if (v == na) return true; return false; }

constexpr Geom make_geom(int na)
{
    Geom g{};
    g.na = na; g.ngrp = na / 8; g.gpw = g.ngrp / NWC;
    g.xs_bytes = (uint32_t)(na / 4) * 32u * 4u;
    g.gin_row = (uint32_t)na + 8u;
    g.tile_bytes = HALF * g.gin_row * 4u;
    g.t_hbs = g.tile_bytes - NB * HALF * 4u;
    g.late_row0 = (int)(g.t_hbs / (g.gin_row * 4u));
    g.sm_xs = 0;
    g.sm_xb = g.sm_xs + 2 * g.xs_bytes;
    g.sm_tiles = g.sm_xb + 2 * 2 * 4 * HALF * 4;
    g.sm_idx = g.sm_tiles + NTILE * g.tile_bytes;
    g.sm_mbar = al128(g.sm_idx + 2 * 3 * HALF * 4);
    g.mb_image = g.sm_mbar; g.mb_full = g.sm_mbar + 8; g.mb_empty = g.mb_full + 8 * NTILE; g.mb_idx = g.mb_empty + 8 * NTILE;
    g.mb_x = g.mb_idx + 16; g.mb_accb = g.mb_x + 16;
    g.mb_cond = g.sm_mbar + 128;
    g.sm_image = g.sm_mbar + 128 + 8 * NTILE;      // (32-byte aligned: enough for the bulk copies and every vector access into the image)
    g.im_logit = 0;
    g.im_u2l = g.im_logit + 256 * 4;
    g.im_dira = g.im_u2l + 256 * 4;
    g.im_grpa = g.im_dira + (uint32_t)(NWC * g.gpw * 3 * 2 * 4);
    g.im_dirb = g.im_grpa + (uint32_t)(NWC * g.gpw * 4);
    g.im_pre_end = g.im_dirb + NWB * 2 * 4;
    g.im_rcp = g.im_pre_end + (8192u - (SMEM_RESERVED + g.sm_image + g.im_pre_end) % 8192u) % 8192u;
    if (g.im_rcp - g.im_pre_end < 4) g.im_rcp += 8192u;      // room for the dual_fc row count in front of the table
    g.im_fcwn = g.im_pre_end;
    g.im_para = g.im_rcp + 2048 * 4;
    g.im_wbrec = g.im_para + (uint32_t)(NWC * g.gpw * 3 * 16 * 4);
    g.im_parb = g.im_wbrec + 3 * NB * NB;
    g.im_fcw = al128(g.im_parb + 6 * NB * 4);
    g.im_var = g.im_fcw + FCW_SMEM_NODES * FCW_ROW * 4;
    // float, lane == stream
    g.f_gpw = g.ngrp / F_NWC;
    g.f_xs = 0;
    g.f_hb = g.f_xs + (uint32_t)na * 32 * 4;
    g.f_accb = g.f_hb + 2 * NB * 32 * 4;
    g.f_idx = g.f_accb + 3 * NB * 32 * 4;
    g.f_mbar = al128(g.f_idx + 3 * 32 * 4);
    g.f_image = g.f_mbar + 128;
    g.fi_rcp = 0;
    g.fi_logit = g.fi_rcp + 2048 * 2;
    g.fi_u2l = g.fi_logit + 256 * 4;
    g.fi_fcb = g.fi_u2l + 256 * 4;
    g.fi_fcf = g.fi_fcb + 512 * 4;
    g.fi_para = g.fi_fcf + 512 * 4;
    g.fi_dira = g.fi_para + (uint32_t)(F_NWC * g.f_gpw * 3 * 16 * 4);
    g.fi_grpa = g.fi_dira + (uint32_t)(F_NWC * g.f_gpw * 3 * 2 * 4);
    g.fi_dirb = g.fi_grpa + (uint32_t)(F_NWC * g.f_gpw * 4);
    g.fi_parb = g.fi_dirb + F_NWB * 2 * 4;
    g.fi_var = al128(g.fi_parb + 6 * NB * 4);
    // float, neuron per lane
    g.fn_nwc = na / 32;
    g.fn_threads = (g.fn_nwc + 1) * 32;
    g.fn_x = 0;
    g.fn_hb = g.fn_x + 2 * FN_S * (uint32_t)na * 4;
    g.fn_accb = g.fn_hb + 2 * NB * FN_S * 4;
    g.fn_idx = g.fn_accb + 3 * NB * FN_S * 4;
    g.fn_mbar = al128(g.fn_idx + 3 * FN_S * 4);
    g.fn_image = g.fn_mbar + 128;
    g.fni_rcp = 0;
    g.fni_logit = g.fni_rcp + 2048 * 2;
    g.fni_u2l = g.fni_logit + 256 * 4;
    g.fni_fcw = g.fni_u2l + 256 * 4;
    g.fni_neur = g.fni_fcw + 256 * FCW_ROW * 4;
    g.fni_dira = g.fni_neur + (uint32_t)na * 2;
    g.fni_para = g.fni_dira + (uint32_t)g.ngrp * 3 * 2 * 4;
    g.fni_dirb = g.fni_para + 3 * 2 * (uint32_t)na * 4;
    g.fni_parb = g.fni_dirb + 64;
    g.fni_wbrec = g.fni_parb + 6 * NB * 4;
    g.fni_var = al128(g.fni_wbrec + 3 * NB * NB * 4);
    return g;
}

// offsets used by the (flavour-agnostic) image builder
struct ImageMap { uint32_t sm_image, rcp, logit, u2l, fcw, fcb, fcf, parA, dirA, grpA, dirB, wBrec, parB, var; };
constexpr ImageMap map_int8(const Geom &g) { return {g.sm_image, g.im_rcp, g.im_logit, g.im_u2l, g.im_fcw, 0xFFFFFFFFu, 0xFFFFFFFFu, g.im_para, g.im_dira, g.im_grpa, g.im_dirb, g.im_wbrec, g.im_parb, g.im_var}; }
constexpr ImageMap map_f32(const Geom &g) { return {g.f_image, g.fi_rcp, g.fi_logit, g.fi_u2l, 0xFFFFFFFFu, g.fi_fcb, g.fi_fcf, g.fi_para, g.fi_dira, g.fi_grpa, g.fi_dirb, 0xFFFFFFFFu, g.fi_parb, g.fi_var}; }

#ifdef LPCNET_NA
// ---- kernel translation units: the geometry of THIS compilation as plain compile-time names ----
#define LPCNET_CAT2(a, b) a##b
#define LPCNET_CAT(a, b) LPCNET_CAT2(a, b)
#define LPCNET_KNS LPCNET_CAT(na, LPCNET_NA)          // namespace of the kernels of this size: lpcnet_b200::na384 ...
static_assert(na_supported(LPCNET_NA), "unsupported GRU_A size");
constexpr Geom GEO = make_geom(LPCNET_NA);
constexpr int NA = GEO.na, NGRP = GEO.ngrp, GPW = GEO.gpw;
static_assert(NGRP % NWC == 0, "compute warps must divide the neuron groups");
constexpr int XS_BYTES = (int)GEO.xs_bytes, GIN_ROW = (int)GEO.gin_row;
constexpr uint32_t TILE_BYTES = GEO.tile_bytes;
constexpr uint32_t T_HBS = GEO.t_hbs;
constexpr int LATE_ROW0 = GEO.late_row0;
static_assert(T_ACCB + T_ACCB_BYTES <= T_HBS, "GRU_B scratch must fit inside the gather tile it aliases");
constexpr uint32_t SM_XS = GEO.sm_xs, SM_XB = GEO.sm_xb, SM_TILES = GEO.sm_tiles, SM_IDX = GEO.sm_idx, SM_MBAR = GEO.sm_mbar;
constexpr uint32_t MB_IMAGE = GEO.mb_image, MB_FULL = GEO.mb_full, MB_EMPTY = GEO.mb_empty, MB_IDX = GEO.mb_idx, MB_X = GEO.mb_x, MB_ACCB = GEO.mb_accb, MB_COND = GEO.mb_cond;
constexpr uint32_t SM_IMAGE = GEO.sm_image;
static_assert(MB_ACCB + 16 + 8 <= MB_COND && MB_COND + 8 * NTILE <= SM_IMAGE, "mbarrier block (+ the TMEM base word and the opaque 1.0f behind MB_ACCB)");
constexpr uint32_t IM_LOGIT = GEO.im_logit, IM_U2L = GEO.im_u2l, IM_DIRA = GEO.im_dira, IM_GRPA = GEO.im_grpa, IM_DIRB = GEO.im_dirb, IM_PRE_END = GEO.im_pre_end;
constexpr uint32_t IM_RCP = GEO.im_rcp, IM_FCWN = GEO.im_fcwn, IM_PARA = GEO.im_para, IM_WBREC = GEO.im_wbrec, IM_PARB = GEO.im_parb, IM_FCW = GEO.im_fcw, IM_VAR = GEO.im_var;
static_assert((SMEM_RESERVED + SM_IMAGE + IM_RCP) % 8192u == 0, "rcp table alignment");
static_assert(IM_RCP - IM_PRE_END >= 4, "room for the dual_fc row count");
constexpr int F_GPW = GEO.f_gpw;
constexpr uint32_t F_XS = GEO.f_xs, F_HB = GEO.f_hb, F_ACCB = GEO.f_accb, F_IDX = GEO.f_idx, F_MBAR = GEO.f_mbar, F_IMAGE = GEO.f_image;
constexpr uint32_t FI_RCP = GEO.fi_rcp, FI_LOGIT = GEO.fi_logit, FI_U2L = GEO.fi_u2l, FI_FCB = GEO.fi_fcb, FI_FCF = GEO.fi_fcf, FI_PARA = GEO.fi_para;
constexpr uint32_t FI_DIRA = GEO.fi_dira, FI_GRPA = GEO.fi_grpa, FI_DIRB = GEO.fi_dirb, FI_PARB = GEO.fi_parb, FI_VAR = GEO.fi_var;
constexpr int FN_NWC = GEO.fn_nwc, FN_THREADS = GEO.fn_threads;
constexpr uint32_t FN_X = GEO.fn_x, FN_HB = GEO.fn_hb, FN_ACCB = GEO.fn_accb, FN_IDX = GEO.fn_idx, FN_MBAR = GEO.fn_mbar, FN_IMAGE = GEO.fn_image;
constexpr uint32_t FNI_RCP = GEO.fni_rcp, FNI_LOGIT = GEO.fni_logit, FNI_U2L = GEO.fni_u2l, FNI_FCW = GEO.fni_fcw, FNI_NEUR = GEO.fni_neur, FNI_DIRA = GEO.fni_dira;
constexpr uint32_t FNI_PARA = GEO.fni_para, FNI_DIRB = GEO.fni_dirb, FNI_PARB = GEO.fni_parb, FNI_WBREC = GEO.fni_wbrec, FNI_VAR = GEO.fni_var;
#endif

struct SmemLayout {          // run-time part; offsets are absolute (from the start of dynamic shared memory)
    uint32_t wA;        // GRU_A weights, ordered (warp, slot, gate): int8 flavour 128-byte quads, float flavour 64-byte fp16 blocks
    uint32_t metaA;     // int8: 4 x u16 per quad (xs_offset of each slot's column block); float: u16 per block
    uint32_t wB;        // GRU_B input weights, ordered (row group, K part)
    uint32_t metaB;
    uint32_t wBrecF;    // float flavour, lane==stream image: fp32 [16 in][48 out] GRU_B recurrent weights.  Neuron-per-lane image (its
                        // recurrent weights sit at fni_wbrec): 1 if every GRU_B row group lists all na/4 column blocks in order
    uint32_t sm_image;  // where the image starts (sm_image for int8, f_image / fn_image for the float flavour)
    uint32_t image_bytes;
    uint32_t total_bytes;
    uint32_t nblkA_padded, nblkB_padded;   // units in wA / wB: quads (int8 flavour) or blocks (float flavour)
};

// Per-model switches the reference bakes into the generated nnet_data.h (training_tf2/dump_lpcnet.py:306-329).
struct ModelConfig {
    float lpc_gamma;        // LPC_GAMMA (lpc_weighting, freq.c:299-308); 1 = none
    int features_delay;     // FEATURES_DELAY 0..2: look-ahead of the conditioning network = silent frames after a reset, age of the LPC used (lpcnet.c:101,109-115,239)
    int end2end;            // END2END: LPC from the first 16 outputs of feature_dense2 taken as reflection coefficients (rc2lpc, lpcnet.c:57-78,107-108)
};

// Device-resident model (one per batch; weights replicated per GPU, ~4 MB).
struct DeviceModel {
    int is_float;                    // 0: int8 DOT_PROD semantics (oracle A); 1: float semantics (oracle B)
    int fast_cvt;                    // int8: GRU_A pre-activations provably < 2^22 accumulator units (conversion-free rounding allowed)
    int na;                          // GRU_A units of the loaded blob
    ModelConfig cfg;
    SmemLayout L;
    uint8_t *image;                  // [L.image_bytes] global copy of the SMEM image
    SmemLayout Ln;                   // float flavour: layout / image of the neuron-per-lane kernel (small batches)
    uint8_t *image_n;
    // per-sample gathers (L2-resident): [256][3*na] each
    float *emb_sig, *emb_pred, *emb_exc;
    float *fcw;                      // dual_fc rows [256][FCW_ROW] = 32 weights, 2 biases, 2 factors (the lower tree levels are read from here)
    // frame network (fp32, reference layouts kept: column-major W[j*N+i], conv W[(k*in+i)*out+o])
    float *embed_pitch;              // [256][64]
    float *conv1_w, *conv1_b, *conv2_w, *conv2_b;
    float *dense1_w, *dense1_b, *dense2_w, *dense2_b;
    float *gad_w, *gad_b, *gbd_w, *gbd_b;
    // tables
    uint16_t *rcp16;                 // [2048]
    float *dct;                      // [18*18]
    float *twiddles;                 // [320*2]
    int16_t *bitrev;                 // [320]
    float *gamma_pow;                // [16] gamma^(i+1) accumulated in float exactly like lpc_weighting (freq.c:299-308)
    float *pitch_pow;                // [64] (float)(pow(2.f, k/21.)*32) for the packet decoder (lpcnet_dec.c:124)
    float *codebooks;                // cb1,cb2,cb3,diff4 or NULL
    // accounting
    long algo_bytes_total, algo_bytes_sparse;
    int nblkA, nblkB;
};

struct SampleParams {
    SmemLayout L;
    const uint8_t *image;
    const float *emb_sig, *emb_pred, *emb_exc;
    const float *fcw;        // [256][FCW_ROW] dual_fc rows (levels 6,7 of the sampling tree)
    const float *condA;      // int8 flavour [nframes][3 gates][n][na + 8], float flavour [nframes][n][3*na]: condA_frame_floats()
    const float *condB;      // [nframes][n][3*NB]
    const float *lpc_raw;    // [nframes][n][16]: entry f = the raw LPC the sample loop of frame f uses (the caller applies the model's FEATURES_DELAY)
    const float *gamma_pow;  // [16]
    float *hA;               // [na][n]
    float *hB;               // [NB][n]
    float *last_sig;         // [16][n]
    float *deemph;           // [n]
    int *last_exc;           // [n]
    uint32_t *rng;           // [4][n]
    short *pcm;              // stream s, frame f, sample t at pcm[s*pcm_stream_stride + f*spf + t]
    long long pcm_stream_stride;
    int n_streams, nframes, spf;
    int fast_cvt;            // bit 0: conversion-free accumulator rounding; bits 8..: `preload` of lpcnet_synthesize_impl (lpcnet.c:256-259,269): the
                             // first (fast_cvt >> 8) samples of the call's FIRST frame are teacher-forced from the PCM already in `pcm`
    int spc;                 // live streams per CTA (1..32): chosen by the launcher so that the grid covers the SMs
    int one_half;            // spc <= 16: all live streams sit in half A and half B is not stepped at all (a small batch is bound by the
                             // latency of one sample, which the second half would only lengthen)
#ifdef LPCNET_TRACE
    long long *trace;        // tuning builds only: clock64 stamps of CTA 0, [8 samples][32 events]
#endif
};
// (the layout of SampleParams is frozen: one more word measured -6 % on the int8 kernel, see DESIGN.md; new per-call switches
// are packed into existing words)

// gru_a_dense_feature output of one frame (the GRU_A conditioning rows).  int8 flavour: gate-major with the row pitch of a gather tile
// (na + 8 floats), so that the rows of consecutive streams for one gate are one contiguous piece of memory that a single TMA bulk copy
// drops into a tile (sample_kernel.cu, gather_half_tma); float flavour: the reference's [stream][3*na].
inline size_t condA_frame_floats(bool is_float, size_t n, int na) { return is_float ? n * 3 * (size_t)na : 3 * n * (size_t)(na + 8); }

// ---- host-side API of the internal modules ----
int model_load(DeviceModel *m, const unsigned char *blob, int len, const ModelConfig *cfg);   // 0 / -1 (sets error); cfg NULL = blob metadata / defaults
void model_free(DeviceModel *m);
int debug_build_image(const unsigned char *blob, int len, unsigned char *out, size_t cap, SmemLayout *L, Geom *g, int *fast_cvt, int *is_float);
int debug_build_image_n(const unsigned char *blob, int len, unsigned char *out, size_t cap, SmemLayout *L, Geom *g);
void set_error(const char *fmt, ...);

struct FrameState {           // per-batch persistent state of the 100 Hz path
    float *conv1_state;       // [n][FRAME_IN*2]
    float *conv2_state;       // [n][COND*2]
    float *lpc_carry;         // [2][n][16] raw LPC of the two previous frames
    float *vq_mem;            // [n][18] decoder memory
    int *frame_count;         // [n] frames seen since the stream's last reset, saturating at 1000 (lpcnet.c:119)
    float *work;              // scratch of the layer-by-layer conditioning network (frame_work_floats(n) floats; not part of the state)
    cudaStream_t side;        // side stream + fork / join events: cepstrum -> LPC runs next to the conditioning network (NULL: in line)
    cudaEvent_t ev_fork, ev_join;
};

// lpc_raw [nframes+2][n][16]: entry e = raw LPC of frame e-2 of the call (entries 0,1 = carry); frame f reads entry f + 2 - delay
void launch_frame_network(const DeviceModel &m, const FrameState &fs, const float *d_features, long long stream_stride,
                          int frame_stride, int n, int nframes, float *condA, float *condB, float *lpc_raw, cudaStream_t st);
int frame_network_launches(const DeviceModel &m);           // engine kernels one launch_frame_network call launches
size_t frame_work_floats(size_t n);
void launch_decode_packets(const DeviceModel &m, const FrameState &fs, const uint8_t *d_packets, int n, int npackets,
                           float *d_features /* [n][4*npackets][20] */, cudaStream_t st);
// one set of launchers per compiled GRU_A size
#define LPCNET_DECLARE_LAUNCHERS(ns) namespace ns { \
    cudaError_t launch_sample_kernel(const SampleParams &p, cudaStream_t st); \
    cudaError_t launch_sample_kernel_f32(const SampleParams &p, cudaStream_t st); \
    cudaError_t launch_sample_kernel_f32n(const SampleParams &p, cudaStream_t st);   /* p.L / p.image = DeviceModel::Ln / image_n, p.spc <= FN_S */ }
LPCNET_DECLARE_LAUNCHERS(na128)
LPCNET_DECLARE_LAUNCHERS(na256)
LPCNET_DECLARE_LAUNCHERS(na384)
int sample_kernel_smem_ok(uint32_t bytes);
int streams_per_cta_for(int n_streams, int override_spc);   // min(32, ceil(n / SM count)) on the current device unless overridden

}  // namespace lpcnet_b200
