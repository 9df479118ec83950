// model.cu — "DNNw" blob ingest and device model construction.
//
// Replaces (reference file:line): parse_weights / parse_record  src/parse_lpcnet_weights.c:37-77,
// find_idx_check :90-113, the per-layer *_init validators :115-221 and the generated init_lpcnet_model
// (training_tf2/dump_lpcnet.py:147,181,199,224,242,252).  Instead of pointing layer structs into the blob it builds
//   * the shared-memory image of the per-sample kernel (block-sparse int8 GRU_A/GRU_B weights re-ordered by
//     owning warp, su-bias/diag per row group, dual_fc, sampler tables) and
//   * plain device copies of the frame-rate fp32 layers and the three 1.18 MB gather tables.
#include <algorithm>
#include <array>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <string>
#include <vector>
#include <cuda_fp16.h>
#include "engine.h"

namespace lpcnet_b200 {

static thread_local char g_err[512] = "";
void set_error(const char *fmt, ...)
{
    va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof(g_err), fmt, ap); va_end(ap);
}
const char *get_error() { return g_err; }

static const uint16_t kRcpTable[2048] = {
#include "rcpps_table.inc"
};

namespace {

struct WeightHead { char head[4]; int version; int type; int size; int block_size; char name[44]; };
static_assert(sizeof(WeightHead) == 64, "DNNw header is 64 bytes (nnet.h:53-60)");

struct Arr { const unsigned char *data; int size; int type; };

// parse_record semantics (parse_lpcnet_weights.c:37-52): walk 64-byte headers, reject malformed records.
bool parse_blob(const unsigned char *d, int len, std::vector<std::pair<std::string, Arr>> &out)
{
    while (len > 0) {
        if (len < 64) return false;
        const WeightHead *h = reinterpret_cast<const WeightHead *>(d);
        if (h->block_size < h->size) return false;
        if (h->block_size > len - 64) return false;
        if (h->name[43] != 0) return false;
        if (h->size <= 0) return false;
        out.push_back({std::string(h->name), Arr{d + 64, h->size, h->type}});
        d += 64 + h->block_size; len -= 64 + h->block_size;
    }
    return true;
}

const Arr *find(const std::vector<std::pair<std::string, Arr>> &v, const char *name)
{
    for (auto &p : v) if (p.first == name) return &p.second;
    return nullptr;
}
const float *need_f(const std::vector<std::pair<std::string, Arr>> &v, const char *name, int count)
{
    const Arr *a = find(v, name);
    if (!a || a->size != count * 4) { set_error("model: array '%s' missing or wrong size (want %d floats)", name, count); return nullptr; }
    return reinterpret_cast<const float *>(a->data);
}
// find_idx_check (parse_lpcnet_weights.c:90-113)
const int *need_idx(const std::vector<std::pair<std::string, Arr>> &v, const char *name, int nb_in, int nb_out, int *total)
{
    const Arr *a = find(v, name);
    *total = 0;
    if (!a) { set_error("model: index array '%s' missing", name); return nullptr; }
    const int *idx = reinterpret_cast<const int *>(a->data);
    int remain = a->size / 4;
    const int *p = idx;
    while (remain > 0) {
        int nb = *p++;
        if (nb < 0 || remain < nb + 1) { set_error("model: '%s' truncated", name); return nullptr; }
        for (int i = 0; i < nb; i++) { int pos = *p++; if (pos < 0 || pos + 3 >= nb_in || (pos & 3)) { set_error("model: '%s' bad position", name); return nullptr; } }
        nb_out -= 8; remain -= nb + 1; *total += nb;
    }
    if (nb_out != 0) { set_error("model: '%s' does not cover all output rows", name); return nullptr; }
    return idx;
}

template <typename T> T *to_device(const T *h, size_t count)
{
    T *d = nullptr;
    if (cudaMalloc(&d, count * sizeof(T)) != cudaSuccess) return nullptr;
    if (cudaMemcpy(d, h, count * sizeof(T), cudaMemcpyHostToDevice) != cudaSuccess) { cudaFree(d); return nullptr; }
    return d;
}

uint32_t align_up(uint32_t x, uint32_t a) { return (x + a - 1) / a * a; }

}  // namespace

struct HostModel {               // everything model_load needs after parsing, before any CUDA call
    std::vector<uint8_t> img;
    std::vector<uint8_t> img_n;  // float flavour: image of the neuron-per-lane kernel
    std::vector<float> fc_rows;  // [256][FCW_ROW]
    const float *embed_pitch, *conv1_w, *conv1_b, *conv2_w, *conv2_b, *dense1_w, *dense1_b, *dense2_w, *dense2_b;
    const float *gad_w, *gad_b, *gbd_w, *gbd_b, *emb_sig, *emb_pred, *emb_exc;
};

// Optional metadata record of blobs written by this library's exporter (lpcnet_b200_write_blob / tools/import_nnet_data.py):
// float [4] = {LPC_GAMMA, FEATURES_DELAY, END2END, format version}.  The reference keeps these three in the generated
// nnet_data.h (dump_lpcnet.py:306-329), i.e. outside the blob; its parser ignores arrays it does not look up, so the record
// does not disturb lpcnet_load_model of the reference.
static const char *kConfigRecord = "lpcnet_b200_config";

static int build_host_model(DeviceModel *m, HostModel &hm, const unsigned char *blob, int len, const ModelConfig *cfg_in)
{
    memset(m, 0, sizeof(*m));
    std::vector<std::pair<std::string, Arr>> A;
    if (!blob || len <= 0 || !parse_blob(blob, len, A)) { set_error("model: malformed DNNw blob"); return -1; }
    // ---- per-model switches: explicit argument > metadata record > the reference's defaults (gamma 1 = no weighting would be
    // wrong for most models, so callers without metadata must pass it: lpcnet_b200_batch_create has the argument) ----
    m->cfg = ModelConfig{1.0f, MAX_FEATURES_DELAY, 0};
    if (const Arr *c = find(A, kConfigRecord)) {
        if (c->size >= 12) { const float *v = reinterpret_cast<const float *>(c->data); m->cfg = ModelConfig{v[0], (int)v[1], v[2] != 0.f}; }
    }
    if (cfg_in) {
        if (cfg_in->lpc_gamma > 0.f) m->cfg.lpc_gamma = cfg_in->lpc_gamma;
        if (cfg_in->features_delay >= 0) m->cfg.features_delay = cfg_in->features_delay;
        if (cfg_in->end2end >= 0) m->cfg.end2end = cfg_in->end2end;
    }
    if (m->cfg.features_delay < 0 || m->cfg.features_delay > MAX_FEATURES_DELAY) { set_error("model: FEATURES_DELAY %d not in 0..%d", m->cfg.features_delay, MAX_FEATURES_DELAY); return -1; }
    // ---- GRU_A size from the blob (training_tf2/train_lpcnet.py --grua-size); GRU_B / conditioning widths are fixed ----
    {
        const Arr *d = find(A, "sparse_gru_a_recurrent_weights_diag");
        if (!d || d->size % 12) { set_error("model: array 'sparse_gru_a_recurrent_weights_diag' missing"); return -1; }
        m->na = d->size / 12;
        if (!na_supported(m->na)) {
            set_error("model: GRU_A has %d units; per-sample kernels are built for 128, 256 and 384 (larger models do not fit one SM's shared memory with this mapping)", m->na);
            return -1;
        }
    }
    const int NA = m->na;
    const Geom G = make_geom(NA);
    const int NGRP = G.ngrp;

#define NEED(var, name, count) const float *var = need_f(A, name, count); if (!var) return -1;
    NEED(embed_pitch, "embed_pitch_weights", 256 * PITCH_EMBED)
    NEED(conv1_w, "feature_conv1_weights", 3 * FRAME_IN * COND) NEED(conv1_b, "feature_conv1_bias", COND)
    NEED(conv2_w, "feature_conv2_weights", 3 * COND * COND) NEED(conv2_b, "feature_conv2_bias", COND)
    NEED(dense1_w, "feature_dense1_weights", COND * COND) NEED(dense1_b, "feature_dense1_bias", COND)
    NEED(dense2_w, "feature_dense2_weights", COND * COND) NEED(dense2_b, "feature_dense2_bias", COND)
    NEED(gad_w, "gru_a_dense_feature_weights", COND * 3 * NA) NEED(gad_b, "gru_a_dense_feature_bias", 3 * NA)
    NEED(gbd_w, "gru_b_dense_feature_weights", COND * 3 * NB) NEED(gbd_b, "gru_b_dense_feature_bias", 3 * NB)
    NEED(emb_sig, "gru_a_embed_sig_weights", 256 * 3 * NA) NEED(emb_pred, "gru_a_embed_pred_weights", 256 * 3 * NA)
    NEED(emb_exc, "gru_a_embed_exc_weights", 256 * 3 * NA)
    NEED(ga_bias, "sparse_gru_a_bias", 6 * NA) NEED(ga_subias, "sparse_gru_a_subias", 6 * NA)
    NEED(ga_diag, "sparse_gru_a_recurrent_weights_diag", 3 * NA)
    NEED(gb_bias, "gru_b_bias", 6 * NB) NEED(gb_subias, "gru_b_subias", 6 * NB)
    NEED(fc_w, "dual_fc_weights", 256 * 2 * NB) NEED(fc_b, "dual_fc_bias", 512) NEED(fc_f, "dual_fc_factor", 512)
#undef NEED
    int nblkA = 0, nblkB = 0;
    const int *idxA = need_idx(A, "sparse_gru_a_recurrent_weights_idx", NA, 3 * NA, &nblkA); if (!idxA) return -1;
    const int *idxB = need_idx(A, "gru_b_weights_idx", NA, 3 * NB, &nblkB); if (!idxB) return -1;
    const Arr *wA = find(A, "sparse_gru_a_recurrent_weights");
    const Arr *wB = find(A, "gru_b_weights");
    const Arr *wBrec = find(A, "gru_b_recurrent_weights");
    if (!wA || !wB || !wBrec) { set_error("model: recurrent weight arrays missing"); return -1; }
    if (wA->size == 32 * nblkA) m->is_float = 0;
    else if (wA->size == 128 * nblkA) m->is_float = 1;
    else { set_error("model: sparse_gru_a_recurrent_weights has %d bytes for %d blocks", wA->size, nblkA); return -1; }
    if (wB->size != (m->is_float ? 128 : 32) * nblkB || wBrec->size != (m->is_float ? 4 : 1) * 3 * NB * NB) {
        set_error("model: gru_b weight sizes inconsistent with the blob flavour"); return -1;
    }
    const int src_blk = m->is_float ? 128 : 32;      // bytes per 8x4 block in the blob
    const int img_blk = m->is_float ? 64 : 32;       // bytes per block in shared memory (float flavour: fp16 storage)
    if (m->is_float) {
        // The float flavour keeps the recurrent weights in shared memory as fp16 (BASELINE config 2): only lossless when
        // every weight is exactly representable (true for the k/128 weights of quantisation-aware models, lpcnet.py:118-126).
        auto fp16_exact = [](const unsigned char *d, int bytes) {
            const float *f = reinterpret_cast<const float *>(d);
            for (int i = 0; i < bytes / 4; i++) if (__half2float(__float2half_rn(f[i])) != f[i]) return false;
            return true;
        };
        if (!fp16_exact(wA->data, wA->size) || !fp16_exact(wB->data, wB->size)) {
            set_error("model: float blob whose recurrent weights are not fp16-exact; the fp32-weight variant is not built"); return -1;
        }
    }
    m->nblkA = nblkA; m->nblkB = nblkB;

    // ---------------- GRU_A: assign the 48 neuron groups to the 16 compute warps (LPT on block count) ----------------
    // per 8-row group rg (0..143): list of (pos, weight ptr)
    struct Blk { int pos; const unsigned char *w; };
    std::vector<std::vector<Blk>> rowsA(3 * NGRP), rowsB(3 * NB / 8);
    {
        const int *p = idxA; const unsigned char *w = wA->data;
        for (int rg = 0; rg < 3 * NGRP; rg++) { int nb = *p++; for (int j = 0; j < nb; j++) { rowsA[rg].push_back({*p++, w}); w += src_blk; } }
        p = idxB; w = wB->data;
        for (int rg = 0; rg < 3 * NB / 8; rg++) { int nb = *p++; for (int j = 0; j < nb; j++) { rowsB[rg].push_back({*p++, w}); w += src_blk; } }
    }
    // int8 flavour: the reference multiplies pairs of inputs with _mm256_maddubs_epi16 (vec_avx.h:811-812), whose int16 pair sum
    // SATURATES; the exact integer sums of IMMA/dp4a equal it only while no pair can saturate, i.e. (u8 activations <= 255)
    // 255 * (|w0| + |w1|) <= 32767 for same-sign pairs and 255 * max|w| <= 32768 otherwise.  Quantisation-aware models satisfy
    // it by construction (WeightClip, training_tf2/lpcnet.py:216-232); a blob that does not would silently diverge from the
    // reference, so it is refused here.
    if (!m->is_float) {
        auto pair_ok = [](const unsigned char *w, size_t bytes) {
            const signed char *q = reinterpret_cast<const signed char *>(w);
            for (size_t i = 0; i + 1 < bytes; i += 2) {
                const int a = q[i], b = q[i + 1];
                if ((a >= 0) == (b >= 0) && 255 * (abs(a) + abs(b)) > 32767) return false;
            }
            return true;
        };
        if (!pair_ok(wA->data, wA->size) || !pair_ok(wB->data, wB->size) || !pair_ok(wBrec->data, wBrec->size)) {
            set_error("model: int8 weights violate the pair constraint |w0|+|w1| <= 128 (maddubs would saturate in the reference; the exact integer GEMV would differ)");
            return -1;
        }
    }
    // geometry of the kernel that will consume the image
    const bool is_float = m->is_float != 0;
    const int nwc = is_float ? F_NWC : NWC, gpw = NGRP / nwc, kparts = is_float ? F_KPARTS : KPARTS, nwb = 6 * kparts;
    std::vector<int> cost(NGRP), order(NGRP);
    for (int g = 0; g < NGRP; g++) cost[g] = (int)(rowsA[g].size() + rowsA[NGRP + g].size() + rowsA[2 * NGRP + g].size());
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return cost[a] > cost[b]; });
    std::vector<std::vector<int>> grp(nwc);
    std::vector<int> load(nwc, 0);
    if (!is_float) {
        // The compute warps do not carry the same load besides GRU_A: warps < 6*KPARTS also walk a (row group, K part) of the dense GRU_B
        // input GEMV (blocks counted like GRU_A's), the NFIN warps from FIN0 on finish GRU_B (worth about `fin` blocks).  Starting the LPT from these
        // loads hands the heavier neuron groups to the warps with less GRU_B work.
        const int wgt = 1, fin = 48;                             // measured: 18.9 -> 18.6 ms per 1600 samples at 4096 streams (profiles/r02v_lpt.txt)
        for (int w = 0; w < nwc; w++) {
            if (w < nwb) load[w] += wgt * (int)(rowsB[w / kparts].size() / kparts);
            if (w >= FIN0) load[w] += fin;
        }
    }
    for (int g : order) {
        int best = -1;
        for (int w = 0; w < nwc; w++) if ((int)grp[w].size() < gpw && (best < 0 || load[w] < load[best])) best = w;
        grp[best].push_back(g); load[best] += cost[g];
    }

    // ---------------- SMEM layout ----------------
    // unit of the weight arrays: int8 flavour = quad (4 blocks, one MMA), float flavour = block (lists padded to even length)
    SmemLayout &L = m->L;
    auto padded = [is_float](size_t n) { return is_float ? (uint32_t)((n + 1) & ~size_t(1)) : (uint32_t)((n + 3) / 4); };
    uint32_t nA_pad = 0, nB_pad = 0;
    for (int w = 0; w < nwc; w++) for (int s = 0; s < gpw; s++) for (int q = 0; q < 3; q++) nA_pad += padded(rowsA[q * NGRP + grp[w][s]].size());
    // GRU_B input GEMV: warp (rg, part) takes a contiguous KPARTS-th of the row group's block list
    std::vector<std::array<uint32_t, 2>> dirB_h(nwb);
    auto part_lo = [is_float, kparts](size_t n, int k) { return is_float ? (k == 0 ? (size_t)0 : n) : (n * k + kparts - 1) / kparts; };
    for (int rg = 0; rg < 6; rg++) {
        size_t n = rowsB[rg].size();
        for (int k = 0; k < kparts; k++) {
            dirB_h[rg * kparts + k][1] = padded(part_lo(n, k + 1) - part_lo(n, k));
            nB_pad += dirB_h[rg * kparts + k][1];
        }
    }
    const ImageMap M = is_float ? map_f32(G) : map_int8(G);
    // int8 flavour: the dual_fc rows of the upper tree levels sit right in front of the variable arrays; keep as many (64, 32, 16,
    // 8) as the model's block lists leave room for
    int fcw_nodes = FCW_SMEM_NODES;
    if (const char *e = getenv("LPCNET_B200_FCW_NODES")) { const int v = atoi(e); if (v == 8 || v == 16 || v == 32) fcw_nodes = v; }   // (tests)
    for (;; fcw_nodes /= 2) {
        uint32_t off = M.sm_image + (is_float ? M.var : M.fcw + align_up((uint32_t)fcw_nodes * FCW_ROW * 4, 128));
        auto take = [&](uint32_t bytes, uint32_t align = 16) { off = align_up(off, align); uint32_t o = off; off += bytes; return o; };
        // readable slack behind every array: the pipelined GEMVs prefetch past the list end (values never used)
        const uint32_t unit_w = is_float ? img_blk : QUAD_BYTES, unit_m = is_float ? 2 : QUAD_META_BYTES, slack_w = is_float ? 2 : 4, slack_m = is_float ? 4 : 6;
        L.wA = take((nA_pad + slack_w) * unit_w, 128);
        L.metaA = take((nA_pad + slack_m) * unit_m);
        L.wB = take((nB_pad + slack_w) * unit_w, 128);
        L.metaB = take((nB_pad + slack_m) * unit_m);
        L.wBrecF = is_float ? take(3 * NB * NB * 4, 16) : 0;
        L.total_bytes = align_up(off, 128);
        if (sample_kernel_smem_ok(L.total_bytes) || is_float || fcw_nodes <= 8) break;
    }
    L.sm_image = M.sm_image;
    L.image_bytes = L.total_bytes - M.sm_image;
    L.nblkA_padded = nA_pad; L.nblkB_padded = nB_pad;
    if (!sample_kernel_smem_ok(L.total_bytes)) { set_error("model: %u bytes of shared memory needed, more than one SM offers", L.total_bytes); return -1; }

    // ---------------- build the image ----------------
    std::vector<uint8_t> img(L.image_bytes, 0);
    auto put_block = [is_float](uint8_t *dst, const unsigned char *src) {
        if (!is_float) { memcpy(dst, src, 32); return; }
        const float *f = reinterpret_cast<const float *>(src);          // [4 in][8 out] fp32 -> fp16, same order
        __half *h = reinterpret_cast<__half *>(dst);
        for (int i = 0; i < 32; i++) h[i] = __float2half_rn(f[i]);
    };
    const uint32_t oWA = L.wA - M.sm_image, oMA = L.metaA - M.sm_image, oWB = L.wB - M.sm_image, oMB = L.metaB - M.sm_image;
    // int8 flavour: write one block list as quads.  Any order of the blocks gives the same integer sum, so the blocks are
    // dealt into quads such that the four slots of a quad have column blocks of different (c & 3) classes whenever the
    // list allows it (the four LDS.128 of a quarter-warp then hit disjoint bank groups, see xs_offset()).  Empty slots
    // keep zero weights and point at a column block of an unused class.
    auto put_quads = [&](const Blk *lst, size_t n, uint32_t q0, uint32_t owq, uint32_t omq) {
        std::vector<int> bucket[4];
        for (size_t j = 0; j < n; j++) bucket[(lst[j].pos / 4) & 3].push_back((int)j);
        const uint32_t nq = (uint32_t)((n + 3) / 4);
        size_t left = n;
        for (uint32_t q = 0; q < nq; q++) {
            std::array<int, 4> pick = {-1, -1, -1, -1};
            bool used[4] = {false, false, false, false};
            int filled = 0;
            const size_t later = (size_t)(nq - 1 - q) * 4;                // capacity of the quads after this one
            const int need = left > later ? (int)(left - later) : 0;      // blocks this quad must take
            int ord[4] = {0, 1, 2, 3};
            std::stable_sort(ord, ord + 4, [&](int a, int b) { return bucket[a].size() > bucket[b].size(); });
            for (int k : ord)                                             // one block per class, largest classes first
                if (!bucket[k].empty()) { pick[filled++] = bucket[k].back(); bucket[k].pop_back(); used[k] = true; left--; }
            for (int k : ord)                                             // repeats only when the list forces them
                while (filled < need && !bucket[k].empty()) { pick[filled++] = bucket[k].back(); bucket[k].pop_back(); left--; }
            uint8_t *wq = &img[owq + (size_t)(q0 + q) * QUAD_BYTES];
            uint16_t *mq = reinterpret_cast<uint16_t *>(&img[omq + (size_t)(q0 + q) * QUAD_META_BYTES]);
            for (int t = 0; t < 4; t++) {
                if (pick[t] >= 0) {
                    const unsigned char *src = lst[pick[t]].w;                       // [8 out][4 in] int8
                    for (int o = 0; o < 8; o++) memcpy(wq + o * 16 + t * 4, src + o * 4, 4);
                    mq[t] = (uint16_t)xs_offset((uint32_t)lst[pick[t]].pos / 4, 0);
                } else {
                    int k = 0; while (k < 3 && used[k]) k++;
                    used[k] = true;
                    mq[t] = (uint16_t)xs_offset((uint32_t)k, 0);
                }
            }
        }
    };
    uint16_t *metaA = reinterpret_cast<uint16_t *>(&img[oMA]);
    float *parA = reinterpret_cast<float *>(&img[M.parA]);
    uint32_t *dirA = reinterpret_cast<uint32_t *>(&img[M.dirA]);
    uint32_t *grpA = reinterpret_cast<uint32_t *>(&img[M.grpA]);
    uint32_t blk = 0;
    // order of the lists in memory.  float flavour: (warp, slot, gate z r h).  int8 flavour: per warp the r and h lists of
    // all its slots first (r0 h0 r1 h1 ...: one contiguous quad stream for the GEMVs that precede the reset gate), then
    // the z lists (z0 z1 ...): the pipelined loader of the kernel runs across list boundaries.
    for (int w = 0; w < nwc; w++) {
        std::vector<std::pair<int, int>> seq;    // (slot, gate)
        if (is_float) { for (int s = 0; s < gpw; s++) for (int q = 0; q < 3; q++) seq.push_back({s, q}); }
        else { for (int s = 0; s < gpw; s++) { seq.push_back({s, 1}); seq.push_back({s, 2}); } for (int s = 0; s < gpw; s++) seq.push_back({s, 0}); }
        for (auto sq : seq) {
            const int s = sq.first, q = sq.second, g = grp[w][s];
            grpA[w * gpw + s] = (uint32_t)g;
            const auto &lst = rowsA[q * NGRP + g];
            uint32_t np = padded(lst.size());
            dirA[((w * gpw + s) * 3 + q) * 2 + 0] = blk;
            dirA[((w * gpw + s) * 3 + q) * 2 + 1] = np;
            if (is_float) {
                for (size_t j = 0; j < lst.size(); j++) {
                    put_block(&img[oWA + (size_t)(blk + j) * img_blk], lst[j].w);
                    metaA[blk + j] = (uint16_t)(lst[j].pos * 128);
                }
            } else put_quads(lst.data(), lst.size(), blk, oWA, oMA);
            blk += np;    // padding stays all-zero (weights 0, x row 0): contributes exactly 0
            float *pp = &parA[((w * gpw + s) * 3 + q) * 16];
            for (int i = 0; i < 8; i++) {
                pp[i] = (is_float ? ga_bias : ga_subias)[3 * NA + q * NA + 8 * g + i];   // recurrent (su-)bias (nnet.c:425-430)
                pp[8 + i] = ga_diag[q * NA + 8 * g + i];
            }
        }
    }
    uint16_t *metaB = reinterpret_cast<uint16_t *>(&img[oMB]);
    uint32_t *dirB = reinterpret_cast<uint32_t *>(&img[M.dirB]);
    const uint32_t quadsA_total = blk;
    blk = 0;
    for (int rg = 0; rg < 6; rg++) {
        const auto &lst = rowsB[rg];
        for (int k = 0; k < kparts; k++) {
            size_t b0 = part_lo(lst.size(), k), b1 = part_lo(lst.size(), k + 1);
            dirB[(rg * kparts + k) * 2 + 0] = blk;
            dirB[(rg * kparts + k) * 2 + 1] = dirB_h[rg * kparts + k][1];
            if (is_float) {
                for (size_t j = b0; j < b1; j++) {
                    put_block(&img[oWB + (size_t)(blk + (j - b0)) * img_blk], lst[j].w);
                    metaB[blk + (j - b0)] = (uint16_t)(lst[j].pos * 128);
                }
            } else put_quads(lst.data() + b0, b1 - b0, blk, oWB, oMB);
            blk += dirB_h[rg * kparts + k][1];
        }
    }
    if (!is_float) {
        // the int8 kernel keeps each compute warp's quads in tensor memory: 2 columns per quad, 128 columns per warp (sample_kernel.cu)
        for (int w = 0; w < nwc; w++) {
            const uint32_t firstA = dirA[((w * gpw + 0) * 3 + 1) * 2], lastA = w + 1 < nwc ? dirA[(((w + 1) * gpw + 0) * 3 + 1) * 2] : quadsA_total;
            const uint32_t nb = w < 6 * kparts ? dirB[w * 2 + 1] : 0;
            const uint32_t room = 128 - 8 * (uint32_t)gpw;          // the last 8*gpw columns hold the parked fp32 state, 2 tail quads follow the streams
            if (2 * ((lastA - firstA) + nb + 2) > room) {
                set_error("model: compute warp %d walks %u + %u quads, more than its %u tensor-memory columns hold", w, lastA - firstA, nb, room);
                return -1;
            }
        }
    }
    if (is_float) memcpy(&img[L.wBrecF - M.sm_image], wBrec->data, 3 * NB * NB * 4);    // float [in 16][out 48] (sgemv_accum16 layout)
    else memcpy(&img[M.wBrec], wBrec->data, 3 * NB * NB);
    {
        float *pb = reinterpret_cast<float *>(&img[M.parB]);
        for (int i = 0; i < 6 * NB; i++) pb[i] = (is_float ? gb_bias : gb_subias)[i];   // nnet.c:346-360 (USE_SU_BIAS only with DOT_PROD)
    }
    if (is_float) memcpy(&img[M.rcp], kRcpTable, sizeof(kRcpTable));
    else {
        uint32_t *r32 = reinterpret_cast<uint32_t *>(&img[M.rcp]);
        for (int k = 0; k < 2048; k++) r32[k] = 0x3f000000u + ((uint32_t)kRcpTable[k] << 11) + 0x3f800000u;
    }
    {
        float *lg = reinterpret_cast<float *>(&img[M.logit]);
        for (int i = 0; i < 256; i++) {                                   // lpcnet.c:188-191 (host libm, double log)
            float prob = .025f + .95f * i / 255.f;
            lg[i] = -log((1 - prob) / prob);
        }
        float *u2l = reinterpret_cast<float *>(&img[M.u2l]);
        for (int i = 0; i < 256; i++) {                                   // ulaw2lin, common.h:37-45 (double exp)
            float u = (float)i, s, scale_1 = 32768.f / 255.f;
            u = u - 128.f; s = u >= 0.f ? 1.f : -1.f; u = fabs(u);
            u2l[i] = s * scale_1 * (exp(u / 128. * 5.5451774445f) - 1);
        }
        hm.fc_rows.resize(256 * FCW_ROW);                                 // node i: 32 weights, bias[2], factor[2] (nnet.c:186-211)
        for (int i = 0; i < 256; i++) {
            float *r = &hm.fc_rows[(size_t)i * FCW_ROW];
            for (int j = 0; j < 32; j++) r[j] = fc_w[i * 32 + j];
            r[32] = fc_b[i]; r[33] = fc_b[256 + i]; r[34] = fc_f[i]; r[35] = fc_f[256 + i];
        }
        if (!is_float) {
            memcpy(&img[M.fcw], hm.fc_rows.data(), (size_t)fcw_nodes * FCW_ROW * 4);
            *reinterpret_cast<uint32_t *>(&img[G.im_fcwn]) = (uint32_t)fcw_nodes;
        }
        else { memcpy(&img[M.fcb], fc_b, 512 * 4); memcpy(&img[M.fcf], fc_f, 512 * 4); }
    }

    // Range proof for the conversion-free rounding of the GRU_A accumulators (devmath.cuh, acc_init_t): with |h| <= 1 and
    // the conditioning vector in [-1, 1] (tanh outputs of feature_dense2), every float that enters the accumulator and
    // every accumulator value is bounded by   (|bias| + |diag| + |gru_a_dense_feature row| + 3 max|E|) * 16256 + 255 * sum|w|.
    if (!is_float) {
        double cmax = 0, emax = 0, bmax = 0, dmax = 0, smax = 0;
        for (int i = 0; i < 3 * NA; i++) {
            double c = fabs(gad_b[i]);
            for (int j = 0; j < COND; j++) c += fabs(gad_w[(size_t)j * 3 * NA + i]);
            cmax = std::max(cmax, c);
            bmax = std::max(bmax, (double)fabs(ga_subias[3 * NA + i]));
            dmax = std::max(dmax, (double)fabs(ga_diag[i]));
        }
        for (size_t i = 0; i < (size_t)256 * 3 * NA; i++)
            emax = std::max(emax, (double)std::max(fabs(emb_sig[i]), std::max(fabs(emb_pred[i]), fabs(emb_exc[i]))));
        for (int rg = 0; rg < 3 * NGRP; rg++) {
            double rs[8] = {0};
            for (auto &b : rowsA[rg]) for (int o = 0; o < 8; o++) for (int i = 0; i < 4; i++) rs[o] += abs((int)(signed char)b.w[o * 4 + i]);
            for (int o = 0; o < 8; o++) smax = std::max(smax, rs[o]);
        }
        const double bound = (bmax + dmax + cmax + 3 * emax) * 1.01 * (128.0 * 127.0) + 255.0 * smax + 2;
        m->fast_cvt = bound < 4194304.0 * 0.99;
    }
    // ---------------- float flavour: second image for the neuron-per-lane kernel (small batches) ----------------
    if (is_float) {
        SmemLayout &Ln = m->Ln;
        memset(&Ln, 0, sizeof(Ln));
        uint32_t o = G.fn_image + G.fni_var;
        auto takeN = [&](uint32_t bytes, uint32_t align) { o = align_up(o, align); uint32_t r = o; o += bytes; return r; };
        Ln.wA = takeN((uint32_t)(nblkA + 4) * 64, 128);          // (+4 blocks / +8 meta entries of slack: the pipelined chains read ahead)
        Ln.metaA = takeN((uint32_t)(nblkA + 8) * 2, 16);
        Ln.wB = takeN((uint32_t)(nblkB + 4) * 64, 128);
        Ln.metaB = takeN((uint32_t)(nblkB + 8) * 2, 16);
        Ln.total_bytes = align_up(o, 128);
        Ln.sm_image = G.fn_image;
        Ln.image_bytes = Ln.total_bytes - G.fn_image;
        Ln.nblkA_padded = (uint32_t)nblkA; Ln.nblkB_padded = (uint32_t)nblkB;
        if (!sample_kernel_smem_ok(Ln.total_bytes)) { set_error("model: %u bytes of shared memory needed by the small-batch float kernel", Ln.total_bytes); return -1; }
        std::vector<uint8_t> &im = hm.img_n;
        im.assign(Ln.image_bytes, 0);
        memcpy(&im[G.fni_rcp], kRcpTable, sizeof(kRcpTable));
        memcpy(&im[G.fni_logit], &img[M.logit], 256 * 4);
        memcpy(&im[G.fni_u2l], &img[M.u2l], 256 * 4);
        memcpy(&im[G.fni_fcw], hm.fc_rows.data(), (size_t)256 * FCW_ROW * 4);
        // lanes: groups sorted by the length of their longest (candidate-gate) list so that the four groups sharing a warp are alike
        std::vector<int> ord(NGRP);
        std::iota(ord.begin(), ord.end(), 0);
        std::stable_sort(ord.begin(), ord.end(), [&](int a, int b) { return rowsA[2 * NGRP + a].size() > rowsA[2 * NGRP + b].size(); });
        uint16_t *neur = reinterpret_cast<uint16_t *>(&im[G.fni_neur]);
        for (int l = 0; l < NA; l++) neur[l] = (uint16_t)(8 * ord[l / 8] + (l & 7));
        // blocks: [8 rows][4 cols] fp16 (the blob holds [4 cols][8 rows] fp32), lists in blob order (gate, group), idx order inside
        auto put_t = [](uint8_t *dst, const unsigned char *src) {
            const float *f = reinterpret_cast<const float *>(src);
            __half *h = reinterpret_cast<__half *>(dst);
            for (int r = 0; r < 8; r++) for (int c = 0; c < 4; c++) h[r * 4 + c] = __float2half_rn(f[c * 8 + r]);
        };
        uint32_t *dA = reinterpret_cast<uint32_t *>(&im[G.fni_dira]);
        uint16_t *mA = reinterpret_cast<uint16_t *>(&im[Ln.metaA - G.fn_image]);
        uint32_t bk = 0;
        for (int g = 0; g < NGRP; g++) for (int q = 0; q < 3; q++) {
            const auto &lst = rowsA[q * NGRP + g];
            dA[(g * 3 + q) * 2 + 0] = bk; dA[(g * 3 + q) * 2 + 1] = (uint32_t)lst.size();
            for (size_t j = 0; j < lst.size(); j++) { put_t(&im[Ln.wA - G.fn_image + (size_t)(bk + j) * 64], lst[j].w); mA[bk + j] = (uint16_t)(lst[j].pos * 4); }
            bk += (uint32_t)lst.size();
        }
        float *pa = reinterpret_cast<float *>(&im[G.fni_para]);
        for (int q = 0; q < 3; q++) for (int j = 0; j < NA; j++) {
            pa[(q * 2 + 0) * NA + j] = ga_bias[3 * NA + q * NA + j];            // recurrent bias (nnet.c:425-430)
            pa[(q * 2 + 1) * NA + j] = ga_diag[q * NA + j];
        }
        uint32_t *dB = reinterpret_cast<uint32_t *>(&im[G.fni_dirb]);
        uint16_t *mB = reinterpret_cast<uint16_t *>(&im[Ln.metaB - G.fn_image]);
        bk = 0;
        for (int rg = 0; rg < 6; rg++) {
            const auto &lst = rowsB[rg];
            dB[rg * 2 + 0] = bk; dB[rg * 2 + 1] = (uint32_t)lst.size();
            for (size_t j = 0; j < lst.size(); j++) { put_t(&im[Ln.wB - G.fn_image + (size_t)(bk + j) * 64], lst[j].w); mB[bk + j] = (uint16_t)(lst[j].pos * 4); }
            bk += (uint32_t)lst.size();
        }
        Ln.wBrecF = 1;
        for (int rg = 0; rg < 6; rg++) { if (rowsB[rg].size() != NA / 4) Ln.wBrecF = 0; else for (size_t j = 0; j < rowsB[rg].size(); j++) if (rowsB[rg][j].pos != (int)(4 * j)) Ln.wBrecF = 0; }
        memcpy(&im[G.fni_parb], gb_bias, 6 * NB * 4);
        memcpy(&im[G.fni_wbrec], wBrec->data, 3 * NB * NB * 4);
    }
    hm.embed_pitch = embed_pitch; hm.conv1_w = conv1_w; hm.conv1_b = conv1_b; hm.conv2_w = conv2_w; hm.conv2_b = conv2_b;
    hm.dense1_w = dense1_w; hm.dense1_b = dense1_b; hm.dense2_w = dense2_w; hm.dense2_b = dense2_b;
    hm.gad_w = gad_w; hm.gad_b = gad_b; hm.gbd_w = gbd_w; hm.gbd_b = gbd_b;
    hm.emb_sig = emb_sig; hm.emb_pred = emb_pred; hm.emb_exc = emb_exc;
    hm.img.swap(img);
    // algorithmic bytes per synthesized sample (SURVEY.md 8d)
    {   // float flavour: weights are read as fp16 (64 B per block); recurrent GRU_B weights as stored
        const long bb = is_float ? 64 : 32, wrec = is_float ? 3L * NB * NB * 4 : 3L * NB * NB;
        m->algo_bytes_sparse = bb * nblkA + 4L * (3 * NGRP + nblkA);
        m->algo_bytes_total = m->algo_bytes_sparse + 3 * NA * 4 /*diag*/ + 3 * NA * 4 /*bias*/ + 3 * 3 * NA * 4 /*3 embedding rows*/
                            + 3 * NA * 4 /*gru_a_condition*/ + bb * nblkB + 4L * (6 + nblkB) + wrec + 6 * NB * 4 + 3 * NB * 4
                            + 8 * (2 * NB + 2 + 2) * 4 + 32;
    }
    return 0;
}

// Test hook (no CUDA needed): build the shared-memory image on the host and hand it out.
int debug_build_image(const unsigned char *blob, int len, unsigned char *out, size_t cap, SmemLayout *L, Geom *g, int *fast_cvt, int *is_float)
{
    DeviceModel m; HostModel hm;
    if (build_host_model(&m, hm, blob, len, nullptr) != 0) return -1;
    *L = m.L; *g = make_geom(m.na); *fast_cvt = m.fast_cvt; *is_float = m.is_float;
    if (hm.img.size() > cap) { set_error("debug image: buffer too small"); return -1; }
    memcpy(out, hm.img.data(), hm.img.size());
    return (int)hm.img.size();
}

// Same for the second image of float models (neuron-per-lane kernel).
int debug_build_image_n(const unsigned char *blob, int len, unsigned char *out, size_t cap, SmemLayout *L, Geom *g)
{
    DeviceModel m; HostModel hm;
    if (build_host_model(&m, hm, blob, len, nullptr) != 0) return -1;
    if (!m.is_float) { set_error("debug image: not a float blob"); return -1; }
    *L = m.Ln; *g = make_geom(m.na);
    if (hm.img_n.size() > cap) { set_error("debug image: buffer too small"); return -1; }
    memcpy(out, hm.img_n.data(), hm.img_n.size());
    return (int)hm.img_n.size();
}

// DCT / FFT tables exactly as src/dump_lpcnet_tables.c:53,87-93 and kiss_fft.c:406-421 build them (host libm); shared with the
// analysis side (enc_kernels.cu)
void build_fft_tables(std::vector<float> &dct, std::vector<float> &tw, std::vector<int16_t> &br)
{
    static const int factors[8] = {5, 64, 4, 16, 4, 4, 4, 1};
    dct.assign(NB_BANDS * NB_BANDS, 0.f); tw.assign(2 * WINDOW_SIZE, 0.f); br.assign(WINDOW_SIZE, 0);
    for (int i = 0; i < NB_BANDS; i++) for (int j = 0; j < NB_BANDS; j++) {
        dct[i * NB_BANDS + j] = cos((i + .5) * j * M_PI / NB_BANDS);
        if (j == 0) dct[i * NB_BANDS + j] *= sqrt(.5);
    }
    for (int i = 0; i < WINDOW_SIZE; i++) {
        const double pi = 3.14159265358979323846264338327;
        double phase = (-2 * pi / WINDOW_SIZE) * i;
        tw[2 * i] = (float)cos(phase); tw[2 * i + 1] = (float)sin(phase);
    }
    // digit-reversal permutation of the 5x4x4x4 decomposition (compute_bitrev_table, kiss_fft.c:314-345)
    struct Rec { static void go(int Fout, int16_t *f, int fstride, const int *fac) {
        int p = fac[0], mm = fac[1];
        if (mm == 1) { for (int j = 0; j < p; j++) { *f = (int16_t)(Fout + j); f += fstride; } }
        else { for (int j = 0; j < p; j++) { go(Fout, f, fstride * p, fac + 2); f += fstride; Fout += mm; } }
    } };
    Rec::go(0, br.data(), 1, factors);
}

int model_load(DeviceModel *m, const unsigned char *blob, int len, const ModelConfig *cfg)
{
    HostModel hm;
    if (build_host_model(m, hm, blob, len, cfg) != 0) return -1;
    const int NA = m->na;
    const float lpc_gamma = m->cfg.lpc_gamma;
    const std::vector<uint8_t> &img = hm.img;
    const float *embed_pitch = hm.embed_pitch, *conv1_w = hm.conv1_w, *conv1_b = hm.conv1_b, *conv2_w = hm.conv2_w, *conv2_b = hm.conv2_b;
    const float *dense1_w = hm.dense1_w, *dense1_b = hm.dense1_b, *dense2_w = hm.dense2_w, *dense2_b = hm.dense2_b;
    const float *gad_w = hm.gad_w, *gad_b = hm.gad_b, *gbd_w = hm.gbd_w, *gbd_b = hm.gbd_b;
    const float *emb_sig = hm.emb_sig, *emb_pred = hm.emb_pred, *emb_exc = hm.emb_exc;
    // ---------------- device copies ----------------
    bool ok = true;
#define UP(field, src, count) ok = ok && ((m->field = to_device(src, (size_t)(count))) != nullptr);
    UP(image, img.data(), img.size())
    if (m->is_float) { UP(image_n, hm.img_n.data(), hm.img_n.size()) }
    UP(emb_sig, emb_sig, 256 * 3 * NA) UP(emb_pred, emb_pred, 256 * 3 * NA) UP(emb_exc, emb_exc, 256 * 3 * NA)
    UP(fcw, hm.fc_rows.data(), hm.fc_rows.size())
    UP(embed_pitch, embed_pitch, 256 * PITCH_EMBED)
    UP(conv1_w, conv1_w, 3 * FRAME_IN * COND) UP(conv1_b, conv1_b, COND)
    UP(conv2_w, conv2_w, 3 * COND * COND) UP(conv2_b, conv2_b, COND)
    UP(dense1_w, dense1_w, COND * COND) UP(dense1_b, dense1_b, COND)
    UP(dense2_w, dense2_w, COND * COND) UP(dense2_b, dense2_b, COND)
    UP(gad_w, gad_w, COND * 3 * NA) UP(gad_b, gad_b, 3 * NA)
    UP(gbd_w, gbd_w, COND * 3 * NB) UP(gbd_b, gbd_b, 3 * NB)
    UP(rcp16, kRcpTable, 2048)
    {
        std::vector<float> dct, tw;
        std::vector<int16_t> br;
        build_fft_tables(dct, tw, br);
        UP(dct, dct.data(), dct.size()) UP(twiddles, tw.data(), tw.size()) UP(bitrev, br.data(), br.size())
        float gp[LPC_ORDER]; float gi = lpc_gamma;
        for (int i = 0; i < LPC_ORDER; i++) { gp[i] = gi; gi *= lpc_gamma; }   // freq.c:299-308
        UP(gamma_pow, gp, LPC_ORDER)
        float pp[64];
        for (int k = 0; k < 64; k++) pp[k] = pow(2.f, k / 21.) * 32;            // lpcnet_dec.c:124 (PITCH_MIN_PERIOD 32)
        UP(pitch_pow, pp, 64)
    }
#undef UP
    if (!ok) { set_error("model: device allocation/copy failed: %s", cudaGetErrorString(cudaGetLastError())); model_free(m); return -1; }

    return 0;
}

void model_free(DeviceModel *m)
{
    void *ptrs[] = {m->image, m->image_n, m->fcw, m->emb_sig, m->emb_pred, m->emb_exc, m->embed_pitch, m->conv1_w, m->conv1_b, m->conv2_w, m->conv2_b,
                    m->dense1_w, m->dense1_b, m->dense2_w, m->dense2_b, m->gad_w, m->gad_b, m->gbd_w, m->gbd_b, m->rcp16, m->dct,
                    m->twiddles, m->bitrev, m->gamma_pow, m->pitch_pow, m->codebooks};
    for (void *p : ptrs) if (p) cudaFree(p);
    memset(m, 0, sizeof(*m));
}

}  // namespace lpcnet_b200
