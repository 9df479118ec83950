/* lpcnet_oracle.c — CPU RESTATEMENT of the LPCNet synthesis hot path.
 *
 * >>> TEST INFRASTRUCTURE.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may use this
 * >>> file.  It is never linked into liblpcnet_b200.so and the product path never falls back to it.
 *
 * Scalar, portable C (no intrinsics) that reproduces, operation for operation, what the reference computes
 * when built as pinned oracle "A" (gcc -O2 -mavx2 -mfma -ffp-contract=off, int8 DOT_PROD path) or "B"
 * (A + -DDISABLE_DOT_PROD, float path).  Explicit fmaf() appears exactly where the reference has
 * _mm256_fmadd_ps; everything else is separate IEEE mul/add (compile THIS file with -ffp-contract=off).
 * `_mm256_rcp_ps` is emulated from a 2048-entry table captured on the host that produced the goldens
 * (oracle/capture_rcp.py), so the restatement gives identical results on any CPU.
 *
 * Parity pin: tests/test_oracle_vs_ref.py checks this file bit-for-bit against the compiled reference
 * (oracle/_ref, built from /root/reference by oracle/Makefile) and against tests/golden/.
 *
 * Reference map (file:line under /root/reference):
 *   blob records .................. src/nnet.h:41-61, src/parse_lpcnet_weights.c:37-77
 *   layer validation .............. src/parse_lpcnet_weights.c:90-221
 *   kiss99 ........................ src/kiss99.c:32-81
 *   u-law ......................... src/common.h:18-58
 *   tanh/sigmoid (AVX Pade+rcp) ... src/vec_avx.h:393-450
 *   vector_ps_to_epi8 ............. src/vec_avx.h:321-336
 *   sgemv_accum16 ................. src/vec_avx.h:618-643
 *   sgemv_accum8x4 (int8) ......... src/vec_avx.h:690-755
 *   sparse_sgemv_accum8x4 int8 .... src/vec_avx.h:790-858      float: src/vec_avx.h:865-903
 *   dense / conv1d / embedding .... src/nnet.c:122-135,452-481
 *   compute_gru_a_input ........... src/nnet.c:484-491
 *   compute_sparse_gru ............ src/nnet.c:410-448
 *   compute_gruB .................. src/nnet.c:326-372
 *   sample_mdense ................. src/nnet.c:163-214
 *   run_frame_network ............. src/lpcnet.c:82-120
 *   run_sample_network ............ src/lpcnet.c:146-167
 *   lpcnet_synthesize_tail_impl ... src/lpcnet.c:235-271
 *   lpcnet_reset / lpcnet_init .... src/lpcnet.c:174-200
 *   lpc_from_cepstrum & friends ... src/freq.c:86-127,202-215,230-240,256-320
 *   320-point FFT ................. src/kiss_fft.c:101-170,232-311,518-587 ; tables src/dump_lpcnet_tables.c:53,87-93
 *   decode_packet ................. src/lpcnet_dec.c:59-155, src/common.c:37-65
 */
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <pthread.h>

#define NB_FEATURES 20
#define NB_TOTAL_FEATURES 36
#define NB_BANDS 18
#define LPC_ORDER 16
#define FRAME_SIZE 160
#define WINDOW_SIZE 320
#define FREQ_SIZE 161
#define N_A_MAX 384     /* largest GRU_A the port handles; the actual size comes from the blob (OModel.na) */
#define N_B 16
#define COND 128
#define PITCH_EMBED 64
#define FRAME_IN (NB_FEATURES + PITCH_EMBED)
#define FEATURES_DELAY_MAX 2   /* FEATURES_DELAY is a per-model value 0..2 (OModel.features_delay), dump_lpcnet.py:323-329 */
#define MAX_FEATURE_BUFFER_SIZE 4   /* lpcnet_private.h:26 */
#define PREEMPH 0.85f

typedef struct { float r, i; } cpx;

typedef struct {
    int is_float;                 /* 0: oracle A (int8), 1: oracle B (float) */
    int na;                       /* GRU_A units (from the blob) */
    int features_delay;           /* FEATURES_DELAY of the generated nnet_data.h */
    int end2end;                  /* END2END of the generated nnet_data.h */
    float lpc_gamma;
    /* frame network */
    const float *embed_pitch;     /* [256][64] */
    const float *conv1_w, *conv1_b, *conv2_w, *conv2_b;
    const float *dense1_w, *dense1_b, *dense2_w, *dense2_b;
    const float *gad_w, *gad_b;   /* gru_a_dense_feature 128 -> 1152 */
    const float *gbd_w, *gbd_b;   /* gru_b_dense_feature 128 -> 48 */
    /* sample network */
    const float *emb_sig, *emb_pred, *emb_exc;    /* [256][1152] */
    const float *ga_bias, *ga_subias, *ga_diag;   /* [2][1152], [2][1152], [1152] */
    const void *ga_w; const int *ga_idx;
    const float *gb_bias, *gb_subias;             /* [2][48] */
    const void *gb_w; const int *gb_idx; const void *gb_rw;
    const float *fc_w, *fc_b, *fc_f;              /* [256][2][16], [2][256], [2][256] */
    /* tables */
    uint32_t rcp[2048];
    float logit[256];
    float ulaw2lin_tab[256];
    cpx tw[WINDOW_SIZE];
    int bitrev[WINDOW_SIZE];
    float dct[NB_BANDS * NB_BANDS];
    const float *cb1, *cb2, *cb3, *cbd4;          /* VQ codebooks (decoder only) */
    unsigned char *blob_copy;
    float *cb_copy;
} OModel;

typedef struct { uint32_t z, w, jsr, jcong; } kiss99;

typedef struct {
    const OModel *m;
    kiss99 rng;
    /* resettable part — mirrors struct LPCNetState (src/lpcnet_private.h:28-48) */
    float conv1_state[FRAME_IN * 2];
    float conv2_state[COND * 2];
    float gru_a_state[N_A_MAX];
    float gru_b_state[N_B];
    int last_exc;
    float last_sig[LPC_ORDER];
    float feature_buffer[NB_FEATURES * MAX_FEATURE_BUFFER_SIZE];
    int feature_buffer_fill;
    float old_lpc[FEATURES_DELAY_MAX][LPC_ORDER];
    float gru_a_condition[3 * N_A_MAX];
    float gru_b_condition[3 * N_B];
    int frame_count;
    float deemph_mem;
    float lpc[LPC_ORDER];
    float vq_mem[NB_BANDS];      /* LPCNetDecState.vq_mem */
    /* optional trace of the last synthesize call */
    int *trace_exc;              /* if non-NULL: exc index per generated sample */
    int32_t acc_peak;            /* int8: largest |GRU_A accumulator| (entry value or final sum) since the last reset */
} OState;

/* ------------------------------------------------------------------ blob ------------------------------------------------------------------ */
typedef struct { char head[4]; int version; int type; int size; int block_size; char name[44]; } WeightHead;

static const void *find_array(const unsigned char *data, int len, const char *name, int *size)
{
    while (len >= 64) {
        const WeightHead *h = (const WeightHead *)data;
        if (h->block_size < h->size || h->block_size > len - 64 || h->size < 0) return NULL;
        if (strncmp(h->name, name, 44) == 0) { *size = h->size; return data + 64; }
        data += 64 + h->block_size; len -= 64 + h->block_size;
    }
    return NULL;
}

static const void *need(const unsigned char *d, int len, const char *name, int size)
{
    int sz = -1;
    const void *p = find_array(d, len, name, &sz);
    if (!p || (size >= 0 && sz != size)) return NULL;
    return p;
}

/* find_idx_check (parse_lpcnet_weights.c:90-113) */
static const int *need_idx(const unsigned char *d, int len, const char *name, int nb_in, int nb_out, int *total_blocks)
{
    int sz = -1, remain;
    const int *idx = find_array(d, len, name, &sz), *p;
    *total_blocks = 0;
    if (!idx) return NULL;
    p = idx; remain = sz / 4;
    while (remain > 0) {
        int nb = *p++, i;
        if (remain < nb + 1) return NULL;
        for (i = 0; i < nb; i++) { int pos = *p++; if (pos + 3 >= nb_in || (pos & 3)) return NULL; }
        nb_out -= 8; remain -= nb + 1; *total_blocks += nb;
    }
    if (nb_out != 0) return NULL;
    return idx;
}

/* ------------------------------------------------------------------ tables ------------------------------------------------------------------ */
static void bitrev_rec(int Fout, int *f, int fstride, const int *factors)
{
    /* compute_bitrev_table (kiss_fft.c:314-345), in_stride == 1 */
    int p = factors[0], m = factors[1], j;
    if (m == 1) { for (j = 0; j < p; j++) { *f = Fout + j; f += fstride; } }
    else { for (j = 0; j < p; j++) { bitrev_rec(Fout, f, fstride * p, factors + 2); f += fstride; Fout += m; } }
}

static void build_tables(OModel *m)
{
    static const int factors[8] = {5, 64, 4, 16, 4, 4, 4, 1};   /* kf_factor(320) — lpcnet_tables.c:200 */
    int i, j;
    for (i = 0; i < WINDOW_SIZE; i++) {                       /* compute_twiddles kiss_fft.c:406-421 */
        const double pi = 3.14159265358979323846264338327;
        double phase = (-2 * pi / WINDOW_SIZE) * i;
        m->tw[i].r = (float)cos(phase); m->tw[i].i = (float)sin(phase);
    }
    bitrev_rec(0, m->bitrev, 1, factors);
    for (i = 0; i < NB_BANDS; i++) for (j = 0; j < NB_BANDS; j++) {   /* dump_lpcnet_tables.c:87-93 */
        m->dct[i * NB_BANDS + j] = cos((i + .5) * j * M_PI / NB_BANDS);
        if (j == 0) m->dct[i * NB_BANDS + j] *= sqrt(.5);
    }
    for (i = 0; i < 256; i++) {                                /* lpcnet.c:188-191 */
        float prob = .025f + .95f * i / 255.f;
        m->logit[i] = -log((1 - prob) / prob);
    }
    for (i = 0; i < 256; i++) {                                /* ulaw2lin common.h:37-45 */
        float u = (float)i, s, scale_1 = 32768.f / 255.f;
        u = u - 128.f; s = u >= 0.f ? 1.f : -1.f; u = fabs(u);
        m->ulaw2lin_tab[i] = s * scale_1 * (exp(u / 128. * 5.5451774445f) - 1);
    }
}

/* ------------------------------------------------------------------ scalar primitives ------------------------------------------------------------------ */
static inline float rcp_emul(const OModel *m, float x)
{
    union { float f; uint32_t u; } in, out;
    in.f = x;
    out.u = m->rcp[(in.u >> 12) & 0x7FF] - ((in.u & 0x7F800000u) - 0x3F800000u);
    return out.f;
}
static inline float minps(float a, float b) { return a < b ? a : b; }   /* _mm_min_ps(a,b): a<b ? a : b */
static inline float maxps(float a, float b) { return a > b ? a : b; }

static inline float tanh_a(const OModel *m, float x)       /* tanh8_approx vec_avx.h:393-411 */
{
    const float N0 = 952.52801514f, N1 = 96.39235687f, N2 = 0.60863042f;
    const float D0 = 952.72399902f, D1 = 413.36801147f, D2 = 11.88600922f;
    float X2 = x * x;
    float num = fmaf(fmaf(N2, X2, N1), X2, N0);
    float den = fmaf(fmaf(D2, X2, D1), X2, D0);
    num = num * x; den = rcp_emul(m, den); num = num * den;
    return maxps(-1.f, minps(1.f, num));
}
static inline float sigmoid_a(const OModel *m, float x)    /* sigmoid8_approx vec_avx.h:421-440 */
{
    const float N0 = 238.13200378f, N1 = 6.02452230f, N2 = 0.00950985f;
    const float D0 = 952.72399902f, D1 = 103.34200287f, D2 = 0.74287558f;
    float X2 = x * x;
    float num = fmaf(fmaf(N2, X2, N1), X2, N0);
    float den = fmaf(fmaf(D2, X2, D1), X2, D0);
    num = num * x; den = rcp_emul(m, den); num = fmaf(num, den, 0.5f);
    return maxps(0.f, minps(1.f, num));
}

static inline float log2_approx(float x)                   /* common.h:18-33 */
{
    int integer; float frac; union { float f; int i; } in;
    in.f = x; integer = (in.i >> 23) - 127; in.i -= integer << 23;
    frac = in.f - 1.5f;
    frac = -0.41445418f + frac * (0.95909232f + frac * (-0.33951290f + frac * 0.16541097f));
    return 1 + integer + frac;
}
static inline int lin2ulaw(float x)                        /* common.h:47-58 */
{
    float u, scale = 255.f / 32768.f; int s = x >= 0 ? 1 : -1;
    x = fabs(x);
    u = (s * (128 * (0.69315f * log2_approx(1 + scale * x)) / 5.5451774445f));
    u = 128 + u;
    if (u < 0) u = 0;
    if (u > 255) u = 255;
    return (int)floor(.5 + u);
}

static void kiss99_srand(kiss99 *t, const unsigned char *d, int n)   /* kiss99.c:32-57 */
{
    int i; uint32_t kiss99_rand(kiss99 *);
    t->z = 362436069; t->w = 521288629; t->jsr = 123456789; t->jcong = 380116160;
    for (i = 3; i < n; i += 4) { t->z ^= d[i - 3]; t->w ^= d[i - 2]; t->jsr ^= d[i - 1]; t->jcong ^= d[i]; kiss99_rand(t); }
    if (i - 3 < n) t->z ^= d[i - 3];
    if (i - 2 < n) t->w ^= d[i - 2];
    if (i - 1 < n) t->jsr ^= d[i - 1];
    if (t->z == 0 || t->z == 0x9068FFFF) t->z++;
    if (t->w == 0 || t->w == 0x464FFFFF) t->w++;
    if (t->jsr == 0) t->jsr++;
}
uint32_t kiss99_rand(kiss99 *t)                                      /* kiss99.c:59-81 */
{
    uint32_t znew = 36969 * (t->z & 0xFFFF) + (t->z >> 16), wnew = 18000 * (t->w & 0xFFFF) + (t->w >> 16);
    uint32_t mwc = (znew << 16) + wnew, shr3 = t->jsr ^ (t->jsr << 13), cong;
    shr3 ^= shr3 >> 17; shr3 ^= shr3 << 5; cong = 69069 * t->jcong + 1234567;
    t->z = znew; t->w = wnew; t->jsr = shr3; t->jcong = cong;
    return (mwc ^ cong) + shr3;
}

/* sgemv_accum16 (vec_avx.h:618-643): per output row an FMA chain over columns in ascending order */
static void sgemv_fma(float *out, const float *w, int rows, int cols, int col_stride, const float *x)
{
    int i, j;
    for (i = 0; i < rows; i++) { float y = out[i]; for (j = 0; j < cols; j++) y = fmaf(w[j * col_stride + i], x[j], y); out[i] = y; }
}
static void dense(const OModel *m, float *out, const float *w, const float *b, int nin, int nout, const float *in, int tanh_act)
{
    int i;
    for (i = 0; i < nout; i++) out[i] = b[i];
    sgemv_fma(out, w, nout, nin, nout, in);
    if (tanh_act) for (i = 0; i < nout; i++) out[i] = tanh_a(m, out[i]);
}
static void conv1d(const OModel *m, float *out, float *mem, const float *w, const float *b, int nin, int nout, const float *in)
{
    float tmp[3 * COND]; int i;                               /* nnet.c:452-470, kernel 3 */
    memcpy(tmp, mem, sizeof(float) * 2 * nin); memcpy(tmp + 2 * nin, in, sizeof(float) * nin);
    for (i = 0; i < nout; i++) out[i] = b[i];
    sgemv_fma(out, w, nout, 3 * nin, nout, tmp);
    for (i = 0; i < nout; i++) out[i] = tanh_a(m, out[i]);
    memcpy(mem, tmp + nin, sizeof(float) * 2 * nin);
}

static inline unsigned char quant_u8(float x)              /* vector_ps_to_epi8 vec_avx.h:321-336 */
{
    float xf = fmaf(x, 127.f, 127.f);
    long v = lrintf(xf);                                   /* cvtps_epi32: round-to-nearest-even (default mode) */
    if (v < 0) v = 0;
    if (v > 255) v = 255;
    return (unsigned char)v;
}

/* ------------------------------------------------------------------ FFT + LPC ------------------------------------------------------------------ */
#define CMUL(m_, a_, b_) do { (m_).r = (a_).r * (b_).r - (a_).i * (b_).i; (m_).i = (a_).r * (b_).i + (a_).i * (b_).r; } while (0)
#define CADD(r_, a_, b_) do { (r_).r = (a_).r + (b_).r; (r_).i = (a_).i + (b_).i; } while (0)
#define CSUB(r_, a_, b_) do { (r_).r = (a_).r - (b_).r; (r_).i = (a_).i - (b_).i; } while (0)

static void bfly4(cpx *Fout, int fstride, const cpx *twid, int m, int N, int mm)   /* kiss_fft.c:101-170 */
{
    int i, j;
    if (m == 1) {
        for (i = 0; i < N; i++) {
            cpx s0, s1;
            CSUB(s0, Fout[0], Fout[2]); CADD(Fout[0], Fout[0], Fout[2]);
            CADD(s1, Fout[1], Fout[3]); CSUB(Fout[2], Fout[0], s1); CADD(Fout[0], Fout[0], s1);
            CSUB(s1, Fout[1], Fout[3]);
            Fout[1].r = s0.r + s1.i; Fout[1].i = s0.i - s1.r;
            Fout[3].r = s0.r - s1.i; Fout[3].i = s0.i + s1.r;
            Fout += 4;
        }
    } else {
        cpx *beg = Fout; const int m2 = 2 * m, m3 = 3 * m;
        for (i = 0; i < N; i++) {
            const cpx *tw1 = twid, *tw2 = twid, *tw3 = twid;
            Fout = beg + i * mm;
            for (j = 0; j < m; j++) {
                cpx s[6];
                CMUL(s[0], Fout[m], *tw1); CMUL(s[1], Fout[m2], *tw2); CMUL(s[2], Fout[m3], *tw3);
                CSUB(s[5], Fout[0], s[1]); CADD(Fout[0], Fout[0], s[1]);
                CADD(s[3], s[0], s[2]); CSUB(s[4], s[0], s[2]);
                CSUB(Fout[m2], Fout[0], s[3]);
                tw1 += fstride; tw2 += fstride * 2; tw3 += fstride * 3;
                CADD(Fout[0], Fout[0], s[3]);
                Fout[m].r = s[5].r + s[4].i; Fout[m].i = s[5].i - s[4].r;
                Fout[m3].r = s[5].r - s[4].i; Fout[m3].i = s[5].i + s[4].r;
                ++Fout;
            }
        }
    }
}
static void bfly5(cpx *Fout, int fstride, const cpx *tw, int m, int N, int mm)   /* kiss_fft.c:232-311 */
{
    int i, u; cpx *beg = Fout;
    cpx ya = tw[fstride * m], yb = tw[fstride * 2 * m];
    for (i = 0; i < N; i++) {
        cpx *F0, *F1, *F2, *F3, *F4;
        Fout = beg + i * mm; F0 = Fout; F1 = F0 + m; F2 = F0 + 2 * m; F3 = F0 + 3 * m; F4 = F0 + 4 * m;
        for (u = 0; u < m; ++u) {
            cpx s[13];
            s[0] = *F0;
            CMUL(s[1], *F1, tw[u * fstride]); CMUL(s[2], *F2, tw[2 * u * fstride]);
            CMUL(s[3], *F3, tw[3 * u * fstride]); CMUL(s[4], *F4, tw[4 * u * fstride]);
            CADD(s[7], s[1], s[4]); CSUB(s[10], s[1], s[4]); CADD(s[8], s[2], s[3]); CSUB(s[9], s[2], s[3]);
            F0->r = F0->r + (s[7].r + s[8].r); F0->i = F0->i + (s[7].i + s[8].i);
            s[5].r = s[0].r + (s[7].r * ya.r + s[8].r * yb.r); s[5].i = s[0].i + (s[7].i * ya.r + s[8].i * yb.r);
            s[6].r = s[10].i * ya.i + s[9].i * yb.i; s[6].i = -(s[10].r * ya.i + s[9].r * yb.i);
            CSUB(*F1, s[5], s[6]); CADD(*F4, s[5], s[6]);
            s[11].r = s[0].r + (s[7].r * yb.r + s[8].r * ya.r); s[11].i = s[0].i + (s[7].i * yb.r + s[8].i * ya.r);
            s[12].r = s[9].i * ya.i - s[10].i * yb.i; s[12].i = s[10].r * yb.i - s[9].r * ya.i;
            CADD(*F2, s[11], s[12]); CSUB(*F3, s[11], s[12]);
            ++F0; ++F1; ++F2; ++F3; ++F4;
        }
    }
}
static void fft320(const OModel *m, const cpx *fin, cpx *fout)    /* opus_fft_c kiss_fft.c:566-587 + opus_fft_impl :518-564 */
{
    int i; const float scale = 1.f / WINDOW_SIZE;
    for (i = 0; i < WINDOW_SIZE; i++) { fout[m->bitrev[i]].r = scale * fin[i].r; fout[m->bitrev[i]].i = scale * fin[i].i; }
    bfly4(fout, 80, m->tw, 1, 80, 4);
    bfly4(fout, 20, m->tw, 4, 20, 16);
    bfly4(fout, 5, m->tw, 16, 5, 64);
    bfly5(fout, 1, m->tw, 64, 1, 1);
}

static const short eband5ms[] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 10, 12, 14, 16, 20, 24, 28, 34, 40};
static const float compensation[] = {0.8f, 1.f, 1.f, 1.f, 1.f, 1.f, 1.f, 1.f, 0.666667f, 0.5f, 0.5f, 0.5f, 0.333333f, 0.25f, 0.25f, 0.2f, 0.166667f, 0.173913f};

static void lpc_from_cepstrum(const OModel *m, float *lpc, const float *cepstrum)   /* freq.c:310-320 */
{
    float Ex[NB_BANDS], tmp[NB_BANDS], Xr[FREQ_SIZE], ac[LPC_ORDER + 1], x_auto[WINDOW_SIZE];
    cpx x[WINDOW_SIZE], y[WINDOW_SIZE];
    int i, j;
    memcpy(tmp, cepstrum, sizeof(tmp));
    tmp[0] += 4;
    for (i = 0; i < NB_BANDS; i++) {                            /* idct freq.c:230-240 */
        float sum = 0;
        for (j = 0; j < NB_BANDS; j++) sum += tmp[j] * m->dct[i * NB_BANDS + j];
        Ex[i] = sum * sqrt(2. / NB_BANDS);
    }
    for (i = 0; i < NB_BANDS; i++) Ex[i] = pow(10.f, Ex[i]) * compensation[i];
    /* lpc_from_bands freq.c:275-297; interp_band_gain :202-215 */
    memset(Xr, 0, sizeof(Xr));
    for (i = 0; i < NB_BANDS - 1; i++) {
        int band_size = (eband5ms[i + 1] - eband5ms[i]) * 4;
        for (j = 0; j < band_size; j++) {
            float frac = (float)j / band_size;
            Xr[(eband5ms[i] * 4) + j] = (1 - frac) * Ex[i] + frac * Ex[i + 1];
        }
    }
    Xr[FREQ_SIZE - 1] = 0;
    /* inverse_transform freq.c:256-273 */
    for (i = 0; i < FREQ_SIZE; i++) { x[i].r = Xr[i]; x[i].i = 0; }
    for (; i < WINDOW_SIZE; i++) { x[i].r = x[WINDOW_SIZE - i].r; x[i].i = -x[WINDOW_SIZE - i].i; }
    fft320(m, x, y);
    x_auto[0] = WINDOW_SIZE * y[0].r;
    for (i = 1; i < WINDOW_SIZE; i++) x_auto[i] = WINDOW_SIZE * y[WINDOW_SIZE - i].r;
    for (i = 0; i < LPC_ORDER + 1; i++) ac[i] = x_auto[i];
    ac[0] += ac[0] * 1e-4 + 320 / 12 / 38.;
    for (i = 1; i < LPC_ORDER + 1; i++) ac[i] *= (1 - 6e-5 * i * i);
    {   /* lpcn_lpc freq.c:86-127 (float build: SHR32/SHL32 are identities, MULT32_32_Q31 is *) */
        float r, error = ac[0];
        memset(lpc, 0, sizeof(float) * LPC_ORDER);
        if (ac[0] != 0) {
            for (i = 0; i < LPC_ORDER; i++) {
                float rr = 0;
                for (j = 0; j < i; j++) rr += lpc[j] * ac[i - j];
                rr += ac[i + 1];
                r = -rr / error;
                lpc[i] = r;
                for (j = 0; j < (i + 1) >> 1; j++) {
                    float tmp1 = lpc[j], tmp2 = lpc[i - 1 - j];
                    lpc[j] = tmp1 + r * tmp2;
                    lpc[i - 1 - j] = tmp2 + r * tmp1;
                }
                error = error - (r * r) * error;
                if (error < .001f * ac[0]) break;
            }
        }
    }
}

/* ------------------------------------------------------------------ frame network ------------------------------------------------------------------ */
static void rc2lpc(float *lpc, const float *rc)                      /* lpcnet.c:57-78 */
{
    int i, j, k;
    float tmp[LPC_ORDER], ntmp[LPC_ORDER] = {0.0};
    memcpy(tmp, rc, sizeof(tmp));
    for (i = 0; i < LPC_ORDER; i++) {
        for (j = 0; j <= i - 1; j++) ntmp[j] = tmp[j] + tmp[i] * tmp[i - j - 1];
        for (k = 0; k <= i - 1; k++) tmp[k] = ntmp[k];
    }
    for (i = 0; i < LPC_ORDER; i++) lpc[i] = tmp[i];
}

static void run_frame_network(OState *st, const float *features)     /* lpcnet.c:82-120 */
{
    const OModel *m = st->m;
    const int N_A = m->na, delay = m->features_delay;
    float in[FRAME_IN], conv1_out[COND], conv2_out[COND], dense1_out[COND], condition[COND];
    float *lpc = st->lpc;
    int pitch, i;
    pitch = (int)floor(.1 + 50 * features[NB_BANDS] + 100);
    pitch = pitch > 255 ? 255 : (pitch < 33 ? 33 : pitch);        /* IMIN(255, IMAX(33, pitch)) */
    memcpy(in, features, sizeof(float) * NB_FEATURES);
    memcpy(in + NB_FEATURES, m->embed_pitch + pitch * PITCH_EMBED, sizeof(float) * PITCH_EMBED);
    conv1d(m, conv1_out, st->conv1_state, m->conv1_w, m->conv1_b, FRAME_IN, COND, in);
    if (st->frame_count < 1) memset(conv1_out, 0, sizeof(conv1_out));
    conv1d(m, conv2_out, st->conv2_state, m->conv2_w, m->conv2_b, COND, COND, conv1_out);
    if (st->frame_count < delay) memset(conv2_out, 0, sizeof(conv2_out));
    dense(m, dense1_out, m->dense1_w, m->dense1_b, COND, COND, conv2_out, 1);
    dense(m, condition, m->dense2_w, m->dense2_b, COND, COND, dense1_out, 1);
    dense(m, st->gru_a_condition, m->gad_w, m->gad_b, COND, 3 * N_A, condition, 0);
    dense(m, st->gru_b_condition, m->gbd_w, m->gbd_b, COND, 3 * N_B, condition, 0);
    if (m->end2end) rc2lpc(lpc, condition);                        /* lpcnet.c:105,107-108 */
    else if (delay > 0) {                                          /* lpcnet.c:109-112 */
        memcpy(lpc, st->old_lpc[delay - 1], sizeof(float) * LPC_ORDER);
        memmove(st->old_lpc[1], st->old_lpc[0], (delay - 1) * LPC_ORDER * sizeof(float));
        lpc_from_cepstrum(m, st->old_lpc[0], features);
    } else lpc_from_cepstrum(m, lpc, features);                    /* lpcnet.c:113-115 */
    {   /* lpc_weighting freq.c:299-308 */
        float gamma_i = m->lpc_gamma;
        for (i = 0; i < LPC_ORDER; i++) { lpc[i] *= gamma_i; gamma_i *= m->lpc_gamma; }
    }
    if (st->frame_count < 1000) st->frame_count++;
}

/* ------------------------------------------------------------------ sample network ------------------------------------------------------------------ */
#define SCALE (128.f * 127.f)
#define SCALE_1 (1.f / 128.f / 127.f)

/* int8: sparse_sgemv_accum8x4 vec_avx.h:790-858 ; float: vec_avx.h:865-903 */
static void sparse_gemv(const OModel *m, float *out, const void *wv, int rows, int cols, const int *idx, const float *xin, int32_t *peak)
{
    int i, j, r, c;
    if (!m->is_float) {
        const signed char *w = wv; unsigned char x[N_A_MAX];
        for (i = 0; i < cols; i++) x[i] = quant_u8(xin[i]);
        for (i = 0; i < rows; i += 8) {
            int nb = *idx++; int32_t acc[8], acc0[8];
            for (r = 0; r < 8; r++) acc0[r] = acc[r] = (int32_t)lrintf(out[i + r] * SCALE);
            for (j = 0; j < nb; j++) {
                int pos = *idx++;
                for (r = 0; r < 8; r++) for (c = 0; c < 4; c++) acc[r] += (int)x[pos + c] * (int)w[r * 4 + c];
                w += 32;
            }
            for (r = 0; r < 8; r++) out[i + r] = (float)acc[r] * SCALE_1;
            if (peak) for (r = 0; r < 8; r++) {
                if (abs(acc0[r]) > *peak) *peak = abs(acc0[r]);
                if (abs(acc[r]) > *peak) *peak = abs(acc[r]);
            }
        }
    } else {
        const float *w = wv;
        for (i = 0; i < rows; i += 8) {
            int nb = *idx++; float y[8];
            for (r = 0; r < 8; r++) y[r] = out[i + r];
            for (j = 0; j < nb; j++) {
                int id = *idx++;
                for (c = 0; c < 4; c++) for (r = 0; r < 8; r++) y[r] = fmaf(w[c * 8 + r], xin[id + c], y[r]);
                w += 32;
            }
            for (r = 0; r < 8; r++) out[i + r] = y[r];
        }
    }
}

static int run_sample_network(OState *st, int last_exc, int last_sig, int pred)     /* lpcnet.c:146-167 */
{
    const OModel *m = st->m;
    const int N_A = m->na;
    float gin[3 * N_A_MAX], recur[3 * N_A_MAX], zrh[3 * N_B], rec_b[3 * N_B];
    float *state = st->gru_a_state, *sb = st->gru_b_state;
    const float *bias;
    int i, k, b, j, val = 0;
    float thresholds[8];
    /* compute_gru_a_input nnet.c:484-491 */
    for (i = 0; i < 3 * N_A; i++)
        gin[i] = st->gru_a_condition[i] + m->emb_sig[last_sig * 3 * N_A + i] + m->emb_pred[pred * 3 * N_A + i] + m->emb_exc[last_exc * 3 * N_A + i];
    /* compute_sparse_gru nnet.c:410-448 */
    bias = m->is_float ? &m->ga_bias[3 * N_A] : &m->ga_subias[3 * N_A];
    for (k = 0; k < 2; k++) for (i = 0; i < N_A; i++) recur[k * N_A + i] = bias[k * N_A + i] + m->ga_diag[k * N_A + i] * state[i] + gin[k * N_A + i];
    for (; k < 3; k++) for (i = 0; i < N_A; i++) recur[k * N_A + i] = bias[k * N_A + i] + m->ga_diag[k * N_A + i] * state[i];
    sparse_gemv(m, recur, m->ga_w, 3 * N_A, N_A, m->ga_idx, state, &st->acc_peak);
    for (i = 0; i < 2 * N_A; i++) recur[i] = sigmoid_a(m, recur[i]);
    for (i = 0; i < N_A; i++) recur[2 * N_A + i] = recur[2 * N_A + i] * recur[N_A + i] + gin[2 * N_A + i];
    for (i = 0; i < N_A; i++) recur[2 * N_A + i] = tanh_a(m, recur[2 * N_A + i]);
    for (i = 0; i < N_A; i++) state[i] = recur[i] * state[i] + (1 - recur[i]) * recur[2 * N_A + i];
    /* compute_gruB nnet.c:326-372 */
    bias = m->is_float ? m->gb_bias : m->gb_subias;
    for (i = 0; i < 3 * N_B; i++) zrh[i] = bias[i] + st->gru_b_condition[i];
    sparse_gemv(m, zrh, m->gb_w, 3 * N_B, N_A, m->gb_idx, state, NULL);
    for (i = 0; i < 3 * N_B; i++) rec_b[i] = bias[3 * N_B + i];
    if (!m->is_float) {                                        /* sgemv_accum8x4 vec_avx.h:690-755 */
        const signed char *w = m->gb_rw; unsigned char x[N_B]; int r, c;
        for (i = 0; i < N_B; i++) x[i] = quant_u8(sb[i]);
        for (i = 0; i < 3 * N_B; i += 8) {
            int32_t acc[8];
            for (r = 0; r < 8; r++) acc[r] = (int32_t)lrintf(rec_b[i + r] * SCALE);
            for (j = 0; j < N_B; j += 4) { for (r = 0; r < 8; r++) for (c = 0; c < 4; c++) acc[r] += (int)x[j + c] * (int)w[r * 4 + c]; w += 32; }
            for (r = 0; r < 8; r++) rec_b[i + r] = (float)acc[r] * SCALE_1;
        }
    } else {
        sgemv_fma(rec_b, m->gb_rw, 3 * N_B, N_B, 3 * N_B, sb);
    }
    for (i = 0; i < 2 * N_B; i++) zrh[i] += rec_b[i];
    for (i = 0; i < 2 * N_B; i++) zrh[i] = sigmoid_a(m, zrh[i]);
    for (i = 0; i < N_B; i++) zrh[2 * N_B + i] += rec_b[2 * N_B + i] * zrh[N_B + i];
    for (i = 0; i < N_B; i++) zrh[2 * N_B + i] = tanh_a(m, zrh[2 * N_B + i]);
    for (i = 0; i < N_B; i++) sb[i] = zrh[i] * sb[i] + (1 - zrh[i]) * zrh[2 * N_B + i];
    /* sample_mdense nnet.c:163-214 */
    for (b = 0; b < 8; b += 4) {
        uint32_t r = kiss99_rand(&st->rng);
        thresholds[b] = m->logit[r & 0xFF]; thresholds[b + 1] = m->logit[(r >> 8) & 0xFF];
        thresholds[b + 2] = m->logit[(r >> 16) & 0xFF]; thresholds[b + 3] = m->logit[(r >> 24) & 0xFF];
    }
    for (b = 0; b < 8; b++) {
        int bit; float sum1, sum2;
        i = (1 << b) | val;
        sum1 = m->fc_b[i]; sum2 = m->fc_b[i + 256];
        for (j = 0; j < N_B; j++) { sum1 += m->fc_w[i * 32 + j] * sb[j]; sum2 += m->fc_w[i * 32 + j + N_B] * sb[j]; }
        sum1 = m->fc_f[i] * tanh_a(m, sum1); sum2 = m->fc_f[256 + i] * tanh_a(m, sum2);
        sum1 += sum2;
        bit = thresholds[b] < sum1;
        val = (val << 1) | bit;
    }
    return val;
}

static void synthesize_tail(OState *st, short *output, int N, int preload)    /* lpcnet_synthesize_tail_impl lpcnet.c:235-271 */
{
    int i, j;
    if (st->frame_count <= st->m->features_delay) { memset(output, 0, sizeof(short) * N); return; }
    for (i = 0; i < N; i++) {
        float pcm, pred = 0; int exc, last_sig_ulaw, pred_ulaw;
        for (j = 0; j < LPC_ORDER; j++) pred -= st->last_sig[j] * st->lpc[j];
        last_sig_ulaw = lin2ulaw(st->last_sig[0]);
        pred_ulaw = lin2ulaw(pred);
        exc = run_sample_network(st, st->last_exc, last_sig_ulaw, pred_ulaw);
        if (st->trace_exc) st->trace_exc[i] = exc;
        if (i < preload) {                                         /* lpcnet.c:256-259 */
            exc = lin2ulaw(output[i] - PREEMPH * st->deemph_mem - pred);
            pcm = output[i] - PREEMPH * st->deemph_mem;
        } else pcm = pred + st->m->ulaw2lin_tab[exc];
        memmove(&st->last_sig[1], &st->last_sig[0], (LPC_ORDER - 1) * sizeof(float));
        st->last_sig[0] = pcm;
        st->last_exc = exc;
        pcm += PREEMPH * st->deemph_mem;
        st->deemph_mem = pcm;
        if (pcm < -32767) pcm = -32767;
        if (pcm > 32767) pcm = 32767;
        if (i >= preload) output[i] = (int)floor(.5 + pcm);
    }
}

/* ------------------------------------------------------------------ decoder front-end ------------------------------------------------------------------ */
static void decode_packet(OState *st, float features[4][NB_TOTAL_FEATURES], const unsigned char buf[8])   /* lpcnet_dec.c:81-155 */
{
    const OModel *m = st->m; float *vq_mem = st->vq_mem;
    uint64_t bits = 0; int pos = 0, i, sub, voiced = 1;
    int c0_id, main_pitch, modulation, corr_id, vq_end[3], vq_mid, interp_id, id0, id1;
    float frame_corr, sign;
#define GET(n) (pos += (n), (int)((bits >> (64 - pos)) & ((1u << (n)) - 1)))
    for (i = 0; i < 8; i++) bits = (bits << 8) | buf[i];        /* MSB-first bit reader == bits_unpack :59-78 */
    c0_id = GET(7); main_pitch = GET(6); modulation = GET(3); corr_id = GET(2);
    vq_end[0] = GET(10); vq_end[1] = GET(10); vq_end[2] = GET(10); vq_mid = GET(13); interp_id = GET(3);
#undef GET
    for (i = 0; i < 4; i++) memset(features[i], 0, sizeof(float) * NB_TOTAL_FEATURES);
    modulation -= 4;
    if (modulation == -4) { voiced = 0; modulation = 0; }
    if (voiced) frame_corr = 0.3875f + .175f * corr_id; else frame_corr = 0.0375f + .075f * corr_id;
    for (sub = 0; sub < 4; sub++) {
        float p = pow(2.f, main_pitch / 21.) * 32;            /* PITCH_MIN_PERIOD 32 (src/lpcnet_private.h) */
        p *= 1.f + modulation / 16.f / 7.f * (2 * sub - 3);
        p = (255 < (33 > p ? 33 : p)) ? 255 : (33 > p ? 33 : p);  /* MIN16(255, MAX16(33, p)) */
        features[sub][NB_BANDS] = .02f * (p - 100.f);
        features[sub][NB_BANDS + 1] = frame_corr - .5f;
    }
    features[3][0] = (c0_id - 64) / 4.f;
    for (i = 0; i < NB_BANDS - 1; i++)
        features[3][i + 1] = m->cb1[vq_end[0] * 17 + i] + m->cb2[vq_end[1] * 17 + i] + m->cb3[vq_end[2] * 17 + i];
    sign = 1;
    if (vq_mid >= 4096) { vq_mid -= 4096; sign = -1; }
    for (i = 0; i < NB_BANDS; i++) features[1][i] = sign * m->cbd4[vq_mid * NB_BANDS + i];
    if ((vq_mid & 3) < 2) { for (i = 0; i < NB_BANDS; i++) features[1][i] += .5f * (vq_mem[i] + features[3][i]); }   /* MULTI_MASK 3 */
    else if ((vq_mid & 3) == 2) { for (i = 0; i < NB_BANDS; i++) features[1][i] += vq_mem[i]; }
    else { for (i = 0; i < NB_BANDS; i++) features[1][i] += features[3][i]; }
    /* perform_double_interp common.c:58-65 (FORBIDDEN_INTERP 7) */
    interp_id += (interp_id >= 7);
    id0 = interp_id / 3; id1 = interp_id % 3;
    for (i = 0; i < NB_BANDS; i++) {
        const float *l0 = vq_mem, *r0 = features[1], *l1 = features[1], *r1 = features[3];
        float a = id0 == 0 ? .5f * (l0[i] + r0[i]) : (id0 == 1 ? l0[i] : r0[i]);
        float c = id1 == 0 ? .5f * (l1[i] + r1[i]) : (id1 == 1 ? l1[i] : r1[i]);
        features[0][i] = a; features[2][i] = c;
    }
    memcpy(vq_mem, features[3], sizeof(float) * NB_BANDS);
}

/* ------------------------------------------------------------------ public test API ------------------------------------------------------------------ */
/* features_delay / end2end: what the reference bakes into the generated nnet_data.h (FEATURES_DELAY, END2END) */
OModel *oracle_model_create_ex(const unsigned char *blob_in, int len, const uint32_t *rcp_table, float lpc_gamma,
                               int features_delay, int end2end, const float *codebooks /* may be NULL */)
{
    OModel *m = calloc(1, sizeof(*m));
    unsigned char *d = malloc(len);
    int tb_a = 0, tb_b = 0, sz = -1, N_A;
    memcpy(d, blob_in, len);
    m->blob_copy = d; m->lpc_gamma = lpc_gamma; m->features_delay = features_delay; m->end2end = end2end;
    if (features_delay < 0 || features_delay > FEATURES_DELAY_MAX) goto fail;
    if (!find_array(d, len, "sparse_gru_a_recurrent_weights_diag", &sz) || sz % 12 || sz / 12 > N_A_MAX) goto fail;
    N_A = m->na = sz / 12; sz = -1;
    memcpy(m->rcp, rcp_table, sizeof(m->rcp));
    build_tables(m);
#define F(field, name, count) if (!(m->field = need(d, len, name, (count) * 4))) { fprintf(stderr, "oracle: bad array %s\n", name); goto fail; }
    F(embed_pitch, "embed_pitch_weights", 256 * PITCH_EMBED)
    F(conv1_w, "feature_conv1_weights", 3 * FRAME_IN * COND) F(conv1_b, "feature_conv1_bias", COND)
    F(conv2_w, "feature_conv2_weights", 3 * COND * COND) F(conv2_b, "feature_conv2_bias", COND)
    F(dense1_w, "feature_dense1_weights", COND * COND) F(dense1_b, "feature_dense1_bias", COND)
    F(dense2_w, "feature_dense2_weights", COND * COND) F(dense2_b, "feature_dense2_bias", COND)
    F(gad_w, "gru_a_dense_feature_weights", COND * 3 * N_A) F(gad_b, "gru_a_dense_feature_bias", 3 * N_A)
    F(gbd_w, "gru_b_dense_feature_weights", COND * 3 * N_B) F(gbd_b, "gru_b_dense_feature_bias", 3 * N_B)
    F(emb_sig, "gru_a_embed_sig_weights", 256 * 3 * N_A) F(emb_pred, "gru_a_embed_pred_weights", 256 * 3 * N_A)
    F(emb_exc, "gru_a_embed_exc_weights", 256 * 3 * N_A)
    F(ga_bias, "sparse_gru_a_bias", 6 * N_A) F(ga_subias, "sparse_gru_a_subias", 6 * N_A)
    F(ga_diag, "sparse_gru_a_recurrent_weights_diag", 3 * N_A)
    F(gb_bias, "gru_b_bias", 6 * N_B) F(gb_subias, "gru_b_subias", 6 * N_B)
    F(fc_w, "dual_fc_weights", 256 * 2 * N_B) F(fc_b, "dual_fc_bias", 512) F(fc_f, "dual_fc_factor", 512)
#undef F
    if (!(m->ga_idx = need_idx(d, len, "sparse_gru_a_recurrent_weights_idx", N_A, 3 * N_A, &tb_a))) goto fail;
    if (!(m->gb_idx = need_idx(d, len, "gru_b_weights_idx", N_A, 3 * N_B, &tb_b))) goto fail;
    m->ga_w = find_array(d, len, "sparse_gru_a_recurrent_weights", &sz);
    if (!m->ga_w) goto fail;
    if (sz == 32 * tb_a) m->is_float = 0; else if (sz == 128 * tb_a) m->is_float = 1; else goto fail;
    if (!(m->gb_w = need(d, len, "gru_b_weights", (m->is_float ? 128 : 32) * tb_b))) goto fail;
    if (!(m->gb_rw = need(d, len, "gru_b_recurrent_weights", (m->is_float ? 4 : 1) * 3 * N_B * N_B))) goto fail;
    if (codebooks) {
        size_t n = 3 * 1024 * 17 + 4096 * 18;
        m->cb_copy = malloc(n * 4); memcpy(m->cb_copy, codebooks, n * 4);
        m->cb1 = m->cb_copy; m->cb2 = m->cb1 + 1024 * 17; m->cb3 = m->cb2 + 1024 * 17; m->cbd4 = m->cb3 + 1024 * 17;
    }
    return m;
fail:
    free(d); free(m); return NULL;
}
OModel *oracle_model_create(const unsigned char *blob_in, int len, const uint32_t *rcp_table, float lpc_gamma, const float *codebooks)
{
    return oracle_model_create_ex(blob_in, len, rcp_table, lpc_gamma, 2, 0, codebooks);
}
int oracle_model_na(const OModel *m) { return m->na; }
void oracle_model_destroy(OModel *m) { if (m) { free(m->blob_copy); free(m->cb_copy); free(m); } }
int oracle_model_is_float(const OModel *m) { return m->is_float; }

void oracle_reset(OState *st)                                   /* lpcnet_reset lpcnet.c:174-182 */
{
    const OModel *m = st->m;
    memset(st, 0, sizeof(*st));
    st->m = m;
    st->last_exc = lin2ulaw(0.f);
    kiss99_srand(&st->rng, (const unsigned char *)"LPCNet", 6);
}
int oracle_state_size(void) { return (int)sizeof(OState); }
OState *oracle_state_create(const OModel *m) { OState *st = calloc(1, sizeof(*st)); st->m = m; oracle_reset(st); return st; }
void oracle_state_destroy(OState *st) { free(st); }

void oracle_synthesize_impl(OState *st, const float *features, short *output, int N, int preload)   /* lpcnet_synthesize_impl lpcnet.c:273-277 */
{
    run_frame_network(st, features);
    synthesize_tail(st, output, N, preload);
}
void oracle_synthesize(OState *st, const float *features, short *output, int N)   /* lpcnet_synthesize lpcnet.c:279-281 */
{
    oracle_synthesize_impl(st, features, output, N, 0);
}
/* the other internal entry points the PLC uses (lpcnet_private.h:125-133) */
void oracle_run_frame_network(OState *st, const float *features) { run_frame_network(st, features); }
void oracle_synthesize_tail(OState *st, short *output, int N, int preload) { synthesize_tail(st, output, N, preload); }
void oracle_frame_network_deferred(OState *st, const float *features)             /* run_frame_network_deferred lpcnet.c:122-132 */
{
    const int max_buffer_size = 3 + 3 - 2;
    if (st->feature_buffer_fill == max_buffer_size) memmove(st->feature_buffer, &st->feature_buffer[NB_FEATURES], (max_buffer_size - 1) * NB_FEATURES * sizeof(float));
    else st->feature_buffer_fill++;
    memcpy(&st->feature_buffer[(st->feature_buffer_fill - 1) * NB_FEATURES], features, NB_FEATURES * sizeof(float));
}
void oracle_frame_network_flush(OState *st)                                       /* run_frame_network_flush lpcnet.c:134-144 */
{
    int i;
    for (i = 0; i < st->feature_buffer_fill; i++) run_frame_network(st, &st->feature_buffer[i * NB_FEATURES]);
    st->feature_buffer_fill = 0;
}
void oracle_reset_signal(OState *st)                                              /* lpcnet_reset_signal lpcnet.c:226-233 */
{
    st->deemph_mem = 0; st->last_exc = lin2ulaw(0.f);
    memset(st->last_sig, 0, sizeof(st->last_sig)); memset(st->gru_a_state, 0, sizeof(st->gru_a_state)); memset(st->gru_b_state, 0, sizeof(st->gru_b_state));
}
/* The state in the layout of lpcnet_b200_batch_export_state (include/lpcnet_b200.h): floats hA[na] hB[16] last_sig[16] deemph
 * conv1[168] conv2[256] old_lpc[0][16] old_lpc[1][16] vq_mem[18], then ints last_exc, frame_count, rng[4]. */
int oracle_export_state(const OState *st, float *buf)
{
    const int na = st->m->na; int o = 0, iv[6];
    memcpy(buf + o, st->gru_a_state, na * 4); o += na;
    memcpy(buf + o, st->gru_b_state, N_B * 4); o += N_B;
    memcpy(buf + o, st->last_sig, LPC_ORDER * 4); o += LPC_ORDER;
    buf[o++] = st->deemph_mem;
    memcpy(buf + o, st->conv1_state, sizeof(st->conv1_state)); o += 2 * FRAME_IN;
    memcpy(buf + o, st->conv2_state, sizeof(st->conv2_state)); o += 2 * COND;
    memcpy(buf + o, st->old_lpc, sizeof(st->old_lpc)); o += 2 * LPC_ORDER;
    memcpy(buf + o, st->vq_mem, sizeof(st->vq_mem)); o += NB_BANDS;
    iv[0] = st->last_exc; iv[1] = st->frame_count; memcpy(&iv[2], &st->rng, 16);
    memcpy(buf + o, iv, sizeof(iv)); o += 6;
    return o * 4;
}
/* int8 models: largest |accumulator| of the GRU_A GEMV seen by this state (the conversion-free rounding of the CUDA kernel is exact
   below 2^22; model.cu proves a bound from the weights, this measures what synthesis reaches) */
int oracle_acc_peak(const OState *st) { return st->acc_peak; }

void oracle_synthesize_trace(OState *st, const float *features, short *output, int N, int *exc)
{
    st->trace_exc = exc; oracle_synthesize(st, features, output, N); st->trace_exc = NULL;
}
int oracle_decode(OState *st, const unsigned char *buf, short *pcm)               /* lpcnet_decode lpcnet.c:310-319 */
{
    float features[4][NB_TOTAL_FEATURES]; int k;
    if (!st->m->cb1) return -1;
    decode_packet(st, features, buf);
    for (k = 0; k < 4; k++) oracle_synthesize(st, features[k], &pcm[k * FRAME_SIZE], FRAME_SIZE);
    return 0;
}
void oracle_decode_packet(OState *st, float *features /*[4][36]*/, const unsigned char *buf)
{
    decode_packet(st, (float (*)[NB_TOTAL_FEATURES])features, buf);
}
/* taps for unit tests */
void oracle_frame_network(OState *st, const float *features, float *ga /*1152*/, float *gb /*48*/, float *lpc /*16*/)
{
    run_frame_network(st, features);
    memcpy(ga, st->gru_a_condition, sizeof(float) * 3 * st->m->na);
    memcpy(gb, st->gru_b_condition, sizeof(st->gru_b_condition));
    memcpy(lpc, st->lpc, sizeof(st->lpc));
}
void oracle_get_tables(const OModel *m, float *tw /*640*/, int *bitrev /*320*/, float *dct /*324*/, float *logit /*256*/, float *u2l /*256*/)
{
    memcpy(tw, m->tw, sizeof(m->tw)); memcpy(bitrev, m->bitrev, sizeof(m->bitrev)); memcpy(dct, m->dct, sizeof(m->dct));
    memcpy(logit, m->logit, sizeof(m->logit)); memcpy(u2l, m->ulaw2lin_tab, sizeof(m->ulaw2lin_tab));
}
float oracle_tanh(const OModel *m, float x) { return tanh_a(m, x); }
float oracle_sigmoid(const OModel *m, float x) { return sigmoid_a(m, x); }
int oracle_lin2ulaw(float x) { return lin2ulaw(x); }
void oracle_get_state(const OState *st, float *gru_a /*384*/, float *gru_b /*16*/, float *last_sig /*16*/, int *misc /*[last_exc, frame_count]*/, uint32_t *rng /*4*/)
{
    memcpy(gru_a, st->gru_a_state, sizeof(float) * st->m->na); memcpy(gru_b, st->gru_b_state, sizeof(st->gru_b_state));
    memcpy(last_sig, st->last_sig, sizeof(st->last_sig)); misc[0] = st->last_exc; misc[1] = st->frame_count;
    memcpy(rng, &st->rng, 16);
}

/* Batch helper: n_streams independent streams x nframes frames, spread over nthreads host threads.
 * features [n_streams][nframes][stride]; pcm [n_streams][nframes*160]. Returns wall seconds (used by the
 * bench's cpu_baseline "port" leg and by parity tests that need many streams). */
typedef struct { const OModel *m; const float *features; int stride, nframes, first, last; short *pcm; const unsigned char *packets; } ojob;
static void *oworker(void *a)
{
    ojob *j = a; int s, f;
    for (s = j->first; s < j->last; s++) {
        OState *st = oracle_state_create(j->m);
        if (j->packets) {
            for (f = 0; f < j->nframes; f++) oracle_decode(st, j->packets + ((size_t)s * j->nframes + f) * 8, j->pcm + ((size_t)s * j->nframes + f) * 640);
        } else {
            for (f = 0; f < j->nframes; f++)
                oracle_synthesize(st, j->features + ((size_t)s * j->nframes + f) * j->stride, j->pcm + ((size_t)s * j->nframes + f) * FRAME_SIZE, FRAME_SIZE);
        }
        oracle_state_destroy(st);
    }
    return NULL;
}
static double run_batch(const OModel *m, const float *features, int stride, const unsigned char *packets, int n_streams, int nframes, int nthreads, short *pcm)
{
    struct timespec t0, t1; int i;
    pthread_t *th; ojob *jobs;
    if (nthreads < 1) nthreads = 1;
    if (nthreads > n_streams) nthreads = n_streams;
    th = malloc(sizeof(*th) * nthreads); jobs = malloc(sizeof(*jobs) * nthreads);
    clock_gettime(CLOCK_MONOTONIC, &t0);
    for (i = 0; i < nthreads; i++) {
        jobs[i].m = m; jobs[i].features = features; jobs[i].stride = stride; jobs[i].nframes = nframes; jobs[i].pcm = pcm; jobs[i].packets = packets;
        jobs[i].first = (int)((long)n_streams * i / nthreads); jobs[i].last = (int)((long)n_streams * (i + 1) / nthreads);
        pthread_create(&th[i], NULL, oworker, &jobs[i]);
    }
    for (i = 0; i < nthreads; i++) pthread_join(th[i], NULL);
    clock_gettime(CLOCK_MONOTONIC, &t1);
    free(th); free(jobs);
    return (t1.tv_sec - t0.tv_sec) + 1e-9 * (t1.tv_nsec - t0.tv_nsec);
}
double oracle_synthesize_batch(const OModel *m, const float *features, int stride, int n_streams, int nframes, int nthreads, short *pcm)
{ return run_batch(m, features, stride, NULL, n_streams, nframes, nthreads, pcm); }
double oracle_decode_batch(const OModel *m, const unsigned char *packets, int n_streams, int npackets, int nthreads, short *pcm)
{ return run_batch(m, NULL, 0, packets, n_streams, npackets, nthreads, pcm); }

/* ------------------------------------------------------------------ analysis side (SURVEY 8f N2) ------------------------------------------------------------------ */
#include "lpcnet_enc_oracle.inc"
