/* lpcnet_b200.h — batched C-ABI of the B200-native LPCNet synthesis engine (the throughput surface).
 *
 * The reference API (include/lpcnet.h) drives ONE stream, 160 samples per call.  The hot path
 * (reference src/lpcnet.c:235-271 `lpcnet_synthesize_tail_impl` -> :146 `run_sample_network`) is strictly serial
 * inside a stream, so GPU throughput comes from stepping thousands of independent streams in lockstep.  This
 * header is the extension SURVEY.md 8(b) calls for: the same operations as `lpcnet_synthesize` /
 * `lpcnet_decode`, applied to a batch of independent streams that all start from a fresh `lpcnet_create()` state
 * (reference src/lpcnet.c:174-200: zero state, RNG seeded with "LPCNet").
 *
 * Plain C: pointers + sizes only.  Host-pointer entry points copy features in and PCM out inside the call;
 * `_device` variants take CUDA device pointers (already resident inputs) and a CUDA stream handle.
 * All functions return 0 on success, negative on error (message: lpcnet_b200_last_error()).
 */
#ifndef LPCNET_B200_H
#define LPCNET_B200_H

#include <stddef.h>
#include <stdint.h>

#ifndef LPCNET_EXPORT
# if defined(__GNUC__)
#  define LPCNET_EXPORT __attribute__ ((visibility ("default")))
# else
#  define LPCNET_EXPORT
# endif
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct LPCNetB200Batch LPCNetB200Batch;
typedef struct LPCNetB200Snapshot LPCNetB200Snapshot;

/* The three per-model switches the reference bakes into the generated nnet_data.h (training_tf2/dump_lpcnet.py:306-329)
 * instead of the weight blob.  A negative / non-positive field means "take it from the blob's `lpcnet_b200_config`
 * metadata record (written by lpcnet_b200_write_blob / tools/import_nnet_data.py) or, failing that, the reference default". */
typedef struct LPCNetB200Config {
    float lpc_gamma;        /* LPC_GAMMA: lpc_weighting factor (src/freq.c:299-308); default 1 (none) */
    int features_delay;     /* FEATURES_DELAY 0..2: look-ahead frames (src/lpcnet.c:101,109-115,239); default 2 */
    int end2end;            /* END2END: LPC from the network's reflection coefficients (src/lpcnet.c:57-78,107-108); default 0 */
} LPCNetB200Config;

/* One named array of a model blob: the reference's WeightArray (src/nnet.h:43-48).  type: 0 float, 1 int, 2 qweight (int8);
 * size in bytes. */
typedef struct LPCNetB200Array {
    const char *name;
    int type;
    int size;
    const void *data;
} LPCNetB200Array;

/* == model blob I/O (host only, no CUDA) ==
 * lpcnet_b200_write_blob: serialise arrays to the "DNNw" weight-blob format exactly like the reference's write_weights()
 * (src/write_lpcnet_weights.c:47-67: 64-byte WeightHead, payload zero-padded to a multiple of 64 bytes).  With cfg != NULL the
 * three switches the reference leaves in nnet_data.h travel as one extra record `lpcnet_b200_config` (float[4]: LPC_GAMMA,
 * FEATURES_DELAY, END2END, format version) which the reference's own loader ignores.  out == NULL: returns the size needed.
 * Returns the number of bytes written, < 0 on error. */
LPCNET_EXPORT long long lpcnet_b200_write_blob(const LPCNetB200Array *arrays, int count, const LPCNetB200Config *cfg,
                                               unsigned char *out, size_t cap);
LPCNET_EXPORT int lpcnet_b200_write_blob_file(const char *path, const LPCNetB200Array *arrays, int count, const LPCNetB200Config *cfg);
/* parse_weights() (src/parse_lpcnet_weights.c:37-76): lists the records of a blob (entries point into `blob`).  Returns the
 * number of records (may exceed cap; only cap are filled), < 0 if the blob is malformed. */
LPCNET_EXPORT int lpcnet_b200_parse_blob(const unsigned char *blob, int len, LPCNetB200Array *arrays, int cap);
/* The blob's `lpcnet_b200_config` record: 1 = found (cfg filled), 0 = the blob has none, < 0 malformed blob. */
LPCNET_EXPORT int lpcnet_b200_blob_config(const unsigned char *blob, int len, LPCNetB200Config *cfg);
/* Whole-file read (weights_blob.bin, .f32 feature files, packet files): out == NULL returns the size. */
LPCNET_EXPORT long long lpcnet_b200_read_file(const char *path, unsigned char *out, size_t cap);

/* Number of usable CUDA devices (0 => the engine cannot run; there is no CPU fallback). */
LPCNET_EXPORT int lpcnet_b200_device_count(void);
/* Last error message of the calling thread ("" if none). */
LPCNET_EXPORT const char *lpcnet_b200_last_error(void);
/* Library/ABI version: major*10000 + minor*100 + patch. */
LPCNET_EXPORT int lpcnet_b200_version(void);

/* Create `n_streams` independent synthesis streams on CUDA device `device`, all using the model in the "DNNw"
 * blob (same format/validation as reference lpcnet_load_model, src/lpcnet.c:202 + src/parse_lpcnet_weights.c:115-221;
 * both the int8 DOT_PROD and the float flavour are accepted and select the arithmetic).  `lpc_gamma` is the
 * reference's compile-time LPC_GAMMA (generated nnet_data.h; training_tf2/dump_lpcnet.py:313-319); pass 1.0f for
 * "no weighting".  Returns NULL on error. */
LPCNET_EXPORT LPCNetB200Batch *lpcnet_b200_batch_create(int n_streams, const unsigned char *blob, int blob_len,
                                                        float lpc_gamma, int device);
/* Same with the per-model switches given explicitly (NULL: blob metadata / defaults).  The number of GRU_A units is read
 * from the blob (128, 256 or 384: training_tf2/train_lpcnet.py --grua-size); GRU_B = 16 and cond = 128 are fixed. */
LPCNET_EXPORT LPCNetB200Batch *lpcnet_b200_batch_create_ex(int n_streams, const unsigned char *blob, int blob_len,
                                                           const LPCNetB200Config *cfg, int device);
LPCNET_EXPORT void lpcnet_b200_batch_destroy(LPCNetB200Batch *b);
/* GRU_A units and the switches in effect. */
LPCNET_EXPORT int lpcnet_b200_batch_model_info(const LPCNetB200Batch *b, int *gru_a_units, LPCNetB200Config *cfg);
/* lpcnet_reset() (reference src/lpcnet.c:174) applied to every stream. */
LPCNET_EXPORT int lpcnet_b200_batch_reset(LPCNetB200Batch *b);
/* lpcnet_reset() for the listed streams only: they start a new utterance (two silent frames, fresh RNG) while the other
 * streams of the batch carry on.  Every stream has its own frame counter. */
LPCNET_EXPORT int lpcnet_b200_batch_reset_streams(LPCNetB200Batch *b, const int *streams, int count);
/* lpcnet_reset_signal() (reference src/lpcnet.c:226-233, used by the PLC): clears the sample-rate state only. */
LPCNET_EXPORT int lpcnet_b200_batch_reset_signal(LPCNetB200Batch *b);
LPCNET_EXPORT int lpcnet_b200_batch_streams(const LPCNetB200Batch *b);

/* VQ codebooks for the decoder front-end (reference src/lpcnet_dec.c:129-143 reads ceps_codebook1..3 [1024][17]
 * and ceps_codebook_diff4 [4096][18]; the reference links them from the un-shipped ceps_codebooks.c).
 * `cb` = the four arrays concatenated in that order (3*1024*17 + 4096*18 floats). */
LPCNET_EXPORT int lpcnet_b200_batch_set_codebooks(LPCNetB200Batch *b, const float *cb, size_t n_floats);

/* == lpcnet_synthesize() per stream, `nframes` times ==
 * features: [n_streams][nframes][feature_stride] floats (first 20 of each frame used; stride 20 or 36 typical)
 * pcm     : [n_streams][nframes*samples_per_frame] int16
 * samples_per_frame is the reference's N argument (160 in the demo/decoder; any N >= 1 like the reference). */
LPCNET_EXPORT int lpcnet_b200_batch_synthesize(LPCNetB200Batch *b, const float *features, int nframes,
                                               int feature_stride, int samples_per_frame, short *pcm);
LPCNET_EXPORT int lpcnet_b200_batch_synthesize_device(LPCNetB200Batch *b, const float *d_features, int nframes,
                                                      int feature_stride, int samples_per_frame, short *d_pcm,
                                                      void *cuda_stream);

/* == lpcnet_synthesize_impl(st, features, out, N, preload) (reference src/lpcnet.c:273-277; PLC entry point) ==
 * The first `preload` samples of the call's FIRST frame are teacher-forced: the network runs (state and RNG advance) but the
 * excitation is derived from the signal the caller supplies in pcm[s][0..preload) and those samples are not overwritten
 * (src/lpcnet.c:256-259,269). */
LPCNET_EXPORT int lpcnet_b200_batch_synthesize_ex(LPCNetB200Batch *b, const float *features, int nframes,
                                                  int feature_stride, int samples_per_frame, short *pcm, int preload);
LPCNET_EXPORT int lpcnet_b200_batch_synthesize_device_ex(LPCNetB200Batch *b, const float *d_features, int nframes,
                                                         int feature_stride, int samples_per_frame, short *d_pcm,
                                                         int preload, void *cuda_stream);
/* == the other internal entry points the reference's PLC uses (src/lpcnet_private.h:125-133), batched ==
 * run_frame_network (src/lpcnet.c:82-120) only: advances the 100 Hz state, keeps the last frame's conditioning */
LPCNET_EXPORT int lpcnet_b200_batch_run_frame_network(LPCNetB200Batch *b, const float *features, int nframes, int feature_stride);
/* lpcnet_synthesize_tail_impl (src/lpcnet.c:235-271): `samples` samples with the conditioning of the last frame-network run;
 * pcm [n_streams][samples] */
LPCNET_EXPORT int lpcnet_b200_batch_synthesize_tail(LPCNetB200Batch *b, int samples, short *pcm, int preload);
/* run_frame_network_deferred / run_frame_network_flush (src/lpcnet.c:122-144): queue one feature frame per stream
 * (features [n_streams][feature_stride], at most 4 queued, older ones drop out) / run the frame network over the queue */
LPCNET_EXPORT int lpcnet_b200_batch_frame_network_deferred(LPCNetB200Batch *b, const float *features, int feature_stride);
LPCNET_EXPORT int lpcnet_b200_batch_frame_network_flush(LPCNetB200Batch *b);

/* == state by value ==  The reference's PLC copies `LPCNetState` structs to roll back speculative synthesis
 * (src/lpcnet_plc.c:216-230).  One stream <-> opaque host blob of lpcnet_b200_batch_state_size() bytes (everything
 * lpcnet_reset() clears: GRU states, signal history, conv/LPC delay lines, decoder memory, RNG, frame counter): */
LPCNET_EXPORT int lpcnet_b200_batch_state_size(const LPCNetB200Batch *b);
LPCNET_EXPORT int lpcnet_b200_batch_export_state(LPCNetB200Batch *b, int stream, void *buf);
LPCNET_EXPORT int lpcnet_b200_batch_import_state(LPCNetB200Batch *b, int stream, const void *buf);
/* ... and the whole batch, device to device: */
LPCNET_EXPORT LPCNetB200Snapshot *lpcnet_b200_batch_snapshot_create(LPCNetB200Batch *b);
LPCNET_EXPORT void lpcnet_b200_batch_snapshot_destroy(LPCNetB200Snapshot *s);
LPCNET_EXPORT int lpcnet_b200_batch_snapshot_save(LPCNetB200Batch *b, LPCNetB200Snapshot *s);
LPCNET_EXPORT int lpcnet_b200_batch_snapshot_restore(LPCNetB200Batch *b, const LPCNetB200Snapshot *s);

/* == multi-GPU: PCM sink ==  Streams shard across GPUs with no data-path exchange (SURVEY.md 8e); the only transfer is the
 * gather of the PCM.  With a sink set, every synthesize/decode `_device` call also copies each finished chunk (<= 16 frames)
 * of its PCM to  sink[(first_row + s) * pitch_samples + t]  on a copy stream (DMA engines over NVLink, no SM time) while the next
 * chunk is being computed; the call's stream completes only after the last copy.  `sink` may live on another device of this
 * process (peer access) or in another process (lpcnet_b200_ipc_export on the owner, lpcnet_b200_ipc_open here).
 * sink == NULL removes it. */
LPCNET_EXPORT int lpcnet_b200_batch_set_pcm_sink(LPCNetB200Batch *b, short *sink, long long pitch_samples, long long first_row);
LPCNET_EXPORT int lpcnet_b200_ipc_export(void *d_ptr, unsigned char handle[64]);
LPCNET_EXPORT void *lpcnet_b200_ipc_open(const unsigned char handle[64]);
LPCNET_EXPORT int lpcnet_b200_ipc_close(void *p);
LPCNET_EXPORT int lpcnet_b200_set_device(int device);

/* == multi-GPU in ONE process ==  `n_streams` independent streams cut into contiguous index ranges over `n_devices` CUDA devices
 * (devices[k] = CUDA ordinal of shard k; NULL = 0..n_devices-1), weights replicated, one LPCNetB200Batch per device.  Every call
 * enqueues all shards (each on its device's own stream) and then waits: the devices run concurrently and nothing is exchanged
 * inside the sample loop.  Host-out calls let every device copy its shard to the caller's buffer over its own PCIe link;
 * `_gather` calls collect the PCM in the memory of devices[0] instead ([n_streams][T] int16, e.g. from lpcnet_b200_device_alloc_on):
 * each finished chunk travels by peer DMA over NVLink while the next chunk is computed (the PCM sink above).
 * Use pinned host buffers (lpcnet_b200_host_alloc) so that the copies of different devices overlap. */
typedef struct LPCNetB200Multi LPCNetB200Multi;
LPCNET_EXPORT LPCNetB200Multi *lpcnet_b200_multi_create(int n_streams, const unsigned char *blob, int blob_len, const LPCNetB200Config *cfg,
                                                        const int *devices, int n_devices);
LPCNET_EXPORT void lpcnet_b200_multi_destroy(LPCNetB200Multi *m);
LPCNET_EXPORT int lpcnet_b200_multi_streams(const LPCNetB200Multi *m);
LPCNET_EXPORT int lpcnet_b200_multi_devices(const LPCNetB200Multi *m);
/* 1 if every device can write devices[0]'s memory directly (NVLink peer access); 0: gathers are staged by the driver */
LPCNET_EXPORT int lpcnet_b200_multi_peer_access(const LPCNetB200Multi *m);
/* shard k: its CUDA device and stream range [first, first + count) */
LPCNET_EXPORT int lpcnet_b200_multi_shard(const LPCNetB200Multi *m, int k, int *device, int *first, int *count);
/* the shard's batch, for the per-stream lifecycle calls (reset_streams, export/import_state, snapshots) with LOCAL stream ids */
LPCNET_EXPORT LPCNetB200Batch *lpcnet_b200_multi_batch(LPCNetB200Multi *m, int k);
LPCNET_EXPORT int lpcnet_b200_multi_reset(LPCNetB200Multi *m);
LPCNET_EXPORT int lpcnet_b200_multi_set_codebooks(LPCNetB200Multi *m, const float *cb, size_t n_floats);
/* same arguments as lpcnet_b200_batch_synthesize / _decode with n = all streams */
LPCNET_EXPORT int lpcnet_b200_multi_synthesize(LPCNetB200Multi *m, const float *features, int nframes, int feature_stride,
                                               int samples_per_frame, short *pcm);
LPCNET_EXPORT int lpcnet_b200_multi_decode(LPCNetB200Multi *m, const unsigned char *packets, int npackets, short *pcm);
/* host in, PCM gathered on devices[0]: d_pcm [n_streams][nframes*samples_per_frame] (resp. [n_streams][npackets*640]) */
LPCNET_EXPORT int lpcnet_b200_multi_synthesize_gather(LPCNetB200Multi *m, const float *features, int nframes, int feature_stride,
                                                      int samples_per_frame, short *d_pcm);
LPCNET_EXPORT int lpcnet_b200_multi_decode_gather(LPCNetB200Multi *m, const unsigned char *packets, int npackets, short *d_pcm);
/* contiguous range of shard k when n items are cut into `parts` (sizes differ by at most one; earlier shards take the remainder) */
LPCNET_EXPORT int lpcnet_b200_shard_range(int n, int k, int parts, int *first, int *count);
LPCNET_EXPORT void *lpcnet_b200_device_alloc_on(int device, size_t bytes);
/* CUDA streams for the `cuda_stream` argument of the `_device` entry points (for callers without their own CUDA binding).
 * The engine orders its state across streams itself: consecutive calls may use different streams. */
LPCNET_EXPORT void *lpcnet_b200_stream_create(void);
LPCNET_EXPORT void lpcnet_b200_stream_destroy(void *stream);
LPCNET_EXPORT int lpcnet_b200_stream_sync(void *stream);

/* == lpcnet_decode() per stream, `npackets` times ==
 * packets: [n_streams][npackets][8] bytes ; pcm: [n_streams][npackets*640] int16 */
LPCNET_EXPORT int lpcnet_b200_batch_decode(LPCNetB200Batch *b, const unsigned char *packets, int npackets, short *pcm);
LPCNET_EXPORT int lpcnet_b200_batch_decode_device(LPCNetB200Batch *b, const unsigned char *d_packets, int npackets,
                                                  short *d_pcm, void *cuda_stream);

/* == the analysis side, batched (SURVEY 8f N2): feature extraction and the 1.6 kb/s encoder ==
 * n independent LPCNetEncState streams (reference src/lpcnet_private.h:55-75) on one device, all starting from
 * lpcnet_encoder_create() (zeroed state, src/lpcnet_enc.c:471-482).  Results equal the reference's per-stream calls. */
typedef struct LPCNetB200EncBatch LPCNetB200EncBatch;
LPCNET_EXPORT LPCNetB200EncBatch *lpcnet_b200_enc_create(int n_streams, int device);
LPCNET_EXPORT void lpcnet_b200_enc_destroy(LPCNetB200EncBatch *e);
LPCNET_EXPORT int lpcnet_b200_enc_reset(LPCNetB200EncBatch *e);                      /* lpcnet_encoder_init() for every stream */
LPCNET_EXPORT int lpcnet_b200_enc_streams(const LPCNetB200EncBatch *e);
/* the VQ codebooks lpcnet_encode searches (same four arrays, same order as lpcnet_b200_batch_set_codebooks) */
LPCNET_EXPORT int lpcnet_b200_enc_set_codebooks(LPCNetB200EncBatch *e, const float *cb, size_t n_floats);
/* == lpcnet_compute_single_frame_features() per stream and frame (src/lpcnet_enc.c:919; `lpcnet_demo -features`) ==
 * pcm [n_streams][nframes*160] int16 (or float: lpcnet_compute_single_frame_features_float) -> features [n_streams][nframes][36]
 * (18 cepstral coefficients, pitch, pitch correlation, 16 LPC: the `.f32` feature-file row the synthesis side reads) */
LPCNET_EXPORT int lpcnet_b200_enc_compute_features(LPCNetB200EncBatch *e, const short *pcm, int nframes, float *features);
LPCNET_EXPORT int lpcnet_b200_enc_compute_features_float(LPCNetB200EncBatch *e, const float *pcm, int nframes, float *features);
LPCNET_EXPORT int lpcnet_b200_enc_compute_features_device(LPCNetB200EncBatch *e, const short *d_pcm, int nframes, float *d_features, void *cuda_stream);
/* == lpcnet_encode() per stream and 640-sample packet (src/lpcnet_enc.c:882) ==  pcm [n][npackets*640] -> packets [n][npackets][8] */
LPCNET_EXPORT int lpcnet_b200_enc_encode(LPCNetB200EncBatch *e, const short *pcm, int npackets, unsigned char *packets);
LPCNET_EXPORT int lpcnet_b200_enc_encode_device(LPCNetB200EncBatch *e, const short *d_pcm, int npackets, unsigned char *d_packets, void *cuda_stream);
/* == lpcnet_compute_features() (src/lpcnet_enc.c:896): unquantised 4-frame analysis ==  pcm [n][npackets*640] -> features [n][npackets*4][36] */
LPCNET_EXPORT int lpcnet_b200_enc_compute_features4(LPCNetB200EncBatch *e, const short *pcm, int npackets, float *features);
/* Test hook (host only): the analysis window and DCT table as the engine builds them (src/dump_lpcnet_tables.c:83-96): hw[160], dct[324] */
LPCNET_EXPORT void lpcnet_b200_enc_tables(float *half_window, float *dct);

/* ---- introspection used by the tests and the benchmark ---- */
/* Device time (ms, CUDA events on the engine's stream) the per-sample kernel took in the last synthesize/decode
 * call, summed over its launches; *launches receives how many engine kernels that call launched in total. */
LPCNET_EXPORT float lpcnet_b200_batch_last_sample_kernel_ms(const LPCNetB200Batch *b, int *launches);
/* CUDA-event stopwatch on the engine's stream, L2 eviction (256 MiB overwrite) and stream sync: what a benchmark
 * needs to time the engine on the device without any other CUDA binding. */
LPCNET_EXPORT int lpcnet_b200_batch_timer_start(LPCNetB200Batch *b);
LPCNET_EXPORT float lpcnet_b200_batch_timer_stop(LPCNetB200Batch *b);     /* ms since timer_start, <0 on error */
LPCNET_EXPORT int lpcnet_b200_batch_flush_l2(LPCNetB200Batch *b);
LPCNET_EXPORT int lpcnet_b200_batch_sync(LPCNetB200Batch *b);
/* Raw device / pinned-host memory for callers without their own CUDA binding. */
LPCNET_EXPORT void *lpcnet_b200_device_alloc(size_t bytes);
LPCNET_EXPORT void lpcnet_b200_device_free(void *p);
LPCNET_EXPORT int lpcnet_b200_memcpy_h2d(void *dst, const void *src, size_t bytes);
LPCNET_EXPORT int lpcnet_b200_memcpy_d2h(void *dst, const void *src, size_t bytes);
LPCNET_EXPORT void *lpcnet_b200_host_alloc(size_t bytes);                 /* pinned */
LPCNET_EXPORT void lpcnet_b200_host_free(void *p);

/* Measured peak of the unit that bounds the per-sample kernel, the L1/shared-memory data pipe: every SM streams
 * conflict-free LDS out of shared memory (lpcnet_b200/csrc/microbench.cu).  out[7] = {LDS.128 GB/s whole chip,
 * LDS.128 bytes/clk/SM, LDS.64 GB/s, LDS.64 B/clk/SM, LDS.32 GB/s, LDS.32 B/clk/SM, SM count}. */
LPCNET_EXPORT int lpcnet_b200_measure_smem_peak(int device, double *out);

/* Algorithmic bytes one synthesized sample of one stream must read (SURVEY.md 8d): total and the
 * sparse-GEMV-only subset (GRU_A weights + indices). */
LPCNET_EXPORT int lpcnet_b200_batch_algorithmic_bytes(const LPCNetB200Batch *b, long *total, long *sparse_gemv);
/* 1 if the loaded blob is the float (DISABLE_DOT_PROD) flavour, 0 for int8. */
LPCNET_EXPORT int lpcnet_b200_batch_is_float(const LPCNetB200Batch *b);
/* Copy the per-stream recurrent state of stream `s` to host (tests): gru_a[384], gru_b[16], last_sig[16],
 * misc[2]={last_exc, frame_count}, rng[4]. Any pointer may be NULL. */
LPCNET_EXPORT int lpcnet_b200_batch_get_state(LPCNetB200Batch *b, int s, float *gru_a, float *gru_b, float *last_sig,
                                              int *misc, uint32_t *rng);
/* Frame-network tap (tests): run ONLY the 100 Hz kernels (reference run_frame_network, src/lpcnet.c:82-120) on
 * host features [n][nframes<=16][feature_stride] and return gru_a_condition [n][nframes][1152], gru_b_condition
 * [n][nframes][48] and the gamma-weighted LPC [n][nframes][16] each frame's sample loop would use. */
LPCNET_EXPORT int lpcnet_b200_debug_frame_network(LPCNetB200Batch *b, const float *features, int nframes,
                                                  int feature_stride, float *ga, float *gb, float *lpc);
/* Test hook (host only, no CUDA): build the per-sample kernel's shared-memory image for a blob.  Returns the
 * image size or <0; layout[24] receives the offsets documented in lpcnet_b200/csrc/batch_api.cu.  layout[21] is 1 when
 * the model's range bound lets the int8 kernel round the GRU_A accumulators without the conversion unit (acc_init_t<true>,
 * lpcnet_b200/csrc/devmath.cuh), 0 when it converts with cvt (always 0 for float blobs); layout[22] is 1 for a float blob, whose
 * image and offsets are those of the lane==stream float kernel. */
LPCNET_EXPORT int lpcnet_b200_debug_image(const unsigned char *blob, int len, unsigned char *out, size_t cap,
                                          uint32_t *layout);

/* Same for the second image of float models (the neuron-per-lane kernel used for small batches); layout[17]. */
LPCNET_EXPORT int lpcnet_b200_debug_image_n(const unsigned char *blob, int len, unsigned char *out, size_t cap,
                                            uint32_t *layout);
/* Test hook: evaluate the engine's two implementations of the reference's _mm256_rcp_ps emulation (memory table /
 * table-free arithmetic) on n host floats. */
LPCNET_EXPORT int lpcnet_b200_debug_rcp(LPCNetB200Batch *b, const float *x, float *out_table, float *out_arith, int n);

/* Default model / codebooks for the lpcnet.h single-stream API (the reference compiles its model in; this
 * library loads it at run time).  Also settable through env LPCNET_B200_MODEL / LPCNET_B200_CODEBOOKS (file
 * paths) and LPCNET_B200_LPC_GAMMA. */
LPCNET_EXPORT int lpcnet_b200_set_default_model(const unsigned char *blob, int len, float lpc_gamma);
LPCNET_EXPORT int lpcnet_b200_set_default_codebooks(const float *cb, size_t n_floats);
/* Release the device resources behind a state that was set up with lpcnet_init() / lpcnet_decoder_init() on
 * caller-owned memory (reference include/lpcnet.h:160-169: get_size + init, no matching deinit).  Without this call they
 * are released at process exit, or when the same memory is initialised again.  `st` is the LPCNetState* (a
 * LPCNetDecState* may be passed as well: it starts with its LPCNetState, src/lpcnet_private.h:50-53). */
struct LPCNetState;
LPCNET_EXPORT void lpcnet_b200_deinit(struct LPCNetState *st);

#ifdef __cplusplus
}
#endif
#endif
