#!/usr/bin/env python3
"""Synthetic LPCNet model generator (TEST INFRASTRUCTURE — not a product path).

The reference ships no weights: `src/nnet_data.[ch]` and `src/ceps_codebooks.c` are downloaded by
`autogen.sh:9-10` / `download_model.sh:4-12`.  This script restates the *format* that
`training_tf2/dump_lpcnet.py` emits (array names, shapes, block-sparse packing, su-bias) and fills it
with deterministic random weights so that the untouched reference C sources, the CPU restatement in
`oracle/lpcnet_oracle.c` and the CUDA engine can all be run on identical inputs.

Format sources (reference file:line):
  * array names / shapes ............ training_tf2/dump_lpcnet.py:331-349 (gru_a_embed_*, *_dense_feature)
  * printSparseVector ............... training_tf2/dump_lpcnet.py:83-117  ([8 out][4 in] int8 blocks,
                                      [4 in][8 out] float blocks, idx = count,pos... per 8 rows)
  * dump_sparse_gru / su-bias ....... training_tf2/dump_lpcnet.py:124-149
  * dump_grub (dotp layout) ......... training_tf2/dump_lpcnet.py:58-59,151-183
  * dump_mdense_layer ............... training_tf2/dump_lpcnet.py:212-227 (transpose (0,2,1), (1,0))
  * conv1d / dense / embedding ...... training_tf2/dump_lpcnet.py:194-262
  * header (#defines, NNetState) .... training_tf2/dump_lpcnet.py:303-385
  * "DNNw" blob records ............. src/write_lpcnet_weights.c:47-67, src/nnet.h:41-61
  * int8 pair constraint ............ training_tf2/lpcnet.py:216-232 (WeightClip 0.992)
  * block densities (5,5,20)% ....... training_tf2/train_lpcnet.py (grua density), lpcnet.py:96-116
  * codebook shapes ................. src/lpcnet_dec.c:129-143 (1024x17 x3, 4096x18)

Outputs (into --out, default oracle/_gen):
  model_int8.bin   DOT_PROD flavour blob   (what the default reference build consumes)
  model_float.bin  DISABLE_DOT_PROD flavour blob (same weights, float block layout)
  codebooks.bin    4 float arrays, concatenated: cb1[1024*17] cb2[1024*17] cb3[1024*17] diff4[4096*18]
  nnet_data.h / nnet_data.c / plc_data.h / dred_rdovae_constants.h / ceps_codebooks.c
                   what the reference sources #include / link (nnet_data.c carries no arrays: the
                   reference is built with -DUSE_WEIGHTS_FILE and fed the blob)
"""
import argparse
import os
import struct
import numpy as np

N_A = 384          # GRU_A units   (training_tf2/lpcnet.py:234 rnn_units1)
N_B = 16           # GRU_B units   (rnn_units2)
COND = 128         # cond_size
EMBED = 128        # embed_size (lpcnet.py:47)
PITCH_EMBED = 64
NB_FEATURES = 20
FRAME_IN = NB_FEATURES + PITCH_EMBED   # 84
DENSITY = (0.05, 0.05, 0.20)           # z, r, h block densities
LPC_GAMMA = 0.9
FEATURES_DELAY = 2

WEIGHT_TYPE_float, WEIGHT_TYPE_int, WEIGHT_TYPE_qweight = 0, 1, 2


def _pair_clip_q(q):
    """q: int array [n_in][n_out]. Enforce |q[2k]|+|q[2k+1]| <= 127 along the input axis
    (the maddubs no-saturation condition, vec_avx.h:811-812 / lpcnet.py:216-232)."""
    q = q.copy()
    a = np.abs(q[0::2, :]) + np.abs(q[1::2, :])
    over = a > 127
    scale = np.where(over, 127.0 / np.maximum(a, 1), 1.0)
    q[0::2, :] = np.trunc(q[0::2, :] * scale).astype(np.int64)
    q[1::2, :] = np.trunc(q[1::2, :] * scale).astype(np.int64)
    assert (np.abs(q[0::2, :]) + np.abs(q[1::2, :])).max() <= 127
    return q


def _quantized_matrix(rng, n_in, n_out, sigma):
    q = np.rint(rng.normal(0.0, sigma * 128.0, size=(n_in, n_out))).astype(np.int64)
    q = np.clip(q, -127, 127)
    return _pair_clip_q(q)


def _sparse_pack(A, have_diag):
    """Restates printSparseVector (dump_lpcnet.py:83-117). A is float64 [n_in][n_out] whose entries are
    exact multiples of 1/128.  Returns dict(diag, w_int8, w_float, idx, AQ)."""
    A = A.copy()
    n_in, n_out = A.shape
    diag = None
    if have_diag:
        N = n_in
        diag = np.concatenate([np.diag(A[:, :N]), np.diag(A[:, N:2 * N]), np.diag(A[:, 2 * N:])])
        for k in range(3):
            A[:, k * N:(k + 1) * N] -= np.diag(np.diag(A[:, k * N:(k + 1) * N]))
    AQ = np.minimum(127, np.maximum(-128, np.round(A * 128))).astype(np.int64)
    idx = []
    w8 = []
    wf = []
    for i in range(n_out // 8):
        pos = len(idx)
        idx.append(-1)
        nnz = 0
        for j in range(n_in // 4):
            block = A[j * 4:(j + 1) * 4, i * 8:(i + 1) * 8]
            if np.sum(np.abs(block)) > 1e-10:
                nnz += 1
                idx.append(j * 4)
                w8.append(AQ[j * 4:(j + 1) * 4, i * 8:(i + 1) * 8].T.reshape(-1))   # [8 out][4 in]
                wf.append(block.reshape(-1))                                          # [4 in][8 out]
        idx[pos] = nnz
    return dict(diag=None if diag is None else diag.astype(np.float32),
                w_int8=np.concatenate(w8).astype(np.int8),
                w_float=np.concatenate(wf).astype(np.float32),
                idx=np.array(idx, dtype=np.int32), AQ=AQ)


def make_model(seed=1234, na=None, variant="", knobs=None):
    """Returns (arrays_common, arrays_int8, arrays_float): ordered lists of (name, type, ndarray).
    na      : GRU_A units (default 384; other sizes are the `--grua-size` models of training_tf2/train_lpcnet.py)
    variant : "" | "clamp" (sampling tree biased towards large excitation so that the output runs into the +-32767 clamp of
              lpcnet.c:265-269) | "dense" (GRU_A block densities 10/10/30 %)
    knobs   : hooks of the stress models (STRESS below); without them the random draws are exactly those of the regular models.
              density (z, r, h); a_mask(k, rng, N_A) -> bool [N_A/4 col blocks][N_A/8 row groups] of gate k or None (random);
              a_q(k, q, mask) -> int GRU_A gate matrix [in][out] after masking; b_in(q) / b_rec(q) -> GRU_B input / recurrent
              int matrix [in][out]; diag(k, d) -> GRU_A diagonal of gate k"""
    N_A = int(na or globals()["N_A"])
    kn = knobs or {}
    DENSITY = kn.get("density") or ((0.10, 0.10, 0.30) if variant == "dense" else globals()["DENSITY"])
    rng = np.random.default_rng(seed)
    f32 = np.float32
    common, only8, onlyf = [], [], []

    def fl(name, a):
        common.append((name, WEIGHT_TYPE_float, np.ascontiguousarray(a, dtype=f32)))

    # --- GRU_A input side: embedding tables pre-multiplied by the input kernel (dump_lpcnet.py:331-343)
    for nm in ("sig", "pred", "exc"):
        # smooth-ish in the u-law index so neighbouring levels behave similarly, plus noise
        base = rng.normal(0.0, 0.35, size=(8, 3 * N_A))
        t = np.linspace(0, 7, 256)
        i0 = np.minimum(6, np.floor(t).astype(int))
        fr = (t - i0)[:, None]
        tab = (1 - fr) * base[i0] + fr * base[i0 + 1] + rng.normal(0.0, 0.12, size=(256, 3 * N_A))
        fl("gru_a_embed_%s_weights" % nm, tab)
    fl("gru_a_dense_feature_weights", rng.normal(0.0, 0.08, size=(COND, 3 * N_A)))
    gru_a_bias = rng.normal(0.0, 0.15, size=(2, 3 * N_A))
    gru_a_bias[:, :N_A] += 0.3            # update gate biased towards keeping state (speech-like slow dynamics)
    fl("gru_a_dense_feature_bias", gru_a_bias[0])

    # --- GRU_B (dump_grub, dump_lpcnet.py:151-183)
    fl("gru_b_dense_feature_weights", rng.normal(0.0, 0.10, size=(COND, 3 * N_B)))
    fl("gru_b_dense_feature_bias", np.zeros(3 * N_B))
    qb_in = _quantized_matrix(rng, N_A, 3 * N_B, 0.09)
    if "b_in" in kn:
        qb_in = kn["b_in"](qb_in)
    pk = _sparse_pack(qb_in / 128.0, have_diag=False)
    only8.append(("gru_b_weights", WEIGHT_TYPE_qweight, pk["w_int8"]))
    onlyf.append(("gru_b_weights", WEIGHT_TYPE_qweight, pk["w_float"]))
    common.append(("gru_b_weights_idx", WEIGHT_TYPE_int, pk["idx"]))
    qb_rec = _quantized_matrix(rng, N_B, 3 * N_B, 0.25)
    if "b_rec" in kn:
        qb_rec = kn["b_rec"](qb_rec)
    # dotp layout: reshape (in/4,4,out/8,8) -> transpose (2,0,3,1) = [out/8][in/4][8][4]  (dump_lpcnet.py:58-59)
    dot = qb_rec.reshape(N_B // 4, 4, 3 * N_B // 8, 8).transpose(2, 0, 3, 1).reshape(-1)
    only8.append(("gru_b_recurrent_weights", WEIGHT_TYPE_qweight, dot.astype(np.int8)))
    onlyf.append(("gru_b_recurrent_weights", WEIGHT_TYPE_float, (qb_rec / 128.0).astype(f32).reshape(-1)))
    gru_b_bias = rng.normal(0.0, 0.15, size=(2, 3 * N_B))
    fl("gru_b_bias", gru_b_bias)
    sub = gru_b_bias.copy()
    sub[0, :] -= np.sum(pk["AQ"] * (1.0 / 128.0), axis=0)
    sub[1, :] -= np.sum(qb_rec * (1.0 / 128.0), axis=0)
    fl("gru_b_subias", sub)

    # --- layers dumped by the generic loop (dump_lpcnet.py:351-354)
    fl("embed_sig_weights", rng.normal(0.0, 0.3, size=(256, EMBED)))
    fl("embed_pitch_weights", rng.normal(0.0, 0.3, size=(256, PITCH_EMBED)))
    fl("feature_conv1_weights", rng.normal(0.0, 0.09, size=(3, FRAME_IN, COND)))
    fl("feature_conv1_bias", rng.normal(0.0, 0.1, size=(COND,)))
    fl("feature_conv2_weights", rng.normal(0.0, 0.07, size=(3, COND, COND)))
    fl("feature_conv2_bias", rng.normal(0.0, 0.1, size=(COND,)))
    fl("feature_dense1_weights", rng.normal(0.0, 0.12, size=(COND, COND)))
    fl("feature_dense1_bias", rng.normal(0.0, 0.1, size=(COND,)))
    fl("feature_dense2_weights", rng.normal(0.0, 0.12, size=(COND, COND)))
    fl("feature_dense2_bias", rng.normal(0.0, 0.1, size=(COND,)))

    # --- dual_fc (dump_mdense_layer, dump_lpcnet.py:212-227): kernel (256,16,2)->(256,2,16); bias,factor (256,2)->(2,256)
    kern = rng.normal(0.0, 0.35, size=(256, N_B, 2))
    bias = rng.normal(0.0, 0.10, size=(256, 2))
    factor = 1.6 + rng.normal(0.0, 0.15, size=(256, 2))
    # Shape the tree so the excitation pdf is unimodal around u-law 128 (SURVEY 8c): node i at level b
    # (i = (1<<b)|prefix).  If the first decision (MSB) was 1 push later bits towards 0 and vice versa.
    for i in range(2, 256):
        b = i.bit_length() - 1                 # level
        first = (i >> (b - 1)) & 1             # MSB decision already taken
        mag = 1.4 - 0.15 * b
        kern[i, :, :] *= min(1.0, 0.15 + 0.17 * b)   # coarse (large-amplitude) decisions depend less on the state
        bias[i, :] *= min(1.0, 0.15 + 0.17 * b)
        bias[i, :] += (-mag if first else mag) * (-0.25 if variant == "clamp" else 1.0)
    # the sign decision (node 1) must be unbiased or the output drifts to a rail through the 1/(1-0.85z^-1) de-emphasis
    kern[1, :, :] *= 0.15
    bias[1, :] = rng.normal(0.0, 0.01, size=2)
    # (variant "clamp": the level biases above push AWAY from the centre instead: large excitation, the de-emphasised
    # output runs into both rails)
    fl("dual_fc_weights", kern.transpose(0, 2, 1))
    fl("dual_fc_bias", bias.transpose(1, 0))
    fl("dual_fc_factor", factor.transpose(1, 0))

    # --- sparse GRU_A recurrent (dump_sparse_gru, dump_lpcnet.py:124-149)
    A = np.zeros((N_A, 3 * N_A))
    for k in range(3):
        nblk = (N_A // 4) * (N_A // 8)
        mask = kn["a_mask"](k, rng, N_A) if "a_mask" in kn else None
        if mask is None:
            keep = nblk - int(round(nblk * (1 - DENSITY[k])))
            chosen = rng.choice(nblk, size=keep, replace=False)
            mask = np.zeros(nblk, dtype=bool)
            mask[chosen] = True
            mask = mask.reshape(N_A // 4, N_A // 8)
        q = _quantized_matrix(rng, N_A, N_A, 0.17 if k < 2 else 0.13)
        # make sure every kept block is non-empty (dump drops all-zero blocks)
        full = np.repeat(np.repeat(mask, 4, axis=0), 8, axis=1)
        q = q * full
        if "a_q" in kn:
            q = kn["a_q"](k, q, mask)
        for (jb, ib) in zip(*np.nonzero(mask)):
            blk = q[jb * 4:(jb + 1) * 4, ib * 8:(ib + 1) * 8]
            # the diagonal is removed by the dump; a kept block must keep an off-diagonal non-zero
            offd = blk.copy()
            for a in range(4):
                for b_ in range(8):
                    if jb * 4 + a == ib * 8 + b_:
                        offd[a, b_] = 0
            if not offd.any():
                a, b_ = (0, 0) if (jb * 4 != ib * 8) else (1, 0)
                q[jb * 4 + a, ib * 8 + b_] = 1
        A[:, k * N_A:(k + 1) * N_A] = q / 128.0
        # diagonal (kept outside the block structure, float, not quantised)
        d = rng.normal(0.25 if k == 2 else 0.1, 0.2, size=N_A)
        if "diag" in kn:
            d = kn["diag"](k, d)
        A[:, k * N_A:(k + 1) * N_A] -= np.diag(np.diag(A[:, k * N_A:(k + 1) * N_A]))
        A[:, k * N_A:(k + 1) * N_A] += np.diag(d.astype(f32).astype(np.float64))
    # pair constraint must hold after diagonal removal as well (true: removing only lowers |q|)
    pk = _sparse_pack(A, have_diag=True)
    fl("sparse_gru_a_recurrent_weights_diag", pk["diag"])
    only8.append(("sparse_gru_a_recurrent_weights", WEIGHT_TYPE_qweight, pk["w_int8"]))
    onlyf.append(("sparse_gru_a_recurrent_weights", WEIGHT_TYPE_qweight, pk["w_float"]))
    common.append(("sparse_gru_a_recurrent_weights_idx", WEIGHT_TYPE_int, pk["idx"]))
    fl("sparse_gru_a_bias", gru_a_bias)
    sub = gru_a_bias.copy()
    sub[1, :] -= np.sum(pk["AQ"] * (1.0 / 128.0), axis=0)
    fl("sparse_gru_a_subias", sub)
    return common, only8, onlyf


def make_codebooks(seed=4321):
    rng = np.random.default_rng(seed)
    decay = np.exp(-np.arange(17) / 9.0)
    cb1 = rng.normal(0.0, 0.9, size=(1024, 17)) * decay
    cb2 = rng.normal(0.0, 0.45, size=(1024, 17)) * decay
    cb3 = rng.normal(0.0, 0.22, size=(1024, 17)) * decay
    d4 = rng.normal(0.0, 0.30, size=(4096, 18)) * np.exp(-np.arange(18) / 9.0)
    return [a.astype(np.float32) for a in (cb1, cb2, cb3, d4)]


def write_blob(path, arrays):
    """'DNNw' records: 64-byte header + payload padded to 64 (write_lpcnet_weights.c:47-67).  Written under a temporary name and
    renamed: several processes (one per GPU under torchrun) may regenerate the same deterministic file at the same time."""
    tmp = "%s.tmp%d" % (path, os.getpid())
    _write_blob(tmp, arrays)
    os.replace(tmp, path)


def _write_blob(path, arrays):
    with open(path, "wb") as f:
        f.write(blob_bytes(arrays))


def blob_bytes(arrays):
    out = []
    for name, typ, a in arrays:
        raw = a.tobytes()
        size = len(raw)
        block = (size + 63) // 64 * 64
        nm = name.encode()
        assert len(nm) < 44
        out += [struct.pack("<4siiii44s", b"DNNw", 0, typ, size, block, nm), raw, b"\0" * (block - size)]
    return b"".join(out)


# ---------------------------------------------------------------------------------------------------------------------------------
# Stress models (test inputs only).  The regular models above share one weight structure (random block masks at 5/5/20 %, dense GRU_B
# input, int8 weights well inside the pair constraint, GRU_A pre-activations far below 2^22 accumulator units); a trained model has
# uneven per-row density and weights at the WeightClip limit.  These models put the loader's and the kernels' edge cases into play:
#   holes / holes128  empty GRU_A lists (one neuron group with all three empty, most z lists empty so that some compute warps hold
#                     only empty z lists), lists of 1, 2, 3, 5, ... blocks; GRU_B input row groups of 0, 1, 3 and 5 blocks
#   one_class         lists whose column blocks all share one class (pos/4) & 3: the repeated-class and empty-slot paths of the quad dealer
#   skewed            density in four neuron groups: their compute warps fill their tensor-memory columns exactly (skewed_over: one
#                     quad more, refused)
#   denser            block densities 6/6/22 %: they load with fewer dual_fc rows in shared memory; denser_over, one step denser
#                     (6.25/6.25/22.5 %, same seed), needs more shared memory than one SM has and is refused
#   pair_edge         int8 weights -128 and same-sign pairs with |w0|+|w1| = 128 (pair_over_pos / pair_over_neg: one pair at 129, refused)
#   cvt_fast_edge     large recurrent su-biases and diagonals on neuron group 5 (candidate gate): the range bound of the conversion-free
#                     rounding lands just below its limit; cvt_exact_edge just above it
STRESS_NAMES = ("holes", "holes128", "one_class", "skewed", "denser", "pair_edge", "cvt_fast_edge", "cvt_exact_edge")
STRESS_REFUSED = ("skewed_over", "denser_over", "pair_over_pos", "pair_over_neg")
CVT_LIMIT = 4194304.0 * 0.99           # model.cu: fast_cvt = bound < 0.99 * 2^22
CVT_GROUP = 5                          # neuron group of the cvt models' large su-biases / diagonals


def _list_mask(rng, n_cols, lengths, cls=None):
    """bool [n_cols col blocks][len(lengths) row groups]: lengths[i] random column blocks for row group i (of class cls if given)."""
    m = np.zeros((n_cols, len(lengths)), bool)
    for i, n in enumerate(lengths):
        cand = np.arange(n_cols) if cls is None else np.arange(cls, n_cols, 4)
        m[rng.choice(cand, size=n, replace=False), i] = True
    return m


def _b_in_mask(q, lengths, rng, cls=None):
    """Keep lengths[rg] column blocks of GRU_B input row group rg (q: int [N_A][48]); every kept block non-zero."""
    q = q.copy()
    keep = _list_mask(rng, q.shape[0] // 4, lengths, cls)
    q *= np.repeat(np.repeat(keep, 4, axis=0), 8, axis=1)
    for jb, rg in zip(*np.nonzero(keep)):
        if not q[jb * 4:jb * 4 + 4, rg * 8:rg * 8 + 8].any():
            q[jb * 4, rg * 8] = 1
    return q


def _holes_knobs(na):
    ng, nc = na // 8, na // 4
    cyc = [1, 2, 3, 5, 0, 4, 7, 9, 1, 6, 13, 3, 2, 5, 8, 11]
    def a_mask(k, rng, N_A):
        if k == 0:      # z: only every fifth group has a list (so some compute warps hold no z block at all)
            L = [cyc[(i * 3) % len(cyc)] if i % 5 == 1 else 0 for i in range(ng)]
        else:
            L = [cyc[(i + 5 * k) % len(cyc)] for i in range(ng)]
        L[0] = 0                                  # neuron group 0: z, r and h lists all empty
        return _list_mask(rng, nc, L)
    brng = np.random.default_rng(77)
    return dict(a_mask=a_mask, b_in=lambda q: _b_in_mask(q, [0, 1, 3, 5, nc, nc // 2], brng))


def _one_class_knobs(na):
    ng, nc = na // 8, na // 4
    def a_mask(k, rng, N_A):
        m = np.zeros((nc, ng), bool)
        for i in range(ng):
            n = (1, 2, 3, 4, 5, 6, 7, 9, 12, 17, 0, 10)[(i + 4 * k) % 12] if i % 3 != 2 else 3 + (i + k) % 9
            # two of three groups: all blocks of one class; the others: any class
            m[:, i] = _list_mask(rng, nc, [n], cls=None if i % 3 == 2 else (i + k) % 4)[:, 0]
        return m
    brng = np.random.default_rng(78)
    return dict(a_mask=a_mask, b_in=lambda q: _b_in_mask(q, [nc // 4, 5, 1, nc // 4, 2, 7], brng, cls=1))


def _skewed_knobs(extra=0):
    """Four heavy neuron groups (z r h = 52 + extra, 52, 48 blocks = 38 quads); 28 light ones, 16 empty.  With the GRU_B input GEMV's
    12 quads the heavy groups' compute warps walk exactly 50 quads = 2 * (50 + 2) = 104 tensor-memory columns, all they have."""
    ng, nc = 48, 96
    def a_mask(k, rng, N_A):
        L = [0] * ng
        for i in range(ng):
            if i in (3, 17, 30, 41):
                L[i] = (52 + (extra if i == 3 else 0), 52, 48)[k]
            elif i % 3 != 0:
                L[i] = (2, 3, 5)[k] + (i % 4)
        return _list_mask(rng, nc, L)
    return dict(a_mask=a_mask)


def _pair_knobs(over=0):
    """Weights at the limits of the pair constraint in GRU_A (every gate), the GRU_B input and the GRU_B recurrent matrix.
    over=+1 / -1: one same-sign pair of GRU_A's candidate gate at |w0|+|w1| = 129 (positive / negative)."""
    pairs = [(-128, 0), (0, -128), (64, 64), (-64, -64), (127, 1), (-1, -127), (-128, 127), (100, 28), (-28, -100), (127, -128)]
    def put(q, slots):
        q = q.copy()
        for t, (r, c) in enumerate(slots):
            q[r, c], q[r + 1, c] = pairs[t % len(pairs)]
        return q
    def a_q(k, q, mask):
        slots = []
        for jb, ib in zip(*np.nonzero(mask)):
            for a in (0, 2):
                r, c = jb * 4 + a, ib * 8 + (len(slots) % 8)
                if r != c and r + 1 != c:
                    slots.append((r, c))
            if len(slots) >= 40:
                break
        q = put(q, slots)
        if over and k == 2:
            r, c = slots[-1]
            q[r, c], q[r + 1, c] = (64, 65) if over > 0 else (-128, -1)
        return q
    return dict(a_q=a_q,
                b_in=lambda q: put(q, [(2 * i, (5 * i) % 48) for i in range(0, 160, 7)]),
                b_rec=lambda q: put(q, [(2 * (i % 8), (7 * i) % 48) for i in range(20)]))


def _cvt_knobs():
    def diag(k, d):
        if k == 2:
            d = d.copy()
            d[8 * CVT_GROUP:8 * CVT_GROUP + 8] = 40.0 + np.arange(8)
        return d
    return dict(diag=diag)


def _int8_dense(w8, idx, n_in, n_out):
    M = np.zeros((n_out, n_in), np.int64)
    p = wp = 0
    for rg in range(n_out // 8):
        nb = idx[p]; p += 1
        for _ in range(nb):
            pos = idx[p]; p += 1
            M[rg * 8:rg * 8 + 8, pos:pos + 4] = w8[wp:wp + 32].reshape(8, 4); wp += 32
    return M


def cvt_bound(common, only8):
    """model.cu's range bound of the GRU_A accumulators (conversion-free rounding iff bound < CVT_LIMIT), in the same double arithmetic."""
    a = {n: v for n, _, v in common + only8}
    na = a["sparse_gru_a_recurrent_weights_diag"].size // 3
    f64 = lambda n: a[n].astype(np.float64)
    cmax = (np.abs(f64("gru_a_dense_feature_bias")) + np.abs(f64("gru_a_dense_feature_weights")).sum(axis=0)).max()
    bmax = np.abs(f64("sparse_gru_a_subias")[1]).max()
    dmax = np.abs(f64("sparse_gru_a_recurrent_weights_diag")).max()
    emax = max(np.abs(f64("gru_a_embed_%s_weights" % s)).max() for s in ("sig", "pred", "exc"))
    W = _int8_dense(a["sparse_gru_a_recurrent_weights"].astype(np.int64), a["sparse_gru_a_recurrent_weights_idx"], na, 3 * na)
    smax = np.abs(W).sum(axis=1).max()
    return (bmax + dmax + cmax + 3 * emax) * 1.01 * (128.0 * 127.0) + 255.0 * smax + 2


def _set_cvt_bias(common, only8, ratio):
    """Recurrent su-biases of neuron group CVT_GROUP's candidate gate (sign alternating, the largest on its first neuron) such that
    cvt_bound = ratio * CVT_LIMIT; the float flavour's recurrent bias gets the same value plus the su-bias correction."""
    a = {n: v for n, _, v in common}
    sub, bias = a["sparse_gru_a_subias"], a["sparse_gru_a_bias"]
    na = sub.shape[1] // 3
    cols = 2 * na + 8 * CVT_GROUP + np.arange(8)
    corr = bias[1, cols].astype(np.float64) - sub[1, cols].astype(np.float64)       # sum(AQ)/128 of those rows
    sub[1, cols] = 0
    rest = cvt_bound(common, only8) - 1.01 * 128.0 * 127.0 * np.abs(sub[1].astype(np.float64)).max()
    b = (ratio * CVT_LIMIT - rest) / (1.01 * 128.0 * 127.0)
    vals = b * (1.0 - 0.02 * np.arange(8)) * np.where(np.arange(8) % 2 == 0, 1.0, -1.0)
    sub[1, cols] = vals.astype(np.float32)
    bias[1, cols] = (vals + corr).astype(np.float32)


def make_stress_model(name):
    """(common, only8, onlyf) of a stress model (STRESS_NAMES, STRESS_REFUSED)."""
    if name in ("holes", "holes128"):
        na = 128 if name == "holes128" else 384
        return make_model(2001, na=na, knobs=_holes_knobs(na))
    if name == "one_class":
        return make_model(2002, knobs=_one_class_knobs(384))
    if name in ("skewed", "skewed_over"):
        return make_model(2003, knobs=_skewed_knobs(extra=4 if name == "skewed_over" else 0))
    if name in ("denser", "denser_over"):
        return make_model(2004, knobs=dict(density=(0.06, 0.06, 0.22) if name == "denser" else (0.0625, 0.0625, 0.225)))
    if name in ("pair_edge", "pair_over_pos", "pair_over_neg"):
        return make_model(2005, knobs=_pair_knobs({"pair_edge": 0, "pair_over_pos": 1, "pair_over_neg": -1}[name]))
    if name in ("cvt_fast_edge", "cvt_exact_edge"):
        common, only8, onlyf = make_model(2006, knobs=_cvt_knobs())
        _set_cvt_bias(common, only8, 0.995 if name == "cvt_fast_edge" else 1.005)
        return common, only8, onlyf
    raise KeyError(name)


def stress_na(name):
    return 128 if name == "holes128" else 384


def stress_blob(name, kind="int8"):
    """DNNw blob of a stress model: kind int8 | float."""
    common, only8, onlyf = make_stress_model(name)
    return blob_bytes(common + (only8 if kind == "int8" else onlyf))


NNET_DATA_H = """/* Generated by oracle/gen_model.py in the format of training_tf2/dump_lpcnet.py:303-385 */
#ifndef RNN_DATA_H
#define RNN_DATA_H

#include "nnet.h"

{e2e_lines}

/* LPC weighting factor */
#define LPC_GAMMA {gamma}f

/* Features look-ahead */
#define FEATURES_DELAY {delay}

#define GRU_A_EMBED_SIG_OUT_SIZE {n3a}
#define GRU_A_EMBED_PRED_OUT_SIZE {n3a}
#define GRU_A_EMBED_EXC_OUT_SIZE {n3a}
#define GRU_A_DENSE_FEATURE_OUT_SIZE {n3a}
#define GRU_B_DENSE_FEATURE_OUT_SIZE {n3b}
#define EMBED_SIG_OUT_SIZE {embed}
#define EMBED_PITCH_OUT_SIZE {pembed}
#define FEATURE_CONV1_OUT_SIZE {cond}
#define FEATURE_CONV1_STATE_SIZE ({fin}*2)
#define FEATURE_CONV1_DELAY 1
#define FEATURE_CONV2_OUT_SIZE {cond}
#define FEATURE_CONV2_STATE_SIZE ({cond}*2)
#define FEATURE_CONV2_DELAY 1
#define FEATURE_DENSE1_OUT_SIZE {cond}
#define FEATURE_DENSE2_OUT_SIZE {cond}
#define GRU_A_OUT_SIZE {na}
#define GRU_A_STATE_SIZE {na}
#define GRU_B_OUT_SIZE {nb}
#define GRU_B_STATE_SIZE {nb}
#define DUAL_FC_OUT_SIZE 256
#define SPARSE_GRU_A_OUT_SIZE {na}
#define SPARSE_GRU_A_STATE_SIZE {na}
#define MAX_RNN_NEURONS {na}

#define MAX_CONV_INPUTS {maxconv}

#define MAX_MDENSE_TMP 512

typedef struct {{
  float feature_conv1_state[FEATURE_CONV1_STATE_SIZE];
  float feature_conv2_state[FEATURE_CONV2_STATE_SIZE];
  float gru_a_state[GRU_A_STATE_SIZE];
  float gru_b_state[GRU_B_STATE_SIZE];
}} NNetState;

typedef struct {{
  EmbeddingLayer gru_a_embed_sig;
  EmbeddingLayer gru_a_embed_pred;
  EmbeddingLayer gru_a_embed_exc;
  DenseLayer gru_a_dense_feature;
  DenseLayer gru_b_dense_feature;
  GRULayer gru_b;
  EmbeddingLayer embed_sig;
  EmbeddingLayer embed_pitch;
  Conv1DLayer feature_conv1;
  Conv1DLayer feature_conv2;
  DenseLayer feature_dense1;
  DenseLayer feature_dense2;
  MDenseLayer dual_fc;
  SparseGRULayer sparse_gru_a;
}} LPCNetModel;

int init_lpcnet_model(LPCNetModel *model, const WeightArray *arrays);

#endif
"""

NNET_DATA_C = """/* Generated by oracle/gen_model.py in the format of training_tf2/dump_lpcnet.py (init sequence :147,181,199,224,242,252).
   No arrays: the oracle build defines USE_WEIGHTS_FILE and loads the DNNw blob. */
#include "nnet.h"
#include "nnet_data.h"

#ifndef DUMP_BINARY_WEIGHTS
int init_lpcnet_model(LPCNetModel *model, const WeightArray *arrays) {{
  if (embedding_init(&model->gru_a_embed_sig, arrays, "gru_a_embed_sig_weights", 256, {n3a})) return 1;
  if (embedding_init(&model->gru_a_embed_pred, arrays, "gru_a_embed_pred_weights", 256, {n3a})) return 1;
  if (embedding_init(&model->gru_a_embed_exc, arrays, "gru_a_embed_exc_weights", 256, {n3a})) return 1;
  if (dense_init(&model->gru_a_dense_feature, arrays, "gru_a_dense_feature_bias", "gru_a_dense_feature_weights", {cond}, {n3a}, ACTIVATION_LINEAR)) return 1;
  if (dense_init(&model->gru_b_dense_feature, arrays, "gru_b_dense_feature_bias", "gru_b_dense_feature_weights", {cond}, {n3b}, ACTIVATION_LINEAR)) return 1;
  if (gru_init(&model->gru_b, arrays, "gru_b_bias", "gru_b_subias", "gru_b_weights", "gru_b_weights_idx", "gru_b_recurrent_weights", {na}, {nb}, ACTIVATION_TANH, 1)) return 1;
  if (embedding_init(&model->embed_sig, arrays, "embed_sig_weights", 256, {embed})) return 1;
  if (embedding_init(&model->embed_pitch, arrays, "embed_pitch_weights", 256, {pembed})) return 1;
  if (conv1d_init(&model->feature_conv1, arrays, "feature_conv1_bias", "feature_conv1_weights", {fin}, 3, {cond}, ACTIVATION_TANH)) return 1;
  if (conv1d_init(&model->feature_conv2, arrays, "feature_conv2_bias", "feature_conv2_weights", {cond}, 3, {cond}, ACTIVATION_TANH)) return 1;
  if (dense_init(&model->feature_dense1, arrays, "feature_dense1_bias", "feature_dense1_weights", {cond}, {cond}, ACTIVATION_TANH)) return 1;
  if (dense_init(&model->feature_dense2, arrays, "feature_dense2_bias", "feature_dense2_weights", {cond}, {cond}, ACTIVATION_TANH)) return 1;
  if (mdense_init(&model->dual_fc, arrays, "dual_fc_bias",  "dual_fc_weights",  "dual_fc_factor",  {nb}, 256, 2, ACTIVATION_SIGMOID)) return 1;
  if (sparse_gru_init(&model->sparse_gru_a, arrays, "sparse_gru_a_bias", "sparse_gru_a_subias", "sparse_gru_a_recurrent_weights_diag", "sparse_gru_a_recurrent_weights", "sparse_gru_a_recurrent_weights_idx",  {na}, ACTIVATION_TANH, 1)) return 1;
  return 0;
}}
#endif
"""

PLC_DATA_H = """/* stub: nnet.c:42 and lpcnet_private.h:9 include plc_data.h; the PLC model is out of scope */
#ifndef PLC_DATA_H
#define PLC_DATA_H
#include "nnet.h"
#define PLC_MAX_RNN_NEURONS 1
typedef struct { float plc_gru1_state[1]; float plc_gru2_state[1]; } PLCNetState;
typedef struct { int unused; } PLCModel;
#endif
"""

DRED_H = """/* stub: nnet.c:41 includes dred_rdovae_constants.h; DRED is out of scope */
#ifndef DRED_RDOVAE_CONSTANTS_H
#define DRED_RDOVAE_CONSTANTS_H
#define DRED_MAX_RNN_NEURONS 1
#define DRED_MAX_CONV_INPUTS 1
#endif
"""


def write_c_sources(out, na=None, e2e=False, delay=None, gamma=None):
    na = int(na or N_A)
    e2e_lines = ("/* This is an end-to-end model */\n#define END2END" if e2e
                 else "/* This is *not* an end-to-end model */\n/* #define END2END */")
    fmt = dict(gamma=repr(LPC_GAMMA if gamma is None else gamma), delay=FEATURES_DELAY if delay is None else delay, n3a=3 * na, n3b=3 * N_B,
               embed=EMBED, pembed=PITCH_EMBED, cond=COND, fin=FRAME_IN, na=na, nb=N_B, maxconv=3 * COND, e2e_lines=e2e_lines)
    open(os.path.join(out, "nnet_data.h"), "w").write(NNET_DATA_H.format(**fmt))
    open(os.path.join(out, "nnet_data.c"), "w").write(NNET_DATA_C.format(**fmt))
    open(os.path.join(out, "plc_data.h"), "w").write(PLC_DATA_H)
    open(os.path.join(out, "dred_rdovae_constants.h"), "w").write(DRED_H)


def _cfloat(x):
    t = "%.9g" % float(x)
    if not any(c in t for c in ".en"):
        t += "."
    return t + "f"


def write_codebook_c(path, cbs):
    names = ("ceps_codebook1", "ceps_codebook2", "ceps_codebook3", "ceps_codebook_diff4")
    with open(path, "w") as f:
        f.write("/* Generated by oracle/gen_model.py: synthetic VQ codebooks (the real ceps_codebooks.c is not in the reference tree) */\n")
        for nm, a in zip(names, cbs):
            v = a.reshape(-1)
            f.write("float %s[%d] = {\n" % (nm, v.size))
            for i in range(0, v.size, 8):
                f.write("  " + ", ".join(_cfloat(x) for x in v[i:i + 8]) + ",\n")
            f.write("};\n")


# Model variants used by the tests (tag -> generator arguments).  Tags whose header differs from the default one
# (sizes, END2END, FEATURES_DELAY) get their own directory oracle/_gen_<tag> and their own compiled reference
# oracle/_ref/liblpcnet_ref_{A,B}_<tag>.so (oracle/Makefile, target `ref`).
VARIANTS = {
    "na256":  dict(na=256),                               # --grua-size 256
    "na128":  dict(na=128),
    "e2e":    dict(e2e=True, delay=2, gamma=1.0),         # END2END: LPC from the network's reflection coefficients (lpcnet.c:57-78,107-108)
    "delay0": dict(delay=0),                              # FEATURES_DELAY 0: no look-ahead, LPC of the current frame (lpcnet.c:113-115)
    "na256e2e": dict(na=256, e2e=True, delay=0, gamma=0.95),
}


def generate(out, seed=1234, c_sources=True, na=None, e2e=False, delay=None, gamma=None):
    os.makedirs(out, exist_ok=True)
    common, only8, onlyf = make_model(seed, na=na)
    write_blob(os.path.join(out, "model_int8.bin"), common + only8)
    write_blob(os.path.join(out, "model_float.bin"), common + onlyf)
    if na is None:      # same header, other weights: the +-32767 clamp fixture
        c2, o8, _ = make_model(seed, variant="clamp")
        write_blob(os.path.join(out, "model_int8_clamp.bin"), c2 + o8)
    cbs = make_codebooks()
    tmp = os.path.join(out, "codebooks.bin.tmp%d" % os.getpid())
    with open(tmp, "wb") as f:
        for a in cbs:
            f.write(a.tobytes())
    os.replace(tmp, os.path.join(out, "codebooks.bin"))
    if c_sources:
        write_c_sources(out, na=na, e2e=e2e, delay=delay, gamma=gamma)
        write_codebook_c(os.path.join(out, "ceps_codebooks.c"), cbs)
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "_gen"))
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--no-c", action="store_true")
    ap.add_argument("--variant", default="", help="one of VARIANTS (default: the 384/16 model); output goes to <out>_<variant>")
    a = ap.parse_args()
    if a.variant:
        generate(a.out + "_" + a.variant, a.seed, not a.no_c, **VARIANTS[a.variant])
        print("generated into", a.out + "_" + a.variant)
    else:
        generate(a.out, a.seed, not a.no_c)
        print("generated into", a.out)
