"""CPU tests of the stress models (oracle/gen_model.py make_stress_model): weight structures the regular synthetic models never have
(empty and short block lists, lists of one column class, a compute warp at its tensor-memory budget, a model one density step short
of the shared-memory limit, int8 weights at the pair-constraint limit, GRU_A pre-activations next to the range bound of the conversion-free rounding).  The generator is
pinned by blob hashes, the CPU restatement by the compiled reference's output on these blobs (tests/golden/stress.npz), and the host
side of the engine by replaying the shared-memory image it builds against the dense matrices of each model."""
import ctypes
import hashlib
import os
import sys
import numpy as np
import pytest
import helpers as H
import gen_model
from fixtures import make_features

sys.path.insert(0, os.path.join(H.GOLDEN))
import make_golden_stress as MG      # noqa: E402  (the inputs the goldens were made from)

INT8_NAMES = list(gen_model.STRESS_NAMES)


@pytest.fixture(scope="module")
def L():
    from lpcnet_b200 import build, api
    build.build()
    L = api.lib()
    L.lpcnet_b200_debug_image.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
    L.lpcnet_b200_debug_image_n.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
    return L


@pytest.fixture(scope="module")
def gold():
    return dict(np.load(os.path.join(H.GOLDEN, "stress.npz")))


def _image(L, blob):
    out = np.zeros(256 * 1024, np.uint8)
    lay = np.zeros(24, np.uint32)
    r = L.lpcnet_b200_debug_image(blob, len(blob), out.ctypes.data, out.size, lay.ctypes.data)
    return r, out, lay


def _arrays(name, kind="int8"):
    common, only8, onlyf = gen_model.make_stress_model(name)
    return {n: a for n, _, a in common + (only8 if kind == "int8" else onlyf)}


def _lists(idx, nrows):
    """block-column positions per 8-row group of an index array"""
    out, p = [], 0
    for _ in range(nrows // 8):
        nb = int(idx[p]); out.append([int(v) for v in idx[p + 1:p + 1 + nb]]); p += nb + 1
    return out


# ---------------------------------------------------------------- generator and oracle pinned to the reference ----------------------------------------------------------------
@pytest.mark.parametrize("kind", ["int8", "float"])
@pytest.mark.parametrize("name", gen_model.STRESS_NAMES)
def test_generator_reproduces_pinned_blobs(gold, name, kind):
    assert hashlib.sha256(H.stress_blob(name, kind)).digest() == gold["sha_%s_%s" % (name, kind)].tobytes(), \
        "gen_model.make_stress_model(%r) no longer produces the blob the goldens were made from" % name


@pytest.mark.parametrize("kind,build", [("int8", "A"), ("float", "B")])
@pytest.mark.parametrize("name", gen_model.STRESS_NAMES)
def test_oracle_matches_reference_on_stress_models(gold, name, kind, build):
    f = MG.stress_features()
    np.testing.assert_array_equal(H.digests(f[None]), gold["features"])
    got = H.oracle_synth(f, kind, stress=name)
    bad = np.nonzero(H.stream_digests(got) != gold["ref_%s_%s" % (name, build)])[0]
    assert bad.size == 0, "%s %s: streams %s differ from the reference" % (name, kind, bad.tolist())
    assert np.abs(got[:, 480:]).max() > 1000


@pytest.mark.parametrize("kind,build", [("int8", "A"), ("float", "B")])
def test_oracle_matches_reference_with_clamped_pitch(gold, kind, build):
    """pitch periods below 33 and above 255 read the embedding's clamp rows (lpcnet.c:93-94)"""
    f = MG.pitch_features()
    np.testing.assert_array_equal(H.digests(f[None]), gold["pitch_features"])
    p = np.floor(.1 + (np.float32(50) * f[:, :, 18]).astype(np.float64) + 100)
    assert (p < 33).any() and (p > 255).any()
    np.testing.assert_array_equal(H.stream_digests(H.oracle_synth(f, kind, stress="holes")), gold["ref_holes_pitch_%s" % build])


@pytest.mark.parametrize("build", ["A", "B"])
@pytest.mark.parametrize("name", ["holes", "holes128"])
def test_oracle_plc_call_sequence_on_holes(gold, name, build):
    import scenarios as S
    kind = "float" if build == "B" else "int8"
    script = S.plc_like_script(MG.PLC_FRAMES)
    for stream in (0, 3):
        got = S.run_single("oracle", H.oracle_lib(), S.OracleState(kind, stress=name), make_features(stream, MG.PLC_FRAMES), stream, script)
        np.testing.assert_array_equal(H.stream_digests(got[None]), gold["plc_%s_%s_s%d" % (name, build, stream)])


# ---------------------------------------------------------------- the structures the models are meant to have ----------------------------------------------------------------
def test_holes_models_have_empty_and_short_lists():
    for name, na in (("holes", 384), ("holes128", 128)):
        a = _arrays(name)
        ng = na // 8
        lists = _lists(a["sparse_gru_a_recurrent_weights_idx"], 3 * na)
        z, r, h = lists[:ng], lists[ng:2 * ng], lists[2 * ng:]
        assert not z[0] and not r[0] and not h[0]                            # a neuron group with no block at all
        assert sum(not l for l in z) >= ng // 2                              # most z lists empty
        lens = {len(l) for l in lists}
        assert {1, 2, 3, 5} <= lens and {n % 4 for n in lens} == {0, 1, 2, 3}
        lb = [len(l) for l in _lists(a["gru_b_weights_idx"], 48)]
        assert lb[:4] == [0, 1, 3, 5] and lb[4] == na // 4                   # GRU_B input row groups: empty, shorter than the K split, odd, full


def test_one_class_model_has_single_class_lists():
    a = _arrays("one_class")
    lists = _lists(a["sparse_gru_a_recurrent_weights_idx"], 3 * 384)
    one = [l for l in lists if len(l) >= 2 and len({(p // 4) & 3 for p in l}) == 1]
    assert len(one) >= 48 and max(len(l) for l in one) >= 9
    lb = _lists(a["gru_b_weights_idx"], 48)
    assert all(len({(p // 4) & 3 for p in l}) == 1 for l in lb) and len(lb[0]) == 24


def test_pair_edge_model_reaches_the_pair_limit_everywhere():
    a = _arrays("pair_edge")
    for nm in ("sparse_gru_a_recurrent_weights", "gru_b_weights", "gru_b_recurrent_weights"):
        q = a[nm].astype(np.int64)
        p0, p1 = q[0::2], q[1::2]
        same = (p0 >= 0) == (p1 >= 0)
        assert q.min() == -128, nm
        assert ((np.abs(p0) + np.abs(p1) == 128) & same & (p0 > 0)).any(), nm
        assert ((np.abs(p0) + np.abs(p1) == 128) & same & (p0 < 0)).any(), nm
        assert not (same & (np.abs(p0) + np.abs(p1) > 128)).any(), nm


# ---------------------------------------------------------------- what the engine's loader makes of them ----------------------------------------------------------------
def _xs_offset(c, s):
    return c * 128 + (((((s >> 4) & 1) << 6) | ((s & 7) << 3)) ^ (((c & 1) << 6) | ((c & 2) << 4))) + ((s >> 3) & 1) * 4


def _dense_int8(w8, idx, nrows, ncols):
    M = np.zeros((nrows, ncols), np.int64)
    for rg, lst in enumerate(_lists(idx, nrows)):
        for pos in lst:
            M[rg * 8:rg * 8 + 8, pos:pos + 4] = w8[:32].reshape(8, 4); w8 = w8[32:]
    return M


@pytest.mark.parametrize("name", INT8_NAMES)
def test_int8_image_replays_to_the_dense_model(L, name):
    """Walk the int8 image like the kernel (warp -> slot -> gate -> quads; (row group, K part) for GRU_B), with two random u8 inputs:
    the integer GEMVs equal the dense matrices of the model.  Also: the warp's lists are contiguous in the kernel's walk order, every
    compute warp's quads + 2 tail quads + parked state fit its 128 tensor-memory columns, and padding quads carry zero weights."""
    a = _arrays(name)
    r, img, lay = _image(L, H.stress_blob(name))
    assert r > 0, L.lpcnet_b200_last_error()
    wA, metaA, wB, metaB, image_bytes, total, nA, nB, SM_IMAGE, PARA, DIRA, GRPA, DIRB, WBREC, PARB, FCW, NWC, GPW, FCN, KP, NA = [int(v) for v in lay[:21]]
    na = gen_model.stress_na(name)
    assert NA == na and r == image_bytes and total == SM_IMAGE + image_bytes and total <= 227 * 1024 and FCN in (8, 16, 32, 64)
    img = img[:image_bytes]
    rel = lambda o: o - SM_IMAGE
    MA = _dense_int8(a["sparse_gru_a_recurrent_weights"].astype(np.int64), a["sparse_gru_a_recurrent_weights_idx"], 3 * na, na)
    MB = _dense_int8(a["gru_b_weights"].astype(np.int64), a["gru_b_weights_idx"], 48, na)
    rng = np.random.default_rng(1)
    X = np.stack([rng.integers(0, 256, na), np.full(na, 255)], axis=1)      # [na][2]: random and all-255 inputs
    dirA = img[DIRA:DIRA + NWC * GPW * 3 * 2 * 4].view(np.uint32).reshape(NWC, GPW, 3, 2)
    grpA = img[GRPA:GRPA + NWC * GPW * 4].view(np.uint32).reshape(NWC, GPW)
    parA = img[PARA:PARA + NWC * GPW * 3 * 16 * 4].view(np.float32).reshape(NWC, GPW, 3, 2, 8)
    dirB = img[DIRB:DIRB + 6 * KP * 2 * 4].view(np.uint32).reshape(6 * KP, 2)
    wAi = img[rel(wA):rel(wA) + nA * 128].view(np.int8).astype(np.int64).reshape(nA, 8, 4, 4)      # [quad][out][slot][in]
    mA = img[rel(metaA):rel(metaA) + nA * 8].view(np.uint16).reshape(nA, 4)
    wBi = img[rel(wB):rel(wB) + nB * 128].view(np.int8).astype(np.int64).reshape(nB, 8, 4, 4)
    mB = img[rel(metaB):rel(metaB) + nB * 8].view(np.uint16).reshape(nB, 4)

    def replay(wq, mq, q0, nq):
        acc = np.zeros((8, 2), np.int64)
        for q in range(q0, q0 + nq):
            for t in range(4):
                e = int(mq[q, t]); c = e >> 7
                assert e == _xs_offset(c, 0) and c < na // 4
                acc += wq[q, :, t, :] @ X[4 * c:4 * c + 4]
        return acc
    assert sorted(grpA.reshape(-1).tolist()) == list(range(na // 8))
    got = np.zeros((3 * na, 2), np.int64)
    for w in range(NWC):
        q = int(dirA[w, 0, 1, 0])
        for sl in range(GPW):
            for gate in (1, 2):
                assert int(dirA[w, sl, gate, 0]) == q; q += int(dirA[w, sl, gate, 1])
        for sl in range(GPW):
            assert int(dirA[w, sl, 0, 0]) == q; q += int(dirA[w, sl, 0, 1])
        for sl in range(GPW):
            g = int(grpA[w, sl])
            for gate in range(3):
                rows = slice(gate * na + 8 * g, gate * na + 8 * g + 8)
                got[rows] += replay(wAi, mA, int(dirA[w, sl, gate, 0]), int(dirA[w, sl, gate, 1]))
                assert int(dirA[w, sl, gate, 1]) == (int(np.count_nonzero(np.abs(MA[rows]).sum(axis=0).reshape(-1, 4).sum(axis=1))) + 3) // 4
                np.testing.assert_array_equal(parA[w, sl, gate, 0], a["sparse_gru_a_subias"][1, rows])
                np.testing.assert_array_equal(parA[w, sl, gate, 1], a["sparse_gru_a_recurrent_weights_diag"][rows])
        quads = int(dirA[w, :, :, 1].sum()) + (int(dirB[w, 1]) if w < 6 * KP else 0)
        assert 2 * (quads + 2) + 8 * GPW <= 128, "compute warp %d: %d quads" % (w, quads)
    np.testing.assert_array_equal(got, MA @ X)
    gotB = np.zeros((48, 2), np.int64)
    for rg in range(6):
        for part in range(KP):
            gotB[rg * 8:rg * 8 + 8] += replay(wBi, mB, int(dirB[rg * KP + part, 0]), int(dirB[rg * KP + part, 1]))
    np.testing.assert_array_equal(gotB, MB @ X)
    np.testing.assert_array_equal(img[WBREC:WBREC + 768].view(np.int8), a["gru_b_recurrent_weights"])
    np.testing.assert_array_equal(img[PARB:PARB + 96 * 4].view(np.float32), a["gru_b_subias"].reshape(-1))


@pytest.mark.parametrize("name", INT8_NAMES)
def test_float_neuron_image_replays_to_the_dense_model(L, name):
    """Float flavour, image of the neuron-per-lane kernel: the fp16 blocks walked per (group, gate) and per GRU_B row group give the
    dense float matrices; the dense-GRU_B flag is set only when every GRU_B row group holds all column blocks in order."""
    a = _arrays(name, "float")
    na = gen_model.stress_na(name)
    blob = H.stress_blob(name, "float")
    out = np.zeros(300000, np.uint8); lay = (ctypes.c_uint32 * 32)()
    r = L.lpcnet_b200_debug_image_n(blob, len(blob), out.ctypes.data, out.size, lay)
    assert r > 0, L.lpcnet_b200_last_error()
    wA, metaA, wB, metaB, image_bytes, total, nA, nB, IMG, NEUR, DIRA, PARA, DIRB, PARB, WBREC, FCW, dense, NA = [int(v) for v in lay[:18]]
    assert NA == na and total <= 227 * 1024
    img = out[:image_bytes]
    rel = lambda o: o - IMG

    def dense_from_sparse(w, idx, nrows, ncols):
        M = np.zeros((nrows, ncols)); wp = 0
        for rg, lst in enumerate(_lists(idx, nrows)):
            for pos in lst:
                M[rg * 8:rg * 8 + 8, pos:pos + 4] = w[wp:wp + 32].reshape(4, 8).T; wp += 32
        return M
    MA = dense_from_sparse(a["sparse_gru_a_recurrent_weights"].astype(np.float64), a["sparse_gru_a_recurrent_weights_idx"], 3 * na, na)
    MB = dense_from_sparse(a["gru_b_weights"].astype(np.float64), a["gru_b_weights_idx"], 48, na)
    ng = na // 8
    dirA = img[DIRA:DIRA + ng * 3 * 2 * 4].view(np.uint32).reshape(ng, 3, 2)
    blkA = img[rel(wA):rel(wA) + max(nA, 1) * 64].view(np.float16).astype(np.float64).reshape(-1, 8, 4)
    mA = img[rel(metaA):rel(metaA) + max(nA, 1) * 2].view(np.uint16)
    got = np.zeros((3 * na, na))
    for g in range(ng):
        for q in range(3):
            for b in range(int(dirA[g, q, 0]), int(dirA[g, q, 0] + dirA[g, q, 1])):
                pos = int(mA[b]) // 4
                got[q * na + 8 * g:q * na + 8 * g + 8, pos:pos + 4] += blkA[b]
    np.testing.assert_array_equal(got, MA)
    dirB = img[DIRB:DIRB + 48].view(np.uint32).reshape(6, 2)
    blkB = img[rel(wB):rel(wB) + max(nB, 1) * 64].view(np.float16).astype(np.float64).reshape(-1, 8, 4)
    mB = img[rel(metaB):rel(metaB) + max(nB, 1) * 2].view(np.uint16)
    gotB = np.zeros((48, na))
    for rg in range(6):
        for b in range(int(dirB[rg, 0]), int(dirB[rg, 0] + dirB[rg, 1])):
            gotB[rg * 8:rg * 8 + 8, int(mB[b]) // 4:int(mB[b]) // 4 + 4] += blkB[b]
    np.testing.assert_array_equal(gotB, MB)
    full = all(l == list(range(0, na, 4)) for l in _lists(a["gru_b_weights_idx"], 48))
    assert bool(dense) == full


@pytest.mark.parametrize("name", INT8_NAMES + [""])
def test_float_lane_stream_image_replays_to_the_dense_model(L, name):
    """Float flavour, image of the lane==stream kernel (sample_kernel_f32.cu; "" = the regular model): lists in the order (warp, slot,
    gate z r h), each padded to an even number of fp16 blocks [4 in][8 out] with zero blocks; GRU_B row groups whole in K part 0.
    Walking it like the kernel gives the dense float matrices, the recurrent biases and diagonals of the owned groups."""
    if name:
        a, na, blob = _arrays(name, "float"), gen_model.stress_na(name), H.stress_blob(name, "float")
    else:
        common, _, onlyf = gen_model.make_model()
        a, na, blob = {n: v for n, _, v in common + onlyf}, 384, H.blob("float")
    r, img, lay = _image(L, blob)
    assert r > 0, L.lpcnet_b200_last_error()
    wA, metaA, wB, metaB, image_bytes, total, nA, nB, IMG, PARA, DIRA, GRPA, DIRB, WBREC, PARB, FCW, NWC, GPW, FCN, KP, NA, FAST, ISF = [int(v) for v in lay[:23]]
    assert ISF == 1 and FAST == 0 and FCN == 0 and NA == na and NWC * GPW * 8 == na and r == image_bytes and total == IMG + image_bytes and total <= 227 * 1024
    img = img[:image_bytes]
    rel = lambda o: o - IMG

    def dense_from_sparse(w, idx, nrows, ncols):
        M = np.zeros((nrows, ncols)); wp = 0
        for rg, lst in enumerate(_lists(idx, nrows)):
            for pos in lst:
                M[rg * 8:rg * 8 + 8, pos:pos + 4] = w[wp:wp + 32].reshape(4, 8).T; wp += 32
        return M
    MA = dense_from_sparse(a["sparse_gru_a_recurrent_weights"].astype(np.float64), a["sparse_gru_a_recurrent_weights_idx"], 3 * na, na)
    MB = dense_from_sparse(a["gru_b_weights"].astype(np.float64), a["gru_b_weights_idx"], 48, na)
    lists = _lists(a["sparse_gru_a_recurrent_weights_idx"], 3 * na)
    dirA = img[DIRA:DIRA + NWC * GPW * 3 * 2 * 4].view(np.uint32).reshape(NWC, GPW, 3, 2)
    grpA = img[GRPA:GRPA + NWC * GPW * 4].view(np.uint32).reshape(NWC, GPW)
    parA = img[PARA:PARA + NWC * GPW * 3 * 16 * 4].view(np.float32).reshape(NWC, GPW, 3, 2, 8)
    blk = lambda w0, n: img[rel(w0):rel(w0) + n * 64].view(np.float16).astype(np.float64).reshape(n, 4, 8)   # [block][in][out]
    bA, mA = blk(wA, nA), img[rel(metaA):rel(metaA) + nA * 2].view(np.uint16)
    assert sorted(grpA.reshape(-1).tolist()) == list(range(na // 8))
    got = np.zeros((3 * na, na)); b_next = 0
    for w in range(NWC):
        for sl in range(GPW):
            g = int(grpA[w, sl])
            for gate in range(3):
                b0, nb = int(dirA[w, sl, gate, 0]), int(dirA[w, sl, gate, 1])
                n_real = len(lists[gate * (na // 8) + g])
                assert b0 == b_next and nb == n_real + (n_real & 1)             # contiguous, padded to even length
                b_next += nb
                rows = slice(gate * na + 8 * g, gate * na + 8 * g + 8)
                for b in range(b0, b0 + nb):
                    assert mA[b] % 512 == 0
                    pos = int(mA[b]) // 128
                    got[rows, pos:pos + 4] += bA[b].T
                if nb > n_real:
                    assert not bA[b0 + nb - 1].any()                              # the padding block contributes exactly 0
                np.testing.assert_array_equal(parA[w, sl, gate, 0], a["sparse_gru_a_bias"][1, rows])
                np.testing.assert_array_equal(parA[w, sl, gate, 1], a["sparse_gru_a_recurrent_weights_diag"][rows])
    assert b_next == nA
    np.testing.assert_array_equal(got, MA)
    dirB = img[DIRB:DIRB + 6 * KP * 2 * 4].view(np.uint32).reshape(6, KP, 2)
    bB, mB = blk(wB, nB), img[rel(metaB):rel(metaB) + nB * 2].view(np.uint16)
    gotB = np.zeros((48, na))
    for rg, lst in enumerate(_lists(a["gru_b_weights_idx"], 48)):
        assert int(dirB[rg, 0, 1]) == len(lst) + (len(lst) & 1) and (dirB[rg, 1:, 1] == 0).all()
        for b in range(int(dirB[rg, 0, 0]), int(dirB[rg, 0, 0] + dirB[rg, 0, 1])):
            gotB[rg * 8:rg * 8 + 8, int(mB[b]) // 128:int(mB[b]) // 128 + 4] += bB[b].T
    np.testing.assert_array_equal(gotB, MB)
    np.testing.assert_array_equal(img[WBREC:WBREC + 768 * 4].view(np.float32), a["gru_b_recurrent_weights"])
    np.testing.assert_array_equal(img[PARB:PARB + 96 * 4].view(np.float32), a["gru_b_bias"].reshape(-1))


def test_holes_images_have_empty_z_warps_and_empty_gru_b_parts(L):
    for name in ("holes", "holes128"):
        r, img, lay = _image(L, H.stress_blob(name))
        NWC, GPW, KP = int(lay[16]), int(lay[17]), int(lay[19])
        img = img[:r]
        dirA = img[int(lay[10]):int(lay[10]) + NWC * GPW * 24].view(np.uint32).reshape(NWC, GPW, 3, 2)
        dirB = img[int(lay[12]):int(lay[12]) + 6 * KP * 8].view(np.uint32).reshape(6, KP, 2)
        assert any((dirA[w, :, 0, 1] == 0).all() for w in range(NWC)), "%s: no compute warp with only empty z lists" % name
        assert (dirA[:, :, :, 1].sum(axis=2) == 0).any()                    # a slot whose three lists are empty
        assert (dirB[0, :, 1] == 0).all() and dirB[1, 0, 1] == 1 and dirB[1, 1, 1] == 0   # empty row group; one block: second K part empty


def test_skewed_model_fills_a_compute_warp_and_one_more_quad_is_refused(L):
    r, img, lay = _image(L, H.stress_blob("skewed"))
    assert r > 0, L.lpcnet_b200_last_error()
    NWC, GPW, KP = int(lay[16]), int(lay[17]), int(lay[19])
    dirA = img[int(lay[10]):int(lay[10]) + NWC * GPW * 24].view(np.uint32).reshape(NWC, GPW, 3, 2)
    dirB = img[int(lay[12]):int(lay[12]) + 6 * KP * 8].view(np.uint32).reshape(6 * KP, 2)
    room = 128 - 8 * GPW
    cols = [2 * (int(dirA[w, :, :, 1].sum()) + (int(dirB[w, 1]) if w < 6 * KP else 0) + 2) for w in range(NWC)]
    assert room - 4 <= max(cols) <= room, cols
    assert _image(L, gen_model.stress_blob("skewed_over"))[0] < 0
    assert b"tensor-memory columns" in L.lpcnet_b200_last_error()


def test_denser_model_loads_with_fewer_dual_fc_rows_and_one_step_more_is_refused(L):
    """denser (6/6/22 %) keeps fewer dual_fc rows in shared memory to fit; denser_over (6.25/6.25/22.5 %, same seed) no longer fits one
    SM in either flavour even with the fewest rows, and is refused with a message"""
    r, img, lay = _image(L, H.stress_blob("denser"))
    assert r > 0 and int(lay[18]) in (8, 16, 32) and int(lay[5]) <= 227 * 1024
    assert _image(L, H.stress_blob("denser", "float"))[0] > 0
    for kind in ("int8", "float"):
        assert _image(L, gen_model.stress_blob("denser_over", kind))[0] < 0
        assert b"shared memory" in L.lpcnet_b200_last_error(), kind


@pytest.mark.parametrize("name", ["pair_over_pos", "pair_over_neg"])
def test_one_pair_over_the_limit_is_refused(L, name):
    assert _image(L, H.stress_blob("pair_edge"))[0] > 0
    assert _image(L, gen_model.stress_blob(name))[0] < 0
    assert b"pair constraint" in L.lpcnet_b200_last_error()


@pytest.mark.parametrize("name,fast", [("cvt_fast_edge", 1), ("cvt_exact_edge", 0), ("holes", 1), ("pair_edge", 1), ("denser", 1)])
def test_conversion_free_rounding_chosen_by_the_range_bound(L, name, fast):
    """layout[21]: the loader's choice between the conversion-free accumulator rounding and cvt; the two edge models sit 0.5 % below /
    above the bound's limit (gen_model.cvt_bound restates model.cu's bound)"""
    common, only8, _ = gen_model.make_stress_model(name)
    ratio = gen_model.cvt_bound(common, only8) / gen_model.CVT_LIMIT
    r, _, lay = _image(L, H.stress_blob(name))
    assert r > 0 and int(lay[21]) == fast and (ratio < 1) == bool(fast)
    if name.startswith("cvt_"):
        assert 0.99 < ratio < 1.01
    assert int(_image(L, H.blob("int8"))[2][21]) == 1


def test_cvt_fast_edge_accumulators_exceed_2_21_during_synthesis():
    """The model picked for the conversion-free rounding with the bound just below its limit really drives the GRU_A accumulators past
    2^21 (and, as the bound proves, below 2^22) in synthesis: measured by the CPU restatement on the golden inputs."""
    Lo = H.oracle_lib()
    f = MG.stress_features()
    for name in ("cvt_fast_edge", "cvt_exact_edge"):
        peak = 0
        for s in range(len(f)):
            st = Lo.oracle_state_create(H.oracle_model("int8", "", name))
            pcm = np.zeros(160, np.int16)
            for t in range(f.shape[1]):
                Lo.oracle_synthesize(st, f[s, t].ctypes.data, pcm.ctypes.data, 160)
            peak = max(peak, Lo.oracle_acc_peak(st))
            Lo.oracle_state_destroy(st)
        assert 2 ** 21 < peak < 2 ** 22, (name, peak)
