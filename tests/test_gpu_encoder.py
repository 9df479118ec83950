"""GPU tests (-m gpu) of the analysis side (SURVEY 8f N2): batched feature extraction and the 1.6 kb/s encoder
(lpcnet_b200_enc_*, csrc/enc_kernels.cu) against the reference's lpcnet_compute_single_frame_features / lpcnet_encode /
lpcnet_compute_features (src/lpcnet_enc.c).  The bar is the same as on the synthesis side: every feature float and every packet
byte equal to the reference's (goldens produced by the compiled reference, tests/golden/make_golden_enc.py, and digests of its
output on fresh inputs, tests/golden/make_golden_ref_checks.py).  Floats are compared as bit patterns."""
import ctypes
import os
import subprocess
import numpy as np
import pytest
import helpers as H
from fixtures import make_pcm_batch

pytestmark = pytest.mark.gpu
G = np.load(os.path.join(H.GOLDEN, "enc_A.npz"))


@pytest.fixture(scope="module")
def eng():
    import lpcnet_b200
    from lpcnet_b200 import build
    build.build()
    assert lpcnet_b200.device_count() > 0, "GPU test selected but no CUDA device is visible"
    return lpcnet_b200


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def assert_same_floats(got, want, what):
    d = np.argwhere(bits(got) != bits(want))
    assert d.size == 0, "%s: %d floats differ, first at %s: got %r want %r" % (what, len(d), tuple(d[0]), got[tuple(d[0])], want[tuple(d[0])])


def test_single_frame_features_match_reference_golden(eng):
    e = eng.EncBatch(8)
    got = e.compute_features(G["pcm"])
    e.close()
    assert_same_floats(got, G["features"], "lpcnet_compute_single_frame_features")


def test_features_stream_in_uneven_chunks_and_ragged_batch(eng):
    """State carries across calls (analysis overlap, pitch history, Viterbi path); a batch that does not fill a warp of blocks."""
    pcm = G["pcm"][:5]
    e = eng.EncBatch(5)
    parts, t = [], 0
    for k in (1, 7, 3, 16, 13):
        parts.append(e.compute_features(pcm[:, t * 160:(t + k) * 160])); t += k
    assert t == 40
    assert_same_floats(np.concatenate(parts, axis=1), G["features"][:5], "chunked features")
    e.reset()
    assert_same_floats(e.compute_features(pcm[:, :1600]), G["features"][:5, :10], "after reset")
    e.close()


def test_float_input_equals_int16_input(eng):
    e = eng.EncBatch(3)
    got = e.compute_features(G["pcm"][:3].astype(np.float32))
    e.close()
    assert_same_floats(got, G["features"][:3], "lpcnet_compute_single_frame_features_float")


def test_encoder_packets_match_reference_golden(eng):
    e = eng.EncBatch(8, codebooks=H.codebooks())
    got = e.encode(G["pcm"])
    np.testing.assert_array_equal(got, G["packets"])
    # packet by packet on a fresh state: the same bytes
    e.reset()
    one = np.concatenate([e.encode(G["pcm"][:, p * 640:(p + 1) * 640]) for p in range(10)], axis=1)
    np.testing.assert_array_equal(one, G["packets"])
    e.close()


def test_encode_needs_codebooks(eng):
    e = eng.EncBatch(2)
    with pytest.raises(eng.LPCNetB200Error, match="codebooks"):
        e.encode(G["pcm"][:2, :640])
    e.close()


def test_unquantised_superframe_features_match_reference_golden(eng):
    e = eng.EncBatch(8)
    got = e.compute_features4(G["pcm"])
    e.close()
    assert_same_floats(got, G["features4"], "lpcnet_compute_features")


def test_mixed_call_sequence_on_one_state(eng):
    """lpcnet_encode leaves pcount at 3; single-frame analysis afterwards keeps using that sub-frame slot, like the reference."""
    e = eng.EncBatch(2, codebooks=H.codebooks())
    pk = e.encode(G["pcm"][:2, :3 * 640])
    f = e.compute_features(G["pcm"][:2, 3 * 640:3 * 640 + 28 * 160])
    e.close()
    np.testing.assert_array_equal(pk, G["mixed_packets"])
    assert_same_floats(f, G["mixed_features"], "single-frame analysis after lpcnet_encode")


def test_single_stream_drop_in_api(eng):
    """include/lpcnet.h: lpcnet_encoder_create / lpcnet_encode / lpcnet_compute_single_frame_features / lpcnet_compute_features."""
    L = eng.lib()
    for fn in ("lpcnet_encoder_create",):
        getattr(L, fn).restype = ctypes.c_void_p
    L.lpcnet_encoder_destroy.argtypes = [ctypes.c_void_p]
    L.lpcnet_encode.argtypes = [ctypes.c_void_p] * 3
    L.lpcnet_compute_single_frame_features.argtypes = [ctypes.c_void_p] * 3
    L.lpcnet_compute_features.argtypes = [ctypes.c_void_p] * 3
    cb = H.codebooks()
    assert L.lpcnet_b200_set_default_codebooks(cb.ctypes.data, cb.size) == 0
    pcm = np.ascontiguousarray(G["pcm"][1])
    st = L.lpcnet_encoder_create()
    assert st
    buf = np.zeros(8, np.uint8)
    for p in range(4):
        assert L.lpcnet_encode(st, pcm[p * 640:].ctypes.data, buf.ctypes.data) == 0
        np.testing.assert_array_equal(buf, G["packets"][1, p])
    L.lpcnet_encoder_destroy(st)
    st = L.lpcnet_encoder_create()
    f = np.zeros(36, np.float32)
    for t in range(6):
        assert L.lpcnet_compute_single_frame_features(st, pcm[t * 160:].ctypes.data, f.ctypes.data) == 0
        assert_same_floats(f, G["features"][1, t], "frame %d" % t)
    L.lpcnet_encoder_destroy(st)
    st = L.lpcnet_encoder_create()
    f4 = np.zeros((4, 36), np.float32)
    assert L.lpcnet_compute_features(st, pcm.ctypes.data, f4.ctypes.data) == 0
    assert_same_floats(f4, G["features4"][1, :4], "lpcnet_compute_features")
    L.lpcnet_encoder_destroy(st)
    assert L.lpcnet_encoder_get_size() >= 16


def test_codec_round_trip_through_both_engines(eng):
    """PCM -> lpcnet_b200_enc_encode -> packets -> lpcnet_b200_batch_decode -> PCM: equals the oracle's decode of the reference's
    packets (the encoder's packets are the reference's, the decoder is bit-exact), and the output is not silence."""
    e = eng.EncBatch(4, codebooks=H.codebooks())
    pk = e.encode(G["pcm"][:4])
    e.close()
    b = eng.Batch(4, H.blob("int8"), lpc_gamma=H.LPC_GAMMA, codebooks=H.codebooks())
    out = b.decode(pk)
    b.close()
    np.testing.assert_array_equal(out, H.oracle_decode(G["packets"][:4], "int8"))
    assert np.abs(out[:, 640:]).max() > 0


def test_fresh_inputs_against_the_oracle_port(eng):
    """48 other streams x 40 frames against the CPU restatement (oracle/lpcnet_enc_oracle.inc, pinned to the reference by the CPU suite)."""
    n, T = 48, 40
    pcm = make_pcm_batch(range(300, 300 + n), T)
    e = eng.EncBatch(n, codebooks=H.codebooks())
    f = e.compute_features(pcm)
    e.reset()
    pk = e.encode(pcm)
    e.reset()
    f4 = e.compute_features4(pcm)
    e.close()
    assert_same_floats(f, H.oracle_features(pcm), "features vs oracle port")
    np.testing.assert_array_equal(pk, H.oracle_encode(pcm))
    assert_same_floats(f4, H.oracle_encode(pcm, features4=True), "features4 vs oracle port")


def test_fresh_inputs_against_the_compiled_reference(eng):
    """96 other streams x 60 frames (15 packets): features and packets equal what the compiled reference returned, stream by stream."""
    n, T = 96, 60
    pcm = make_pcm_batch(range(100, 100 + n), T)
    H.assert_ref_digests(pcm, "gpu_enc_pcm", "test inputs")
    e = eng.EncBatch(n, codebooks=H.codebooks())
    f = e.compute_features(pcm)
    e.reset()
    pk = e.encode(pcm)
    e.close()
    H.assert_ref_digests(f, "gpu_enc_features", "features, fresh streams")
    H.assert_ref_digests(pk, "gpu_enc_packets", "packets, fresh streams")


@pytest.mark.skipif(not os.path.exists(os.path.join(H.ORACLE, "_ref", "lpcnet_demo_b200")), reason="reference CLI linked against liblpcnet_b200.so not built")
def test_reference_cli_features_and_encode_modes_run_on_the_engine(eng, tmp_path):
    """The UNTOUCHED src/lpcnet_demo.c linked against liblpcnet_b200.so: `-features` writes the .f32 rows and `-encode` the packet
    stream the reference CLI itself would write."""
    demo = os.path.join(H.ORACLE, "_ref", "lpcnet_demo_b200")
    pcm = G["pcm"][2]
    (tmp_path / "in.s16").write_bytes(pcm.tobytes())
    env = dict(os.environ, LPCNET_B200_CODEBOOKS=os.path.join(H.gen_dir(), "codebooks.bin"))
    subprocess.run([demo, "-features", str(tmp_path / "in.s16"), str(tmp_path / "out.f32")], check=True, env=env, timeout=300)
    got = np.fromfile(tmp_path / "out.f32", np.float32).reshape(-1, 36)
    assert_same_floats(got, G["features"][2, :len(got)], "lpcnet_demo -features")
    assert len(got) >= 39
    subprocess.run([demo, "-encode", str(tmp_path / "in.s16"), str(tmp_path / "out.lpcnet")], check=True, env=env, timeout=300)
    pk = np.fromfile(tmp_path / "out.lpcnet", np.uint8).reshape(-1, 8)
    np.testing.assert_array_equal(pk, G["packets"][2, :len(pk)])
    assert len(pk) >= 9
