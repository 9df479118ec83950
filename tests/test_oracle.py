"""CPU tests (-m "not gpu"): pin the oracle restatement (oracle/lpcnet_oracle.c).

 * against the committed golden vectors produced by the untouched reference (tests/golden/make_golden.py);
 * against what the compiled reference returned for the inputs used here (tests/golden/make_golden_ref_checks.py);
 * unit-level: tables (FFT twiddles/bitrev, DCT), activations, u-law, frame network taps.
"""
import hashlib
import json
import os
import numpy as np
import pytest
import helpers as H
from fixtures import make_feature_batch, make_packets


def test_model_blobs_are_deterministic():
    dig = json.load(open(os.path.join(H.GOLDEN, "digests.json")))
    assert hashlib.sha256(H.blob("int8")).hexdigest() == dig["model_int8_sha256"]
    assert hashlib.sha256(H.blob("float")).hexdigest() == dig["model_float_sha256"]
    assert hashlib.sha256(H.codebooks().tobytes()).hexdigest() == dig["codebooks_sha256"]


def test_oracle_matches_golden_int8():
    gold = np.load(os.path.join(H.GOLDEN, "synth_A.npz"))["pcm"]
    got = H.oracle_synth(make_feature_batch(range(4), 40), "int8")
    assert (gold[:, :320] == 0).all()            # FEATURES_DELAY warm-up frames are silent (lpcnet.c:239-243)
    assert np.abs(gold[:, 320:]).max() > 1000    # the fixture is not degenerate
    np.testing.assert_array_equal(got, gold)


def test_oracle_matches_golden_float():
    gold = np.load(os.path.join(H.GOLDEN, "synth_B.npz"))["pcm"]
    got = H.oracle_synth(make_feature_batch(range(4), 40), "float")
    np.testing.assert_array_equal(got, gold)


def test_oracle_matches_golden_decode():
    gold = np.load(os.path.join(H.GOLDEN, "decode_A.npz"))["pcm"]
    got = H.oracle_decode(np.stack([make_packets(s, 6) for s in range(3)]), "int8")
    np.testing.assert_array_equal(got, gold)


def test_oracle_matches_golden_digests():
    dig = json.load(open(os.path.join(H.GOLDEN, "digests.json")))
    big = make_feature_batch(range(16), 150)
    assert hashlib.sha256(H.oracle_synth(big, "int8").tobytes()).hexdigest() == dig["synth_A_16x150"]
    assert hashlib.sha256(H.oracle_synth(big, "float").tobytes()).hexdigest() == dig["synth_B_16x150"]
    pk = np.stack([make_packets(s, 25) for s in range(8)])
    assert hashlib.sha256(H.oracle_decode(pk, "int8").tobytes()).hexdigest() == dig["decode_A_8x25"]


def test_int8_pair_constraint_and_sparsity():
    """The synthetic model respects WeightClip (lpcnet.py:216-232) so maddubs cannot saturate, and hits the
    (5,5,20)% block densities => 1382 blocks (SURVEY 8d)."""
    import gen_model
    common, only8, _ = gen_model.make_model()
    arrs = {n: a for n, _, a in common + only8}
    w = arrs["sparse_gru_a_recurrent_weights"].astype(np.int32).reshape(-1, 8, 4)
    assert w.shape[0] == 1382
    assert (np.abs(w[:, :, 0]) + np.abs(w[:, :, 1])).max() <= 127
    assert (np.abs(w[:, :, 2]) + np.abs(w[:, :, 3])).max() <= 127
    idx = arrs["sparse_gru_a_recurrent_weights_idx"]
    assert idx.size == 144 + 1382
    wb = arrs["gru_b_weights"].astype(np.int32).reshape(-1, 8, 4)
    assert wb.shape[0] == 576
    assert (np.abs(wb[:, :, 0]) + np.abs(wb[:, :, 1])).max() <= 127


def test_tables_match_reference():
    L = H.oracle_lib()
    tw = np.zeros(640, np.float32); br = np.zeros(320, np.int32); dct = np.zeros(324, np.float32)
    lg = np.zeros(256, np.float32); u2l = np.zeros(256, np.float32)
    L.oracle_get_tables(H.oracle_model(), tw.ctypes.data, br.ctypes.data, dct.ctypes.data, lg.ctypes.data, u2l.ctypes.data)
    R = H.ref_checks()                   # kiss_fft_state of the reference's 320-point FFT, its dct_table, ulaw2lin(0..255)
    assert list(R["kfft_factors"]) == [5, 64, 4, 16, 4, 4, 4, 1]
    np.testing.assert_array_equal(R["kfft_bitrev"], br)
    np.testing.assert_array_equal(R["kfft_twiddles"].view(np.uint32), tw.view(np.uint32))
    np.testing.assert_array_equal(R["dct_table"].view(np.uint32), dct.view(np.uint32))
    np.testing.assert_array_equal(R["ulaw2lin"].view(np.uint32), u2l.view(np.uint32))


def test_activations_and_ulaw_match_reference():
    L, m = H.oracle_lib(), H.oracle_model()
    x, v = H.activation_test_inputs()
    np.testing.assert_array_equal(np.concatenate([H.digests(x[None]), H.digests(v[None])]), H.ref_checks()["act_inputs"], "test inputs changed")
    H.assert_ref_digests(np.array([L.oracle_tanh(m, float(t)) for t in x], dtype=np.float32)[None], "act_tanh", "tanh (compute_activation)")
    H.assert_ref_digests(np.array([L.oracle_sigmoid(m, float(t)) for t in x], dtype=np.float32)[None], "act_sigmoid", "sigmoid (compute_activation)")
    H.assert_ref_digests(np.array([L.oracle_lin2ulaw(float(t)) for t in v], np.int32)[None], "act_lin2ulaw", "lin2ulaw")


def test_frame_network_matches_reference():
    L = H.oracle_lib()
    f = make_feature_batch([5], 12)[0]
    H.assert_ref_digests(f[None], "fn_features", "test inputs")
    ga = np.zeros((12, 1152), np.float32); gb = np.zeros((12, 48), np.float32); lpc = np.zeros((12, 16), np.float32)
    st = L.oracle_state_create(H.oracle_model())
    for t in range(12):
        L.oracle_frame_network(st, f[t].ctypes.data, ga[t].ctypes.data, gb[t].ctypes.data, lpc[t].ctypes.data)
    L.oracle_state_destroy(st)
    H.assert_ref_digests(ga, "fn_gru_a", "gru_a conditioning per frame")
    H.assert_ref_digests(gb, "fn_gru_b", "gru_b conditioning per frame")
    want = H.ref_checks()["fn_lpc"]
    np.testing.assert_array_equal(lpc.view(np.uint32), want.view(np.uint32))
    assert np.abs(want[3:]).max() > 0.1


@pytest.mark.parametrize("build,kind", [("A", "int8"), ("B", "float")])
def test_oracle_matches_reference_fresh_streams(build, kind):
    f = make_feature_batch(range(100, 106), 80)      # streams not in the other goldens
    H.assert_ref_digests(f[None], "fresh_features", "test inputs")
    H.assert_ref_digests(H.oracle_synth(f, kind), "fresh_" + build, "PCM per stream")


def test_decode_packet_matches_reference():
    L = H.oracle_lib()
    st = L.oracle_state_create(H.oracle_model())
    pk = make_packets(77, 40)
    H.assert_ref_digests(pk[None], "dec_packets", "test inputs")
    fo = np.zeros((40, 4, 36), np.float32)
    for t in range(40):
        L.oracle_decode_packet(st, fo[t].ctypes.data, pk[t].ctypes.data)
    L.oracle_state_destroy(st)
    H.assert_ref_digests(fo, "dec_features", "decoded features per packet")


def test_rcpps_table_closed_form():
    """The captured Intel RCPPS table (tests/golden/rcpps_table.bin, compiled into the engine) is exactly
    T[k] = rint(2^25 / (2k + 4097)) * 2^-13 for the 2048 mantissa bins — evidence that it is a property of the
    instruction, not of one machine."""
    t = H.rcp_table().astype(np.int64)
    k = np.arange(2048, dtype=np.int64)
    m13 = (2 ** 25 + (2 * k + 4097) // 2) // (2 * k + 4097)            # rint(2^25 / d), d odd => no ties
    want = (np.float32(1.0) * (m13.astype(np.float64) / 8192.0)).astype(np.float32).view(np.uint32).astype(np.int64)
    np.testing.assert_array_equal(t, want)


def test_oracle_port_matches_at_size_digests_on_a_sample_of_streams():
    """The per-stream digests of the reference at BASELINE sizes (tests/golden/at_size_digests.npz) also pin the CPU
    restatement: a few streams of every workload, full duration (1000 frames => frame_count saturation, lpcnet.c:119)."""
    import os
    from fixtures import make_feature_batch, make_packets
    dig = np.load(os.path.join(H.GOLDEN, "at_size_digests.npz"))
    ids = [0, 777, 4095]
    got = H.oracle_synth(make_feature_batch(ids, 100), "int8")
    np.testing.assert_array_equal(H.stream_digests(got), dig["config3_int8"][ids])
    ids = [3, 255]
    got = H.oracle_synth(make_feature_batch(ids, 1000), "float")
    np.testing.assert_array_equal(H.stream_digests(got), dig["config2_float"][ids])
    ids = [5, 1023]
    got = H.oracle_decode(np.stack([make_packets(s, 250) for s in ids]), "int8")
    np.testing.assert_array_equal(H.stream_digests(got), dig["config5_decode"][ids])


def test_oracle_port_clamp_fixture():
    """+-32767 clamp branch (lpcnet.c:265-269): golden from the reference with the large-excitation model."""
    import os
    from fixtures import make_feature_batch
    gold = np.load(os.path.join(H.GOLDEN, "clamp_A.npz"))["pcm"]
    assert (gold == 32767).sum() > 100 and (gold == -32767).sum() > 100
    L = H.oracle_lib()
    b = H.blob("int8_clamp")
    m = L.oracle_model_create(b, len(b), H.rcp_table().ctypes.data, H.LPC_GAMMA, H.codebooks().ctypes.data)
    f = make_feature_batch(range(4), 40)
    pcm = np.zeros((4, 40 * 160), np.int16)
    L.oracle_synthesize_batch(m, f.ctypes.data, 20, 4, 40, 4, pcm.ctypes.data)
    np.testing.assert_array_equal(pcm, gold)


VARIANT_TAGS = ["na256", "na128", "e2e", "delay0", "na256e2e"]


@pytest.mark.parametrize("tag", VARIANT_TAGS)
@pytest.mark.parametrize("build", ["A", "B"])
def test_oracle_port_model_variants_match_reference_golden(tag, build):
    """Other model shapes / switches (SURVEY 8f N1: GRU_A 256 and 128 units, END2END, FEATURES_DELAY 0): the CPU restatement
    against goldens of the reference compiled with that variant's generated nnet_data.h (tests/golden/variants.npz)."""
    import os
    from fixtures import make_feature_batch
    gold = np.load(os.path.join(H.GOLDEN, "variants.npz"))["%s_%s" % (tag, build)]
    f = make_feature_batch(range(2), 20)
    kind = "float" if build == "B" else "int8"
    np.testing.assert_array_equal(H.oracle_synth(f, kind, tag=tag), gold)
    if H.have_ref(build, tag):                                   # build container: the compiled reference itself
        np.testing.assert_array_equal(H.ref_synth(f, build, tag=tag), gold)


@pytest.mark.parametrize("build,tag", [("A", ""), ("B", ""), ("A", "na256e2e"), ("A", "delay0")])
def test_oracle_port_plc_entry_points_match_reference(build, tag):
    """lpcnet_synthesize_impl(preload), run_frame_network + lpcnet_synthesize_tail_impl, deferred/flush, lpcnet_reset_signal and
    state copies (what src/lpcnet_plc.c does around the hot path): the CPU restatement against the compiled reference."""
    import scenarios as S
    from fixtures import make_features
    T = 18
    script = S.plc_like_script(T)
    kind = "float" if build == "B" else "int8"
    for stream in (0, 3):
        f = make_features(stream, T)
        got = S.run_single("oracle", H.oracle_lib(), S.OracleState(kind, tag), f, stream, script)
        H.assert_ref_digests(got[None], "plc_%s%s_s%d" % (build, "_" + tag if tag else "", stream), "PCM of the call sequence, stream %d" % stream)
        assert np.abs(got).max() > 0


# ---------------------------------------------------------------- analysis side (SURVEY 8f N2)
def test_oracle_encoder_port_matches_reference_goldens():
    """oracle/lpcnet_enc_oracle.inc (CPU restatement of src/lpcnet_enc.c) against the vectors the compiled reference produced:
    per-frame features, packets and the unquantised 4-frame features, every float bit for bit."""
    G = np.load(os.path.join(H.GOLDEN, "enc_A.npz"))
    assert np.array_equal(H.oracle_features(G["pcm"]).view(np.uint32), G["features"].view(np.uint32))
    assert np.array_equal(H.oracle_encode(G["pcm"]), G["packets"])
    assert np.array_equal(H.oracle_encode(G["pcm"], features4=True).view(np.uint32), G["features4"].view(np.uint32))
    # the packets carry voiced and unvoiced frames and several modulation values (the fixture exercises both branches of :654-665)
    bits = np.zeros(G["packets"].shape[:2], np.uint64)
    for i in range(8):
        bits = (bits << np.uint64(8)) | G["packets"][:, :, i].astype(np.uint64)
    modulation = ((bits >> np.uint64(48)) & np.uint64(7)).astype(int)
    assert (modulation == 0).sum() >= 5 and len(set(modulation.ravel().tolist())) >= 3


def test_oracle_encoder_port_matches_compiled_reference_on_fresh_streams():
    from fixtures import make_pcm_batch
    pcm = make_pcm_batch(range(40, 52), 32)
    H.assert_ref_digests(pcm, "enc_pcm", "test inputs")
    H.assert_ref_digests(H.oracle_features(pcm), "enc_features", "features per stream")
    H.assert_ref_digests(H.oracle_encode(pcm), "enc_packets", "packets per stream")
    H.assert_ref_digests(H.oracle_encode(pcm, features4=True), "enc_features4", "unquantised features per stream")
