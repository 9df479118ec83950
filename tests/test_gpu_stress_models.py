"""GPU parity on the stress models (oracle/gen_model.py make_stress_model; -m gpu): empty and short block lists, lists of one column class,
a compute warp at its tensor-memory budget, a model one density step short of the shared-memory limit (fewer dual_fc rows in shared
memory), int8 weights at the pair-constraint limit, GRU_A pre-activations next to the range bound of the conversion-free rounding.
Against the compiled reference's digests (tests/golden/stress.npz) and, for wider / ragged / split batches, against the CPU restatement
that the CPU suite pins to them.

The launcher picks the kernel schedule from the live stream slots per CTA, min(32, ceil(n / SMs)) (batch_api.cu streams_per_cta_for):
on a B200 every batch below 149 streams gets one slot per CTA, i.e. the int8 half-A-only schedule and the float neuron-per-lane kernel.
So every test here sets the slots per CTA (LPCNET_B200_STREAMS_PER_CTA, and LPCNET_B200_TWO_HALVES) itself: spc <= 16 selects the
half-A-only int8 schedule unless two halves are forced, spc <= 4 the float neuron-per-lane kernel, anything else the two-half int8
schedule / the float lane==stream kernel."""
import os
import sys
import numpy as np
import pytest
import helpers as H
import gen_model
from fixtures import make_feature_batch

sys.path.insert(0, H.GOLDEN)
import make_golden_stress as MG      # noqa: E402

pytestmark = pytest.mark.gpu
NAMES = list(gen_model.STRESS_NAMES)


@pytest.fixture(scope="module")
def eng():
    import lpcnet_b200
    from lpcnet_b200 import build
    build.build()
    assert lpcnet_b200.device_count() > 0, "GPU test selected but no CUDA device is visible"
    return lpcnet_b200


@pytest.fixture(scope="module")
def gold():
    return dict(np.load(os.path.join(H.GOLDEN, "stress.npz")))


def _batch(eng, monkeypatch, n, name, kind, spc, two_halves=False):
    """a Batch of the stress model with `spc` live stream slots per CTA"""
    monkeypatch.setenv("LPCNET_B200_STREAMS_PER_CTA", str(spc))
    if two_halves:
        monkeypatch.setenv("LPCNET_B200_TWO_HALVES", "1")
    else:
        monkeypatch.delenv("LPCNET_B200_TWO_HALVES", raising=False)
    return eng.Batch(n, H.stress_blob(name, kind), config=H.model_config(H.stress_tag(name)))


# (kind, streams, slots per CTA, two halves forced): the schedule they select
SCHEDULES = {
    "int8-two-halves-full-ctas-ragged": ("int8", 70, 32, False),      # CTAs of 32, 32, 6
    "int8-two-halves-odd-ragged": ("int8", 70, 17, False),            # smallest two-half CTA, halves of 9 and 8, last CTA 2 streams
    "int8-two-halves-dead-slots": ("int8", 9, 5, True),               # two halves of 3 and 2 live slots, last CTA 4
    "int8-one-half-ragged": ("int8", 9, 5, False),                    # half-A-only schedule, CTAs of 5 and 4
    "float-lane-stream-ragged": ("float", 37, 32, False),             # lane==stream kernel (odd lists padded to even), CTAs of 32 and 5
    "float-neuron-per-lane-ragged": ("float", 7, 3, False),           # neuron-per-lane kernel, CTAs of 3, 3, 1
    "float-neuron-per-lane-one": ("float", 3, 1, False),              # one stream per CTA
}


def _first_diff(a, b):
    d = np.argwhere(a != b)
    return None if d.size == 0 else tuple(d[0])


@pytest.mark.parametrize("spc", [1, 32])
@pytest.mark.parametrize("kind,build", [("int8", "A"), ("float", "B")])
@pytest.mark.parametrize("name", NAMES)
def test_stress_model_matches_reference_golden(eng, gold, monkeypatch, name, kind, build, spc):
    """spc 1: int8 half-A-only schedule / float neuron-per-lane kernel; spc 32: two-half schedule / lane==stream kernel"""
    f = MG.stress_features()
    b = _batch(eng, monkeypatch, len(f), name, kind, spc)
    assert b.na == gen_model.stress_na(name)
    got = b.synthesize(f)
    b.close()
    bad = np.nonzero(H.stream_digests(got) != gold["ref_%s_%s" % (name, build)])[0]
    assert bad.size == 0, "%s %s: streams %s differ from the reference" % (name, kind, bad.tolist())


@pytest.mark.parametrize("schedule", list(SCHEDULES))
@pytest.mark.parametrize("name", NAMES)
def test_stress_model_batches_match_oracle(eng, monkeypatch, name, schedule):
    """every kernel schedule of the flavour (SCHEDULES) against the CPU restatement; the batch is synthesized in two calls, so the
    state carries across them"""
    kind, n, spc, two = SCHEDULES[schedule]
    T = 9
    f = make_feature_batch(range(700, 700 + n), T)
    b = _batch(eng, monkeypatch, n, name, kind, spc, two)
    got = np.concatenate([b.synthesize(f[:, :4]), b.synthesize(f[:, 4:])], axis=1)
    b.close()
    want = H.oracle_synth(f, kind, stress=name)
    assert _first_diff(got, want) is None, "first mismatch (stream, sample) = %s" % (_first_diff(got, want),)


@pytest.mark.parametrize("spc", [1, 32])
def test_cvt_fast_edge_conversion_unit_path_agrees(eng, gold, monkeypatch, spc):
    """cvt_fast_edge takes the conversion-free rounding with accumulators past 2^21; LPCNET_B200_EXACT_CVT forces the cvt path: same PCM"""
    f = MG.stress_features()
    want = gold["ref_cvt_fast_edge_A"]
    monkeypatch.setenv("LPCNET_B200_EXACT_CVT", "1")
    b = _batch(eng, monkeypatch, len(f), "cvt_fast_edge", "int8", spc)
    got = b.synthesize(f)
    b.close()
    np.testing.assert_array_equal(H.stream_digests(got), want)


@pytest.mark.parametrize("spc", [1, 32])
@pytest.mark.parametrize("kind,build", [("int8", "A"), ("float", "B")])
def test_clamped_pitch_matches_reference_golden(eng, gold, monkeypatch, kind, build, spc):
    """pitch periods below 33 and above 255: the embedding's clamp rows (frame_kernels.cu frame_assemble_kernel)"""
    f = MG.pitch_features()
    b = _batch(eng, monkeypatch, len(f), "holes", kind, spc)
    got = b.synthesize(f)
    b.close()
    np.testing.assert_array_equal(H.stream_digests(got), gold["ref_holes_pitch_%s" % build])


@pytest.mark.parametrize("kind,n,spc", [("int8", 40, 32), ("int8", 5, 3), ("float", 6, 2), ("float", 40, 32)])
@pytest.mark.parametrize("name", ["holes", "holes128"])
def test_plc_like_call_sequence_on_holes(eng, gold, monkeypatch, name, kind, n, spc):
    """scenarios.plc_like_script (preload, tails of 80, a forced frame, deferred + flush, reset_signal, snapshot / restore) on a batch
    == the CPU restatement per stream; streams 0 and 3 also == the reference's digests.  spc 32: two-half schedule / lane==stream
    kernel with a ragged CTA; spc 3 / 2: half-A-only schedule / neuron-per-lane kernel"""
    import scenarios as S
    T = MG.PLC_FRAMES
    streams = [0, 3] + list(range(100, 100 + n - 2))
    f = make_feature_batch(streams, T)
    script = S.plc_like_script(T)
    b = _batch(eng, monkeypatch, n, name, kind, spc)
    got = S.run_engine(b, f, streams, script)
    b.close()
    build = "B" if kind == "float" else "A"
    for i, s in enumerate(streams):
        if s in (0, 3):
            np.testing.assert_array_equal(H.stream_digests(got[i][None]), gold["plc_%s_%s_s%d" % (name, build, s)])
        want = S.run_single("oracle", H.oracle_lib(), S.OracleState(kind, stress=name), f[i], s, script)
        d = np.argwhere(got[i] != want)
        assert d.size == 0, "stream %d: first mismatch at sample %d" % (s, d[0][0])
