#!/usr/bin/env python3
"""What the UNTOUCHED reference (oracle/_ref, `make -C oracle ref`) returns for the stress models of oracle/gen_model.py
(make_stress_model: empty and short block lists, one column class, a compute warp at its tensor-memory budget, a model one density
step short of the shared-memory limit, int8 weights at the pair-constraint limit, GRU_A pre-activations next to the conversion-free rounding's range bound).

Run only where the reference has been compiled into oracle/_ref.

  stress.npz
     sha_<model>_<int8|float>      sha256 of the generated blob (pins the generator)
     features, pitch_features      H.digests of the synthesis inputs
     ref_<model>_<A|B>             per-stream digests of the reference's PCM, build A (int8 blob) / B (float blob), STRESS_STREAMS x STRESS_FRAMES
     ref_holes_pitch_<A|B>         the same on features whose pitch lies outside [33, 255] (the clamped embedding rows)
     plc_<model>_<A|B>_s<stream>   the PLC-style call sequence of scenarios.plc_like_script on the holes models
"""
import hashlib, os, sys
import numpy as np
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, ".."))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
sys.path.insert(0, os.path.join(HERE, "..", "..", "oracle"))
import helpers as H
import scenarios as S
import gen_model
from fixtures import make_feature_batch, make_features

STRESS_STREAMS = range(600, 603)
STRESS_FRAMES = 30
PLC_FRAMES = 18


def stress_features():
    return make_feature_batch(STRESS_STREAMS, STRESS_FRAMES)


def pitch_features():
    """stress_features with the pitch feature pushed below and above the embedding's range in alternate stretches of frames:
    period 50*f+100 of -60 .. 320 (clamped to 33 / 255 by run_frame_network)."""
    f = stress_features()
    t = np.arange(STRESS_FRAMES)
    f[:, (t // 4) % 3 == 1, 18] = -3.2
    f[:, (t // 4) % 3 == 2, 18] = 4.4
    f[1, 5:9, 18] = -1.36          # 31.9 -> 31
    f[2, 5:9, 18] = 3.11           # 255.6 -> 255
    return f


if __name__ == "__main__":
    out = {}
    for name in gen_model.STRESS_NAMES:
        for kind in ("int8", "float"):
            out["sha_%s_%s" % (name, kind)] = np.frombuffer(hashlib.sha256(H.stress_blob(name, kind)).digest(), np.uint8)
    f = stress_features()
    out["features"] = H.digests(f[None])
    for name in gen_model.STRESS_NAMES:
        for build in ("A", "B"):
            out["ref_%s_%s" % (name, build)] = H.stream_digests(H.ref_synth(f, build, stress=name))
    fp = pitch_features()
    out["pitch_features"] = H.digests(fp[None])
    for build in ("A", "B"):
        out["ref_holes_pitch_%s" % build] = H.stream_digests(H.ref_synth(fp, build, stress="holes"))
    script = S.plc_like_script(PLC_FRAMES)
    for name in ("holes", "holes128"):
        for build in ("A", "B"):
            for stream in (0, 3):
                pcm = S.run_single("ref", H.ref_lib(build, H.stress_tag(name)), S.RefState(build, stress=name), make_features(stream, PLC_FRAMES), stream, script)
                assert np.abs(pcm).max() > 0
                out["plc_%s_%s_s%d" % (name, build, stream)] = H.stream_digests(pcm[None])
    np.savez_compressed(os.path.join(HERE, "stress.npz"), **out)
    for key, val in out.items():
        print(key, val.shape, val.dtype)
