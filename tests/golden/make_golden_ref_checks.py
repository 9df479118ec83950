#!/usr/bin/env python3
"""What the UNTOUCHED reference (oracle/_ref, `make -C oracle ref`) returns for the inputs of the tests that used to call it
directly, stored so that those tests run from a plain checkout.  Large outputs are kept as digests (H.digests: the first
8 bytes of sha256 per stream, frame or packet, so that a failure still names where it differs); the digests of the
test inputs are stored too, so that a changed input generator is reported as such.

Run only where the reference has been compiled into oracle/_ref.

  ref_checks.npz
     kfft_factors, kfft_bitrev, kfft_twiddles, dct_table, ulaw2lin   the reference's tables      (test_tables_match_reference)
     act_inputs, act_tanh, act_sigmoid, act_lin2ulaw                   compute_activation, lin2ulaw (test_activations_and_ulaw_match_reference)
     fn_features, fn_gru_a, fn_gru_b, fn_lpc                           run_frame_network taps        (test_frame_network_matches_reference)
     fresh_features, fresh_A, fresh_B                                  lpcnet_synthesize, builds A/B (test_oracle_matches_reference_fresh_streams)
     dec_packets, dec_features                                         decode_packet                 (test_decode_packet_matches_reference)
     plc_<build>[_<tag>]_s<stream>                                     PLC-style call sequence       (test_oracle_port_plc_entry_points_match_reference)
     enc_pcm, enc_features, enc_packets, enc_features4                 analysis side, 12 streams     (test_oracle_encoder_port_matches_compiled_reference_on_fresh_streams)
     cfg_blob, cfg_pcm                                                 blob with the config record   (test_reference_loader_ignores_the_config_record)
     gpu_enc_pcm, gpu_enc_features, gpu_enc_packets                    analysis side, 96 streams     (test_gpu_encoder.py::test_fresh_inputs_against_the_compiled_reference)
"""
import ctypes, os, sys
import numpy as np
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, ".."))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
sys.path.insert(0, os.path.join(HERE, "..", "..", "oracle"))
import helpers as H
import scenarios as S
import lpcnet_b200
from fixtures import make_feature_batch, make_features, make_packets, make_pcm_batch


out = {}
R = H.ref_lib("A")

# tables (src/kiss_fft.c, src/freq.c, src/common.h)
class KissState(ctypes.Structure):   # kiss_fft_state (src/kiss_fft.h)
    _fields_ = [("nfft", ctypes.c_int), ("scale", ctypes.c_float), ("shift", ctypes.c_int),
                ("factors", ctypes.c_int16 * 16), ("bitrev", ctypes.POINTER(ctypes.c_int16)),
                ("twiddles", ctypes.POINTER(ctypes.c_float)), ("arch", ctypes.c_void_p)]
k = KissState.in_dll(R, "kfft")
assert k.nfft == 320
out["kfft_factors"] = np.array(k.factors[:8], np.int32)
out["kfft_bitrev"] = np.ctypeslib.as_array(k.bitrev, (320,)).astype(np.int32)
out["kfft_twiddles"] = np.ctypeslib.as_array(k.twiddles, (640,)).astype(np.float32)
out["dct_table"] = np.ctypeslib.as_array((ctypes.c_float * 324).in_dll(R, "dct_table")).astype(np.float32)
out["ulaw2lin"] = np.array([R.ref_ulaw2lin(float(i)) for i in range(256)], dtype=np.float32)

# activations and u-law on the inputs of test_activations_and_ulaw_match_reference
x, v = H.activation_test_inputs()
out["act_inputs"] = np.concatenate([H.digests(x[None]), H.digests(v[None])])
y = np.zeros_like(x)
R.ref_activation(y.ctypes.data, x.ctypes.data, x.size, 2)   # ACTIVATION_TANH
out["act_tanh"] = H.digests(y[None])
R.ref_activation(y.ctypes.data, x.ctypes.data, x.size, 1)   # ACTIVATION_SIGMOID
out["act_sigmoid"] = H.digests(y[None])
out["act_lin2ulaw"] = H.digests(np.array([R.ref_lin2ulaw(float(t)) for t in v], np.int32)[None])

# run_frame_network on stream 5, 12 frames
f = make_feature_batch([5], 12)[0]
b = H.blob("int8")
ga = np.zeros((12, 1152), np.float32); gb = np.zeros((12, 48), np.float32); lpc = np.zeros((12, 16), np.float32)
assert R.ref_frame_network(b, len(b), f.ctypes.data, 20, 12, ga.ctypes.data, gb.ctypes.data, lpc.ctypes.data) == 0
out.update(fn_features=H.digests(f[None]), fn_gru_a=H.digests(ga), fn_gru_b=H.digests(gb), fn_lpc=lpc)

# lpcnet_synthesize on streams the other goldens do not cover
f = make_feature_batch(range(100, 106), 80)
out.update(fresh_features=H.digests(f[None]), fresh_A=H.stream_digests(H.ref_synth(f, "A")), fresh_B=H.stream_digests(H.ref_synth(f, "B")))

# decode_packet, packet by packet with one VQ memory
pk = make_packets(77, 40)
vq = np.zeros(18, np.float32)
fr = np.zeros((40, 4, 36), np.float32)
for t in range(40):
    R.ref_decode_packet(fr[t].ctypes.data, vq.ctypes.data, pk[t].ctypes.data)
out.update(dec_packets=H.digests(pk[None]), dec_features=H.digests(fr))

# the PLC-style call sequence over the internal synthesis entry points
T = 18
script = S.plc_like_script(T)
for build, tag in (("A", ""), ("B", ""), ("A", "na256e2e"), ("A", "delay0")):
    for stream in (0, 3):
        pcm = S.run_single("ref", H.ref_lib(build, tag), S.RefState(build, tag), make_features(stream, T), stream, script)
        assert np.abs(pcm).max() > 0
        out["plc_%s%s_s%d" % (build, "_" + tag if tag else "", stream)] = H.stream_digests(pcm[None])

# analysis side on 12 streams x 32 frames
pcm = make_pcm_batch(range(40, 52), 32)
out.update(enc_pcm=H.digests(pcm), enc_features=H.digests(H.ref_features(pcm)), enc_packets=H.digests(H.ref_encode(pcm)), enc_features4=H.digests(H.ref_features4(pcm)))

# a blob carrying the lpcnet_b200_config record, loaded by the reference
lpcnet_b200.lib()
f = make_feature_batch(range(2), 5)
b2 = lpcnet_b200.write_blob(lpcnet_b200.parse_blob(H.blob("int8")), config=(0.9, 2, 0))
pcm = np.zeros((2, 5 * 160), np.int16)
assert R.ref_synth_batch(b2, len(b2), f.ctypes.data, f.shape[2], 5, 2, 2, pcm.ctypes.data) == 0
assert np.array_equal(pcm, H.ref_synth(f, "A"))
out.update(cfg_blob=H.digests(np.frombuffer(b2, np.uint8)[None]), cfg_pcm=H.stream_digests(pcm))

# analysis side on 96 streams x 60 frames (GPU test)
pcm = make_pcm_batch(range(100, 196), 60)
out.update(gpu_enc_pcm=H.digests(pcm), gpu_enc_features=H.digests(H.ref_features(pcm)), gpu_enc_packets=H.digests(H.ref_encode(pcm)))

np.savez_compressed(os.path.join(HERE, "ref_checks.npz"), **out)
for key, val in out.items():
    print(key, val.shape, val.dtype)
