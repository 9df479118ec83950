"""Shared test plumbing: builds/loads the checkers (oracle port, compiled reference) through ctypes.

The oracle and the compiled reference are CHECKERS: they are only ever used from tests/, smoke() and the
bench's cpu_baseline leg — never by the product library.
"""
import ctypes
import functools
import os
import subprocess
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE = os.path.join(ROOT, "oracle")
GEN = os.path.join(ORACLE, "_gen")
GOLDEN = os.path.join(ROOT, "tests", "golden")
LPC_GAMMA = 0.9

c_p = ctypes.c_void_p


@functools.lru_cache(None)
def gen_dir(tag=""):
    """Deterministically (re)generate the synthetic model files.  tag: "" (the default 384/16 model) or one of
    gen_model.VARIANTS (other GRU_A sizes, END2END, FEATURES_DELAY) -> oracle/_gen_<tag>."""
    import gen_model
    d = GEN + ("_" + tag if tag else "")
    need = ["model_int8.bin", "model_float.bin", "codebooks.bin"] + ([] if tag else ["model_int8_clamp.bin"])
    if not all(os.path.exists(os.path.join(d, n)) for n in need):
        gen_model.generate(d, c_sources=os.path.isdir("/root/reference/src"), **(gen_model.VARIANTS[tag] if tag else {}))
    return d


@functools.lru_cache(None)
def blob(kind="int8", tag=""):
    """kind: int8 | float | int8_clamp (default model only)."""
    return open(os.path.join(gen_dir(tag), "model_%s.bin" % kind), "rb").read()


def model_config(tag=""):
    """(lpc_gamma, features_delay, end2end) the reference bakes into nnet_data.h for this variant."""
    import gen_model
    v = gen_model.VARIANTS[tag] if tag else {}
    g = v.get("gamma")
    d = v.get("delay")
    return (LPC_GAMMA if g is None else g, gen_model.FEATURES_DELAY if d is None else d, bool(v.get("e2e", False)))


@functools.lru_cache(None)
def codebooks():
    return np.fromfile(os.path.join(gen_dir(), "codebooks.bin"), dtype=np.float32)


@functools.lru_cache(None)
def rcp_table():
    return np.fromfile(os.path.join(GOLDEN, "rcpps_table.bin"), dtype="<u4")


@functools.lru_cache(None)
def oracle_lib():
    so = os.path.join(ORACLE, "_build", "liblpcnet_oracle.so")
    src = os.path.join(ORACLE, "lpcnet_oracle.c")
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src), os.path.getmtime(os.path.join(ORACLE, "lpcnet_enc_oracle.inc"))):
        subprocess.check_call(["make", "-C", ORACLE, "port"], stdout=subprocess.DEVNULL)
    L = ctypes.CDLL(so)
    L.oracle_model_create.restype = c_p
    L.oracle_model_create.argtypes = [ctypes.c_char_p, ctypes.c_int, c_p, ctypes.c_float, c_p]
    L.oracle_model_create_ex.restype = c_p
    L.oracle_model_create_ex.argtypes = [ctypes.c_char_p, ctypes.c_int, c_p, ctypes.c_float, ctypes.c_int, ctypes.c_int, c_p]
    L.oracle_synthesize_impl.argtypes = [c_p, c_p, c_p, ctypes.c_int, ctypes.c_int]
    L.oracle_run_frame_network.argtypes = [c_p, c_p]
    L.oracle_synthesize_tail.argtypes = [c_p, c_p, ctypes.c_int, ctypes.c_int]
    L.oracle_frame_network_deferred.argtypes = [c_p, c_p]
    L.oracle_frame_network_flush.argtypes = [c_p]
    L.oracle_reset_signal.argtypes = [c_p]
    L.oracle_export_state.argtypes = [c_p, c_p]
    L.oracle_model_na.argtypes = [c_p]
    L.oracle_state_size.argtypes = []
    L.oracle_state_create.restype = c_p
    L.oracle_state_create.argtypes = [c_p]
    L.oracle_state_destroy.argtypes = [c_p]
    L.oracle_reset.argtypes = [c_p]
    L.oracle_synthesize.argtypes = [c_p, c_p, c_p, ctypes.c_int]
    L.oracle_synthesize_trace.argtypes = [c_p, c_p, c_p, ctypes.c_int, c_p]
    L.oracle_decode.argtypes = [c_p, c_p, c_p]
    L.oracle_decode_packet.argtypes = [c_p, c_p, c_p]
    L.oracle_frame_network.argtypes = [c_p, c_p, c_p, c_p, c_p]
    L.oracle_get_tables.argtypes = [c_p] * 6
    L.oracle_get_state.argtypes = [c_p] * 6
    L.oracle_tanh.restype = ctypes.c_float
    L.oracle_tanh.argtypes = [c_p, ctypes.c_float]
    L.oracle_sigmoid.restype = ctypes.c_float
    L.oracle_sigmoid.argtypes = [c_p, ctypes.c_float]
    L.oracle_lin2ulaw.argtypes = [ctypes.c_float]
    L.oracle_synthesize_batch.restype = ctypes.c_double
    L.oracle_synthesize_batch.argtypes = [c_p, c_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_p]
    L.oracle_decode_batch.restype = ctypes.c_double
    L.oracle_decode_batch.argtypes = [c_p, c_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_p]
    L.oracle_enc_create.restype = c_p
    L.oracle_enc_create.argtypes = [c_p]
    L.oracle_enc_destroy.argtypes = [c_p]
    L.oracle_enc_single_frame_features.argtypes = [c_p, c_p, c_p]
    L.oracle_enc_encode.argtypes = [c_p, c_p, c_p]
    L.oracle_enc_compute_features.argtypes = [c_p, c_p, c_p]
    return L


@functools.lru_cache(None)
def oracle_model(kind="int8", tag=""):
    """CPU-restatement model for a blob flavour (int8 / float / int8_clamp) of a model variant (tag, gen_model.VARIANTS)."""
    L = oracle_lib()
    b = blob(kind, tag)
    gamma, delay, e2e = model_config(tag)
    m = L.oracle_model_create_ex(b, len(b), rcp_table().ctypes.data, gamma, delay, int(e2e), codebooks().ctypes.data)
    assert m, "oracle failed to parse the blob"
    return m


def oracle_synth(features, kind="int8", nthreads=8, tag=""):
    """features [n][T][20] float32 -> pcm [n][T*160] int16 via the CPU restatement."""
    L = oracle_lib()
    f = np.ascontiguousarray(features, dtype=np.float32)
    n, T, stride = f.shape
    pcm = np.zeros((n, T * 160), dtype=np.int16)
    L.oracle_synthesize_batch(oracle_model(kind, tag), f.ctypes.data, stride, n, T, nthreads, pcm.ctypes.data)
    return pcm


def oracle_decode(packets, kind="int8", nthreads=8):
    """packets [n][P][8] uint8 -> pcm [n][P*640] int16."""
    L = oracle_lib()
    p = np.ascontiguousarray(packets, dtype=np.uint8)
    n, P, _ = p.shape
    pcm = np.zeros((n, P * 640), dtype=np.int16)
    L.oracle_decode_batch(oracle_model(kind), p.ctypes.data, n, P, nthreads, pcm.ctypes.data)
    return pcm


def have_ref(build="A", tag=""):
    return os.path.exists(os.path.join(ORACLE, "_ref", "liblpcnet_ref_%s%s.so" % (build, "_" + tag if tag else "")))


@functools.lru_cache(None)
def ref_lib(build="A", tag=""):
    """The UNTOUCHED reference compiled by oracle/Makefile (`make ref`); tag selects a model variant's build."""
    L = ctypes.CDLL(os.path.join(ORACLE, "_ref", "liblpcnet_ref_%s%s.so" % (build, "_" + tag if tag else "")))
    L.ref_synth_batch.argtypes = [ctypes.c_char_p, ctypes.c_int, c_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_p]
    L.ref_decode_batch.argtypes = [ctypes.c_char_p, ctypes.c_int, c_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_p]
    L.ref_time_streams.restype = ctypes.c_double
    L.ref_time_streams.argtypes = [ctypes.c_char_p, ctypes.c_int, c_p, ctypes.c_int, c_p, ctypes.c_int, ctypes.c_int, c_p]
    L.ref_synth_stream.argtypes = [ctypes.c_char_p, ctypes.c_int, c_p, ctypes.c_int, ctypes.c_int, c_p]
    L.ref_decode_stream.argtypes = [ctypes.c_char_p, ctypes.c_int, c_p, ctypes.c_int, c_p]
    L.ref_decode_packet.argtypes = [c_p, c_p, c_p]
    L.ref_frame_network.argtypes = [ctypes.c_char_p, ctypes.c_int, c_p, ctypes.c_int, ctypes.c_int, c_p, c_p, c_p]
    L.ref_rcp.restype = ctypes.c_float
    L.ref_rcp.argtypes = [ctypes.c_float]
    L.ref_ulaw2lin.restype = ctypes.c_float
    L.ref_ulaw2lin.argtypes = [ctypes.c_float]
    L.ref_lin2ulaw.argtypes = [ctypes.c_float]
    L.ref_activation.argtypes = [c_p, c_p, ctypes.c_int, ctypes.c_int]
    L.ref_state_create.restype = c_p
    L.ref_state_create.argtypes = [ctypes.c_char_p, ctypes.c_int]
    for fn in ("ref_features_stream", "ref_features_stream_float", "ref_encode_stream", "ref_features4_stream"):
        if hasattr(L, fn):
            getattr(L, fn).argtypes = [c_p, ctypes.c_int, c_p]
    if hasattr(L, "ref_encode_then_features"):
        L.ref_encode_then_features.argtypes = [c_p, ctypes.c_int, c_p, ctypes.c_int, c_p]
        L.ref_enc_tables.argtypes = [c_p, c_p]
    for fn, at in (("ref_state_destroy", [c_p]), ("ref_state_reset", [c_p]), ("ref_state_copy", [c_p, c_p]),
                   ("ref_synthesize_impl", [c_p, c_p, c_p, ctypes.c_int, ctypes.c_int]), ("ref_run_frame_network", [c_p, c_p]),
                   ("ref_synthesize_tail", [c_p, c_p, ctypes.c_int, ctypes.c_int]), ("ref_frame_network_deferred", [c_p, c_p]),
                   ("ref_frame_network_flush", [c_p]), ("ref_reset_signal", [c_p])):
        getattr(L, fn).argtypes = at
        getattr(L, fn).restype = None
    return L


def ref_synth(features, build="A", tag="", kind=None, nthreads=None):
    """features [n][T][stride] -> pcm [n][T*160] through the compiled reference (fresh lpcnet_create() per stream)."""
    L = ref_lib(build, tag)
    b = blob(kind or ("float" if build in ("B", "TB") else "int8"), tag)
    f = np.ascontiguousarray(features, dtype=np.float32)
    n, T, stride = f.shape
    pcm = np.zeros((n, T * 160), dtype=np.int16)
    assert L.ref_synth_batch(b, len(b), f.ctypes.data, stride, T, n, nthreads or min(n, os.cpu_count() or 1), pcm.ctypes.data) == 0
    return pcm


def ref_decode(packets, build="A", tag="", nthreads=None):
    L = ref_lib(build, tag)
    b = blob("float" if build in ("B", "TB") else "int8", tag)
    p = np.ascontiguousarray(packets, dtype=np.uint8)
    n, P, _ = p.shape
    pcm = np.zeros((n, P * 640), dtype=np.int16)
    assert L.ref_decode_batch(b, len(b), p.ctypes.data, P, n, nthreads or min(n, os.cpu_count() or 1), pcm.ctypes.data) == 0
    return pcm


def stream_digests(pcm):
    """First 8 bytes of sha256 of every stream's PCM as uint64 [n] (a failing comparison names the stream)."""
    import hashlib
    return np.array([int.from_bytes(hashlib.sha256(np.ascontiguousarray(r).tobytes()).digest()[:8], "little") for r in pcm], dtype=np.uint64)


def digests(a):
    """stream_digests of every a[i], whatever its shape: one digest per stream, frame or packet."""
    return stream_digests(np.reshape(a, (len(a), -1)))


@functools.lru_cache(None)
def ref_checks():
    """What the compiled reference returned for the inputs of the tests that compare with it (tests/golden/make_golden_ref_checks.py)."""
    return dict(np.load(os.path.join(GOLDEN, "ref_checks.npz")))


def assert_ref_digests(got, key, what):
    """digests(got) against the stored digests of the reference's output; a failure names the rows that differ."""
    want = ref_checks()[key]
    bad = np.nonzero(digests(got) != want)[0]
    assert bad.size == 0, "%s: %d of %d rows differ from the reference, first: %s" % (what, bad.size, len(want), bad[:16].tolist())


def activation_test_inputs():
    """(x, v): float32 inputs of the tanh / sigmoid and of the lin2ulaw comparison."""
    rng = np.random.default_rng(3)
    x = np.concatenate([rng.normal(0, 3, 20000), rng.uniform(-12, 12, 20000), [0.0, -0.0, 1e-8, 50.0, -50.0]]).astype(np.float32)
    x = x[: x.size // 8 * 8]
    v = np.concatenate([rng.normal(0, 3000, 20000), rng.uniform(-40000, 40000, 5000), [0.0, 32767.0, -32768.0]]).astype(np.float32)
    return x, v


# ---- the analysis side (SURVEY 8f N2): the compiled reference's encoder entry points, one fresh state per stream ----
def ref_features(pcm, build="A"):
    """pcm [n][T*160] int16 (or float32) -> features [n][T][36] via lpcnet_compute_single_frame_features(_float)."""
    L = ref_lib(build)
    p = np.ascontiguousarray(pcm)
    n, T = p.shape[0], p.shape[1] // 160
    out = np.zeros((n, T, 36), np.float32)
    for s in range(n):
        row = np.ascontiguousarray(p[s])
        (L.ref_features_stream_float if p.dtype == np.float32 else L.ref_features_stream)(row.ctypes.data, T, out[s].ctypes.data)
    return out


def ref_encode(pcm, build="A"):
    """pcm [n][P*640] int16 -> packets [n][P][8] via lpcnet_encode."""
    L = ref_lib(build)
    p = np.ascontiguousarray(pcm, dtype=np.int16)
    n, P = p.shape[0], p.shape[1] // 640
    out = np.zeros((n, P, 8), np.uint8)
    for s in range(n):
        L.ref_encode_stream(p[s].ctypes.data, P, out[s].ctypes.data)
    return out


def ref_features4(pcm, build="A"):
    """pcm [n][P*640] int16 -> features [n][P*4][36] via lpcnet_compute_features."""
    L = ref_lib(build)
    p = np.ascontiguousarray(pcm, dtype=np.int16)
    n, P = p.shape[0], p.shape[1] // 640
    out = np.zeros((n, P * 4, 36), np.float32)
    for s in range(n):
        L.ref_features4_stream(p[s].ctypes.data, P, out[s].ctypes.data)
    return out


# ---- CPU restatement of the analysis side (oracle/lpcnet_enc_oracle.inc), one fresh state per stream ----
def oracle_features(pcm):
    L = oracle_lib()
    p = np.ascontiguousarray(pcm, dtype=np.int16)
    n, T = p.shape[0], p.shape[1] // 160
    out = np.zeros((n, T, 36), np.float32)
    for s in range(n):
        e = L.oracle_enc_create(None)
        for t in range(T):
            L.oracle_enc_single_frame_features(e, p[s, t * 160:].ctypes.data, out[s, t].ctypes.data)
        L.oracle_enc_destroy(e)
    return out


def oracle_encode(pcm, features4=False):
    """pcm [n][P*640] -> packets [n][P][8] (lpcnet_encode), or with features4 the unquantised features [n][P*4][36] (lpcnet_compute_features)."""
    L = oracle_lib()
    p = np.ascontiguousarray(pcm, dtype=np.int16)
    n, P = p.shape[0], p.shape[1] // 640
    cb = codebooks()
    out = np.zeros((n, P * 4, 36), np.float32) if features4 else np.zeros((n, P, 8), np.uint8)
    for s in range(n):
        e = L.oracle_enc_create(cb.ctypes.data)
        for k in range(P):
            if features4:
                L.oracle_enc_compute_features(e, p[s, k * 640:].ctypes.data, out[s, 4 * k].ctypes.data)
            else:
                L.oracle_enc_encode(e, p[s, k * 640:].ctypes.data, out[s, k].ctypes.data)
        L.oracle_enc_destroy(e)
    return out
