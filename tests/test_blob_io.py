"""CPU tests (-m "not gpu") of the model-format I/O (SURVEY 8f N4): the DNNw blob writer / lister of the C-ABI
(csrc/blob_io.cu; reference src/write_lpcnet_weights.c:47-67, src/parse_lpcnet_weights.c:37-76) and the importer that turns
a model dumped by training_tf2/dump_lpcnet.py (nnet_data.c + nnet_data.h) into a blob with its switches embedded."""
import ctypes
import os
import sys
import numpy as np
import pytest
import helpers as H
import lpcnet_b200
from lpcnet_b200 import api

sys.path.insert(0, os.path.join(H.ROOT, "tools"))


@pytest.fixture(scope="module")
def L():
    from lpcnet_b200 import build
    build.build()
    return api.lib()


def test_writer_round_trip_is_byte_identical(L):
    """blob -> parse -> write reproduces the file gen_model wrote record for record (same padding, same headers)."""
    for kind in ("int8", "float"):
        b = H.blob(kind)
        recs = lpcnet_b200.parse_blob(b)
        assert len(recs) > 25 and recs[0][0] and all(len(d) > 0 for _, _, d in recs)
        assert lpcnet_b200.write_blob(recs) == b


def test_config_record_travels_in_the_blob_and_is_replaced_not_duplicated(L):
    b = H.blob("int8")
    recs = lpcnet_b200.parse_blob(b)
    assert lpcnet_b200.blob_config(b) is None
    b2 = lpcnet_b200.write_blob(recs, config=(0.9, 2, 0))
    assert len(b2) == len(b) + 128
    g, d, e = lpcnet_b200.blob_config(b2)
    assert abs(g - 0.9) < 1e-7 and (d, e) == (2, 0)
    b3 = lpcnet_b200.write_blob(lpcnet_b200.parse_blob(b2), config=(1.0, 0, 1))       # re-export with other switches
    assert [n for n, _, _ in lpcnet_b200.parse_blob(b3)].count("lpcnet_b200_config") == 1
    assert lpcnet_b200.blob_config(b3) == (1.0, 0, 1)
    # the engine's own image builder accepts the blob with the extra record
    out = np.zeros(256 * 1024, np.uint8); lay = np.zeros(24, np.uint32)
    L.lpcnet_b200_debug_image.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
    assert L.lpcnet_b200_debug_image(b2, len(b2), out.ctypes.data, out.size, lay.ctypes.data) > 0


def test_writer_and_lister_reject_bad_input(L):
    with pytest.raises(api.LPCNetB200Error, match="longer than 43"):
        lpcnet_b200.write_blob([("x" * 44, 0, b"\0" * 4)])
    with pytest.raises(api.LPCNetB200Error, match="empty"):
        lpcnet_b200.write_blob([("a", 0, b"")])
    with pytest.raises(api.LPCNetB200Error, match="unknown type"):
        lpcnet_b200.write_blob([("a", 7, b"\0" * 4)])
    with pytest.raises(api.LPCNetB200Error, match="config record"):
        lpcnet_b200.write_blob([("a", 0, b"\0" * 4)], config=(0.9, 5, 0))
    b = H.blob("int8")
    with pytest.raises(api.LPCNetB200Error):
        lpcnet_b200.parse_blob(b[:-10])                       # truncated payload
    bad = bytearray(b); bad[0:4] = b"XXXX"
    with pytest.raises(api.LPCNetB200Error, match="not a DNNw"):
        lpcnet_b200.parse_blob(bytes(bad))
    # size query / short buffer
    recs = (api.Array * 1)()
    nm, data = b"a", ctypes.create_string_buffer(b"\1" * 70, 70)
    recs[0].name = nm; recs[0].type = 0; recs[0].size = 70; recs[0].data = ctypes.addressof(data)
    assert L.lpcnet_b200_write_blob(recs, 1, None, None, 0) == 64 + 128
    small = (ctypes.c_ubyte * 100)()
    assert L.lpcnet_b200_write_blob(recs, 1, None, small, 100) < 0


def test_blob_files(L, tmp_path):
    recs = lpcnet_b200.parse_blob(H.blob("int8"))[:3]
    arr = (api.Array * 3)()
    keep = []
    for i, (n, t, d) in enumerate(recs):
        buf = ctypes.create_string_buffer(d, len(d)); nm = n.encode(); keep += [buf, nm]
        arr[i].name = nm; arr[i].type = t; arr[i].size = len(d); arr[i].data = ctypes.addressof(buf)
    path = str(tmp_path / "w.bin").encode()
    c = api.Config(0.9, 2, 0)
    assert L.lpcnet_b200_write_blob_file(path, arr, 3, ctypes.byref(c)) == 0
    sz = L.lpcnet_b200_read_file(path, None, 0)
    assert sz == os.path.getsize(path) > 0
    buf = (ctypes.c_ubyte * sz)()
    assert L.lpcnet_b200_read_file(path, buf, sz) == sz
    assert bytes(buf) == lpcnet_b200.write_blob(recs, config=(0.9, 2, 0))
    assert L.lpcnet_b200_read_file(b"/nonexistent/x", None, 0) < 0


def _print_vector(name, a, ctype):
    """training_tf2/dump_lpcnet.py:54-81 printVector, same text layout."""
    v = a.reshape(-1)
    s = ["#ifndef USE_WEIGHTS_FILE\n#define WEIGHTS_%s_DEFINED\n#define WEIGHTS_%s_TYPE WEIGHT_TYPE_%s\nstatic const %s %s[%d] = {\n   " % (name, name, ctype, ctype, name, len(v))]
    for i, x in enumerate(v):
        s.append("{}".format(x))
        if i != len(v) - 1:
            s.append(",")
            s.append("\n   " if i % 8 == 7 else " ")
    s.append("\n};\n#endif\n\n")
    return "".join(s)


def _dump_like_reference(common, only8, onlyf, small=200000):
    """nnet_data.c as dump_lpcnet.py writes it: float / int arrays plain, block-sparse weights as an #ifdef DOT_PROD pair."""
    by8 = {n: (t, a) for n, t, a in only8}
    byf = {n: (t, a) for n, t, a in onlyf}
    out = ["/*This file is automatically generated from a Keras model*/\n\n#ifdef HAVE_CONFIG_H\n#include \"config.h\"\n#endif\n\n#include \"nnet.h\"\n#include \"nnet_data.h\"\n\n"]
    order = [n for n, _, _ in common] + [n for n in by8]
    for n, t, a in common:
        out.append(_print_vector(n, a, {0: "float", 1: "int", 2: "qweight"}[t]))
    for n in by8:
        if n in byf and by8[n][0] == 2:
            out.append("#ifdef DOT_PROD\n" + _print_vector(n, by8[n][1], "qweight") + "#else /*DOT_PROD*/\n" + _print_vector(n, byf[n][1], "qweight") + "#endif /*DOT_PROD*/\n")
        else:   # arrays that only differ in value between the two builds (e.g. subias) are printed once by the reference; keep the int8 one
            out.append(_print_vector(n, by8[n][1], {0: "float", 1: "int", 2: "qweight"}[by8[n][0]]))
    out.append("#ifndef USE_WEIGHTS_FILE\nconst WeightArray lpcnet_arrays[] = {\n" + "".join('#ifdef WEIGHTS_%s_DEFINED\n  {"%s", WEIGHTS_%s_TYPE, sizeof(%s), %s},\n#endif\n' % (n, n, n, n, n) for n in order) + "  {NULL, 0, 0, NULL}\n};\n#endif\n")
    return "".join(out)


def test_importer_reads_a_dumped_model(L, tmp_path):
    """nnet_data.c/.h in the reference's dump format -> blob: every array bit-equal to the generator's own blob, the three
    nnet_data.h switches embedded; --float selects the DISABLE_DOT_PROD blocks."""
    import gen_model
    import import_nnet_data as imp
    common, only8, onlyf = gen_model.make_model(na=128)          # the smallest variant keeps the text file small
    (tmp_path / "nnet_data.c").write_text(_dump_like_reference(common, only8, onlyf))
    (tmp_path / "nnet_data.h").write_text("#ifndef RNN_DATA_H\n#define RNN_DATA_H\n#include \"nnet.h\"\n/* #define END2END */\n#define LPC_GAMMA 0.9f\n\n#define FEATURES_DELAY 1\n#endif\n")
    blob8, arrays8, cfg = imp.import_model(str(tmp_path / "nnet_data.c"))
    assert cfg == {"lpc_gamma": 0.9, "features_delay": 1, "end2end": 0}
    want8 = {n: (t, np.ascontiguousarray(a).tobytes()) for n, t, a in common + only8}
    got8 = {n: (t, d) for n, t, d in lpcnet_b200.parse_blob(blob8)}
    assert set(want8) | {"lpcnet_b200_config"} == set(got8)
    for n in want8:
        assert got8[n] == want8[n], n
    g, d, e = lpcnet_b200.blob_config(blob8)
    assert abs(g - 0.9) < 1e-7 and (d, e) == (1, 0)
    # float flavour: the #else branches
    blobf, _, _ = imp.import_model(str(tmp_path / "nnet_data.c"), is_float=True)
    gotf = {n: (t, d) for n, t, d in lpcnet_b200.parse_blob(blobf)}
    for n, t, a in onlyf:
        if t == 2:
            assert gotf[n] == (2, np.ascontiguousarray(a).tobytes()), n
    # END2END header
    (tmp_path / "nnet_data.h").write_text("#define END2END\n#define LPC_GAMMA 1.0f\n#define FEATURES_DELAY 0\n")
    assert imp.parse_header((tmp_path / "nnet_data.h").read_text()) == {"lpc_gamma": 1.0, "features_delay": 0, "end2end": 1}
    # the image builder accepts the imported int8 blob
    out = np.zeros(256 * 1024, np.uint8); lay = np.zeros(24, np.uint32)
    L.lpcnet_b200_debug_image.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
    assert L.lpcnet_b200_debug_image(blob8, len(blob8), out.ctypes.data, out.size, lay.ctypes.data) > 0 and int(lay[20]) == 128


def test_reference_loader_ignores_the_config_record(L):
    """A blob carrying `lpcnet_b200_config` still loads in the UNTOUCHED reference (lpcnet_load_model looks arrays up by name):
    the reference synthesised from exactly this blob what the plain model gives (the oracle, pinned to the reference)."""
    from fixtures import make_feature_batch
    f = make_feature_batch(range(2), 5)
    b2 = lpcnet_b200.write_blob(lpcnet_b200.parse_blob(H.blob("int8")), config=(0.9, 2, 0))
    H.assert_ref_digests(np.frombuffer(b2, np.uint8)[None], "cfg_blob", "blob handed to the reference")
    np.testing.assert_array_equal(H.ref_checks()["cfg_pcm"], H.stream_digests(H.oracle_synth(f, "int8")))


def test_shard_range_matches_the_python_sharding(L):
    from lpcnet_b200.sharding import shard_range
    for n, parts in ((4096, 8), (10, 3), (7, 7), (32768, 8), (5, 2)):
        cover = []
        for k in range(parts):
            lo, hi = lpcnet_b200.shard_range(n, k, parts)
            assert (lo, hi) == shard_range(n, k, parts)
            cover += list(range(lo, hi))
        assert cover == list(range(n))
    with pytest.raises(api.LPCNetB200Error):
        lpcnet_b200.shard_range(4, 3, 2)


def test_multi_create_refuses_without_devices(L):
    if L.lpcnet_b200_device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(api.LPCNetB200Error, match="no CUDA device"):
        lpcnet_b200.Multi(8, H.blob("int8"), [0, 1])


def test_analysis_tables_equal_the_reference_tables(L):
    """half_window / dct_table as the engine generates them (double libm on the host) == the literals of src/lpcnet_tables.c."""
    g = np.load(os.path.join(H.GOLDEN, "enc_A.npz"))
    hw = np.zeros(160, np.float32); dct = np.zeros(324, np.float32)
    L.lpcnet_b200_enc_tables(hw.ctypes.data, dct.ctypes.data)
    assert np.array_equal(hw.view(np.uint32), g["half_window"].view(np.uint32))
    assert np.array_equal(dct.view(np.uint32), g["dct_table"].view(np.uint32))
