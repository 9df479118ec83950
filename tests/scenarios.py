"""Call sequences over the reference's INTERNAL synthesis entry points (lpcnet_private.h:125-133: lpcnet_synthesize_impl with
`preload`, run_frame_network + lpcnet_synthesize_tail_impl, run_frame_network_deferred/_flush, lpcnet_reset_signal, state copies)
— what the reference's PLC does around the hot path (src/lpcnet_plc.c:188-503) — expressed once and run on three back ends:
the compiled reference (oracle/_ref, single stream), the CPU restatement (oracle port, single stream) and the CUDA engine
(a batch of streams).  TEST INFRASTRUCTURE."""
import ctypes
import numpy as np
import helpers as H


def plc_like_script(T):
    """(op, args) list over feature frames 0..T-1; every op consumes at most one frame index."""
    s = [("synth", t, 160, 0) for t in range(5)]                 # normal frames
    s += [("synth", 5, 160, 40)]                                 # lpcnet_synthesize_impl(..., preload=40): teacher-forced head
    s += [("net", 6), ("tail", 80, 0), ("tail", 80, 0)]           # run_frame_network + two half-frame tails (PLC uses N=80)
    s += [("net", 7), ("tail", 160, 160)]                         # a fully teacher-forced frame (state update only)
    s += [("defer", 8), ("defer", 9), ("flush",)]                 # queued conditioning frames, network run later
    s += [("synth", 10, 160, 0), ("reset_signal",), ("synth", 11, 160, 0)]
    s += [("save",), ("synth", 12, 160, 0), ("synth", 13, 160, 0), ("restore",), ("synth", 12, 160, 0), ("synth", 13, 160, 0)]
    s += [("synth", t, 160, 0) for t in range(14, T)]
    return s


def forced_signal(stream, n):
    """The 'known' signal a PLC would teacher-force with (deterministic, speech-like amplitude)."""
    rng = np.random.default_rng(5000 + int(stream))
    return (3000 * np.sin(np.arange(n) * 0.05 * (1 + stream % 3)) + rng.normal(0, 300, n)).astype(np.int16)


def run_single(backend, lib, st_new, feats, stream, script):
    """backend: 'ref' | 'oracle'.  feats [T][20].  Returns the concatenated PCM of all output-producing ops."""
    P = {"ref": dict(impl=lib.ref_synthesize_impl, net=lib.ref_run_frame_network, tail=lib.ref_synthesize_tail, defer=lib.ref_frame_network_deferred,
                     flush=lib.ref_frame_network_flush, rs=lib.ref_reset_signal) if backend == "ref" else None,
         "oracle": dict(impl=lib.oracle_synthesize_impl, net=lib.oracle_run_frame_network, tail=lib.oracle_synthesize_tail, defer=lib.oracle_frame_network_deferred,
                        flush=lib.oracle_frame_network_flush, rs=lib.oracle_reset_signal) if backend == "oracle" else None}[backend]
    st = st_new()
    saved = None
    out = []
    k = 0
    for op in script:
        if op[0] == "synth":
            _, t, N, pre = op
            buf = np.zeros(N, np.int16); buf[:pre] = forced_signal(stream, 4000)[k:k + pre]
            P["impl"](st, feats[t].ctypes.data, buf.ctypes.data, N, pre)
            out.append(buf); k += N
        elif op[0] == "net":
            P["net"](st, feats[op[1]].ctypes.data)
        elif op[0] == "tail":
            _, N, pre = op
            buf = np.zeros(N, np.int16); buf[:pre] = forced_signal(stream, 4000)[k:k + pre]
            P["tail"](st, buf.ctypes.data, N, pre)
            out.append(buf); k += N
        elif op[0] == "defer":
            P["defer"](st, feats[op[1]].ctypes.data)
        elif op[0] == "flush":
            P["flush"](st)
        elif op[0] == "reset_signal":
            P["rs"](st)
        elif op[0] == "save":
            saved = st_new.copy_of(st)
        elif op[0] == "restore":
            st_new.assign(st, saved)
    return np.concatenate(out)


class RefState:
    """state factory for run_single('ref', ...)"""
    def __init__(self, build="A", tag="", kind=None, stress=""):
        kind = kind or ("float" if build == "B" else "int8")
        tag = H.stress_tag(stress) if stress else tag
        self.L = H.ref_lib(build, tag); self.b = H.stress_blob(stress, kind) if stress else H.blob(kind, tag)
    def __call__(self):
        st = self.L.ref_state_create(self.b, len(self.b)); assert st; return st
    def copy_of(self, st):
        c = self(); self.L.ref_state_copy(c, st); return c
    def assign(self, dst, src):
        self.L.ref_state_copy(dst, src)


class OracleState:
    def __init__(self, kind="int8", tag="", stress=""):
        self.L = H.oracle_lib(); self.m = H.oracle_model(kind, H.stress_tag(stress), stress) if stress else H.oracle_model(kind, tag)
        self.size = 1 << 16
    def __call__(self):
        return self.L.oracle_state_create(self.m)
    def copy_of(self, st):
        c = self(); ctypes.memmove(c, st, self.L.oracle_state_size()); return c
    def assign(self, dst, src):
        ctypes.memmove(dst, src, self.L.oracle_state_size())


def run_engine(batch, feats, streams, script):
    """feats [n][T][20]; the same script on all streams of a lpcnet_b200.Batch.  Returns PCM [n][total]."""
    n = batch.n
    forced = np.stack([forced_signal(s, 4000) for s in streams])
    out, k, snap = [], 0, None
    for op in script:
        if op[0] == "synth":
            _, t, N, pre = op
            out.append(batch.synthesize(feats[:, t:t + 1], samples_per_frame=N, preload=pre, pcm_in=forced[:, k:k + max(pre, 1)])); k += N
        elif op[0] == "net":
            batch.run_frame_network(feats[:, op[1]:op[1] + 1])
        elif op[0] == "tail":
            _, N, pre = op
            out.append(batch.synthesize_tail(N, preload=pre, pcm_in=forced[:, k:k + max(pre, 1)])); k += N
        elif op[0] == "defer":
            batch.frame_network_deferred(feats[:, op[1]])
        elif op[0] == "flush":
            batch.frame_network_flush()
        elif op[0] == "reset_signal":
            batch.reset_signal()
        elif op[0] == "save":
            snap = batch.snapshot()
        elif op[0] == "restore":
            batch.restore(snap)
    if snap is not None:
        batch.free_snapshot(snap)
    return np.concatenate(out, axis=1)
