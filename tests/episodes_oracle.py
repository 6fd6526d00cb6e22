"""ctypes loader for tests/episodes_oracle.c: the CPU oracle's batched drivers with per-episode outputs.

TEST INFRASTRUCTURE ONLY.  Built like redraw_oracle.py: compiled on first use into a temporary directory keyed by the
sources' contents (the repository tree may be read-only), with the oracle's own flags (-ffp-contract=off)."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import redraw_oracle as ro
from oracle import oracle as o

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = [os.path.join(HERE, "episodes_oracle.c")] + ro.SOURCES

_lib = None


def lib():
    global _lib
    if _lib is None:
        digest = hashlib.sha1(b"".join(open(s, "rb").read() for s in SOURCES)).hexdigest()[:16]
        out_dir = os.path.join(tempfile.gettempdir(), f"mgym_episodes_oracle_{os.getuid()}_{digest}")
        path = os.path.join(out_dir, "libepisodes_oracle.so")
        if not os.path.exists(path):
            os.makedirs(out_dir, exist_ok=True)
            tmp = f"{path}.{os.getpid()}"
            subprocess.run([os.environ.get("CC", "gcc"), "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC",
                            "-std=gnu11", "-shared", "-o", tmp, SOURCES[0], "-lm", "-lpthread"], check=True,
                           capture_output=True)
            os.replace(tmp, path)
        L = C.CDLL(path)
        vp, u64 = C.c_void_p, C.c_uint64
        L.oracle_vec_step_e.argtypes = [C.c_int, C.POINTER(o.Config), u64, u64, u64] + [vp] * 6 + [u64] + [vp] * 4 + [
            C.POINTER(o.Stats), vp, vp, vp, vp, vp]
        L.oracle_vec_rollout_e.argtypes = [C.c_int, C.POINTER(o.Config), u64, u64, u64, C.c_uint32] + [vp] * 6 + [
            u64] + [vp] * 3 + [C.POINTER(C.c_uint64), C.POINTER(o.Stats), vp, vp, vp, vp, vp]
        _lib = L
    return _lib


_p = o._p
SENTINEL_RET = np.float32(-12345.5)
SENTINEL_LEN = np.uint32(0xDEADBEEF)


class VecState(ro.VecState):
    """redraw_oracle.VecState whose step_e / rollout_e also return the per-episode outputs, in buffers pre-filled with
    a sentinel (entries of envs that did not finish keep it)."""

    def step_e(self, actions, want_return=True, want_length=True):
        od = o.OBS_DIM[self.kind]
        obs = np.zeros((od, self.ld), dtype=np.float32)
        rew = np.zeros(self.ld, dtype=np.float32)
        flg = np.zeros(self.ld, dtype=np.uint8)
        ret = np.full(self.ld, SENTINEL_RET, dtype=np.float32) if want_return else None
        length = np.full(self.ld, SENTINEL_LEN, dtype=np.uint32) if want_length else None
        a = np.ascontiguousarray(actions, dtype=np.float32 if o.CONTINUOUS[self.kind] else np.uint8)
        pp, pl = self._pool()
        lib().oracle_vec_step_e(self.kind, C.byref(self.cfg), self.n, self.ld, self.t, _p(self.state), _p(self.steps),
                                _p(self.sbt), _p(self.ep_return), _p(a), pp, pl, _p(obs), _p(rew), _p(flg), None,
                                C.byref(self.stats), _p(self.params), _p(self.low), _p(self.high), _p(ret),
                                _p(length))
        self.t += 1
        return obs, rew, flg, ret, length

    def rollout_e(self, K, actions=None, want_return=True, want_length=True):
        od = o.OBS_DIM[self.kind]
        obs = np.zeros((K, od, self.ld), dtype=np.float32)
        rew = np.zeros((K, self.ld), dtype=np.float32)
        flg = np.zeros((K, self.ld), dtype=np.uint8)
        ret = np.full((K, self.ld), SENTINEL_RET, dtype=np.float32) if want_return else None
        length = np.full((K, self.ld), SENTINEL_LEN, dtype=np.uint32) if want_length else None
        a = None
        if actions is not None:
            a = np.ascontiguousarray(actions, dtype=np.float32 if o.CONTINUOUS[self.kind] else np.uint8)
        dc = C.c_uint64(0)
        pp, pl = self._pool()
        lib().oracle_vec_rollout_e(self.kind, C.byref(self.cfg), self.n, self.ld, self.t, K, _p(self.state),
                                   _p(self.steps), _p(self.sbt), _p(self.ep_return), _p(a), pp, pl, _p(obs), _p(rew),
                                   _p(flg), C.byref(dc), C.byref(self.stats), _p(self.params), _p(self.low),
                                   _p(self.high), _p(ret), _p(length))
        self.t += K
        return obs, rew, flg, dc.value, ret, length
