"""ctypes loader for tests/redraw_oracle.c: the CPU oracle's batched drivers with per-episode parameter redraws.

TEST INFRASTRUCTURE ONLY.  Built like params_oracle.py: compiled on first use into a temporary directory keyed by the
sources' contents (the repository tree may be read-only), with the oracle's own flags (-ffp-contract=off)."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import params_oracle as po
from oracle import oracle as o

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = [os.path.join(HERE, "redraw_oracle.c"), os.path.join(HERE, "params_oracle.c"),
           os.path.join(HERE, "..", "oracle", "mgym_oracle.c"), os.path.join(HERE, "..", "oracle", "mgym_oracle.h")]
NUM_PARAMS = po.NUM_PARAMS

_lib = None


def lib():
    global _lib
    if _lib is None:
        digest = hashlib.sha1(b"".join(open(s, "rb").read() for s in SOURCES)).hexdigest()[:16]
        out_dir = os.path.join(tempfile.gettempdir(), f"mgym_redraw_oracle_{os.getuid()}_{digest}")
        path = os.path.join(out_dir, "libredraw_oracle.so")
        if not os.path.exists(path):
            os.makedirs(out_dir, exist_ok=True)
            tmp = f"{path}.{os.getpid()}"
            subprocess.run([os.environ.get("CC", "gcc"), "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC",
                            "-std=gnu11", "-shared", "-o", tmp, SOURCES[0], "-lm", "-lpthread"], check=True,
                           capture_output=True)
            os.replace(tmp, path)
        L = C.CDLL(path)
        vp, u64 = C.c_void_p, C.c_uint64
        L.oracle_vec_step_p.argtypes = [C.c_int, C.POINTER(o.Config), u64, u64, u64] + [vp] * 6 + [u64] + [vp] * 4 + [
            C.POINTER(o.Stats), vp]
        L.oracle_vec_rollout_p.argtypes = [C.c_int, C.POINTER(o.Config), u64, u64, u64, C.c_uint32] + [vp] * 6 + [
            u64] + [vp] * 3 + [C.POINTER(C.c_uint64), C.POINTER(o.Stats), vp]
        L.oracle_vec_step_r.argtypes = [C.c_int, C.POINTER(o.Config), u64, u64, u64] + [vp] * 6 + [u64] + [vp] * 4 + [
            C.POINTER(o.Stats), vp, vp, vp]
        L.oracle_vec_rollout_r.argtypes = [C.c_int, C.POINTER(o.Config), u64, u64, u64, C.c_uint32] + [vp] * 6 + [
            u64] + [vp] * 3 + [C.POINTER(C.c_uint64), C.POINTER(o.Stats), vp, vp, vp]
        L.oracle_reset_r.argtypes = [C.c_int, C.POINTER(o.Config), u64, u64, u64] + [vp] * 6 + [u64] + [vp] * 4
        _lib = L
    return _lib


_p = o._p


class VecState(po.VecState):
    """params_oracle.VecState whose step / rollout / reset also redraw the rows at every reset once
    set_param_redraw(low, high) has been called (rows not set before start from `defaults`)."""

    def __init__(self, kind, n, ld=None, **cfg):
        super().__init__(kind, n, ld, **cfg)
        self.low = self.high = None

    def set_param_redraw(self, low, high, defaults=None):
        if low is None:
            self.low = self.high = None
            return
        if self.params is None:
            self.params = np.repeat(np.asarray(defaults, dtype=np.float32)[:, None], self.ld, axis=1)
        self.low = np.ascontiguousarray(low, dtype=np.float32)
        self.high = np.ascontiguousarray(high, dtype=np.float32)

    def step(self, actions, want_final_obs=False):
        od = o.OBS_DIM[self.kind]
        obs = np.zeros((od, self.ld), dtype=np.float32)
        rew = np.zeros(self.ld, dtype=np.float32)
        flg = np.zeros(self.ld, dtype=np.uint8)
        fin = np.zeros((od, self.ld), dtype=np.float32) if want_final_obs else None
        a = np.ascontiguousarray(actions, dtype=np.float32 if o.CONTINUOUS[self.kind] else np.uint8)
        pp, pl = self._pool()
        lib().oracle_vec_step_r(self.kind, C.byref(self.cfg), self.n, self.ld, self.t, _p(self.state), _p(self.steps),
                                _p(self.sbt), _p(self.ep_return), _p(a), pp, pl, _p(obs), _p(rew), _p(flg), _p(fin),
                                C.byref(self.stats), _p(self.params), _p(self.low), _p(self.high))
        self.t += 1
        return (obs, rew, flg, fin) if want_final_obs else (obs, rew, flg)

    def rollout(self, K, actions=None):
        od = o.OBS_DIM[self.kind]
        obs = np.zeros((K, od, self.ld), dtype=np.float32)
        rew = np.zeros((K, self.ld), dtype=np.float32)
        flg = np.zeros((K, self.ld), dtype=np.uint8)
        a = None
        if actions is not None:
            a = np.ascontiguousarray(actions, dtype=np.float32 if o.CONTINUOUS[self.kind] else np.uint8)
        dc = C.c_uint64(0)
        pp, pl = self._pool()
        lib().oracle_vec_rollout_r(self.kind, C.byref(self.cfg), self.n, self.ld, self.t, K, _p(self.state),
                                   _p(self.steps), _p(self.sbt), _p(self.ep_return), _p(a), pp, pl, _p(obs), _p(rew),
                                   _p(flg), C.byref(dc), C.byref(self.stats), _p(self.params), _p(self.low),
                                   _p(self.high))
        self.t += K
        return obs, rew, flg, dc.value

    def reset(self, mask=None):
        obs = np.zeros((o.OBS_DIM[self.kind], self.ld), dtype=np.float32)
        pp, pl = self._pool()
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        lib().oracle_reset_r(self.kind, C.byref(self.cfg), self.n, self.ld, self.n_resets, _p(m), _p(self.state),
                             _p(self.steps), _p(self.sbt), _p(self.ep_return), pp, pl, _p(obs), _p(self.params),
                             _p(self.low), _p(self.high))
        self.n_resets += 1
        return obs
