"""ctypes binding of the low-level engine C-ABI (include/msckf_b200.h) -- used by bench.py to time the
kernel launch with inputs already resident in HBM, and by tests that exercise the C-ABI directly."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import lib_path

MARGINALIZE, TRIANGULATE, RESIDUALIZE = 0, 1, 2


class Config(C.Structure):
    _fields_ = [("dtype", C.c_int), ("device", C.c_int), ("max_clones", C.c_int), ("max_tracks", C.c_int), ("max_obs", C.c_int)]


class Tracks(C.Structure):
    _fields_ = [("n_tracks", C.c_int), ("obs_offset", C.POINTER(C.c_int)), ("obs", C.c_void_p),
                ("clone_index", C.POINTER(C.c_int)), ("p_f_G", C.c_void_p)]


class Report(C.Structure):
    _fields_ = [("cm_ok", C.POINTER(C.c_int)), ("tri_ok", C.POINTER(C.c_int)), ("valid", C.POINTER(C.c_int)),
                ("accepted", C.POINTER(C.c_int)), ("gamma", C.c_void_p), ("p_f_G", C.c_void_p), ("m", C.c_int), ("rank", C.c_int)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(str(lib_path()))
        _lib.msckf_b200_last_error.restype = C.c_char_p
        _lib.msckf_b200_launch_count.restype = C.c_longlong
        _lib.msckf_b200_stream.restype = C.c_void_p
    return _lib


def check(rc, what):
    if rc < 0:
        raise RuntimeError(f"{what} failed rc={rc}: {(lib().msckf_b200_last_error() or b'').decode()}")
    return rc


class TrackBatch:
    """host-side flat SoA batch (keeps the numpy arrays alive)."""

    def __init__(self, obs_offset, obs, clone_index, dtype, p_f_G=None):
        self.dtype = np.dtype(dtype)
        self.off = np.ascontiguousarray(obs_offset, dtype=np.int32)
        self.obs = np.ascontiguousarray(obs, dtype=self.dtype)
        self.idx = np.ascontiguousarray(clone_index, dtype=np.int32)
        self.pfg = None if p_f_G is None else np.ascontiguousarray(p_f_G, dtype=self.dtype)
        self.c = Tracks(len(self.off) - 1, self.off.ctypes.data_as(C.POINTER(C.c_int)), self.obs.ctypes.data_as(C.c_void_p),
                        self.idx.ctypes.data_as(C.POINTER(C.c_int)), None if self.pfg is None else self.pfg.ctypes.data_as(C.c_void_p))

    @property
    def n_tracks(self):
        return len(self.off) - 1

    def h2d_bytes(self):
        return self.off.nbytes + self.obs.nbytes + self.idx.nbytes + (0 if self.pfg is None else self.pfg.nbytes)


class Batch:
    """msckf_b200_batch: n engines whose updates run as ONE device batch (filter index in blockIdx.z, one CUDA graph, one
    packed copy each way).  While it lives the engines share its stream."""

    def __init__(self, engines):
        self.engines = list(engines)
        n = len(self.engines)
        hs = (C.c_void_p * n)(*[e.h for e in self.engines])
        self.h = C.c_void_p()
        check(lib().msckf_b200_batch_create(hs, C.c_int(n), C.byref(self.h)), "msckf_b200_batch_create")
        lib().msckf_b200_batch_launch_count.restype = C.c_longlong

    def close(self):
        if self.h:
            lib().msckf_b200_batch_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _tracks(self, batches):
        assert len(batches) == len(self.engines)
        return (Tracks * len(batches))(*[b.c for b in batches])

    def stage(self, mode, batches, threads=1):
        self._keep = batches
        check(lib().msckf_b200_batch_stage(self.h, C.c_int(mode), self._tracks(batches), C.c_int(threads)), "msckf_b200_batch_stage")

    def launch(self):
        check(lib().msckf_b200_batch_launch(self.h), "msckf_b200_batch_launch")

    def launch_timed(self):
        ms = C.c_float()
        check(lib().msckf_b200_batch_launch_timed(self.h, C.byref(ms)), "msckf_b200_batch_launch_timed")
        return ms.value

    def fetch(self, batches=None, full=False):
        """per-engine reports: m, rank, accepted; `full` adds every other per-track field of msckf_b200_report"""
        batches = batches or self._keep
        n = len(self.engines)
        reps = (Report * n)()
        bufs = []
        for i, b in enumerate(batches):
            nt, dt = max(b.n_tracks, 1), self.engines[i].dtype
            buf = {"accepted": np.zeros(nt, dtype=np.int32)}
            if full:
                buf.update(cm_ok=np.zeros(nt, dtype=np.int32), tri_ok=np.zeros(nt, dtype=np.int32), valid=np.zeros(nt, dtype=np.int32),
                           gamma=np.zeros(nt, dtype=dt), p_f_G=np.zeros((nt, 3), dtype=dt))
            for k, a in buf.items():
                setattr(reps[i], k, a.ctypes.data_as(C.POINTER(C.c_int) if a.dtype == np.int32 else C.c_void_p))
            bufs.append(buf)
        check(lib().msckf_b200_batch_fetch(self.h, reps), "msckf_b200_batch_fetch")
        return [{"m": reps[i].m, "rank": reps[i].rank, **{k: a[:batches[i].n_tracks] for k, a in bufs[i].items()}} for i in range(n)]

    def update(self, mode, batches, threads=1):
        """host buffers in, reports out: packing + one H2D + kernels + one D2H (the batch's end-to-end call)."""
        n = len(self.engines)
        reps = (Report * n)()
        accs = []
        for i, b in enumerate(batches):
            acc = np.zeros(max(b.n_tracks, 1), dtype=np.int32)
            reps[i].accepted = acc.ctypes.data_as(C.POINTER(C.c_int))
            accs.append(acc)
        check(lib().msckf_b200_batch_update(self.h, C.c_int(mode), self._tracks(batches), reps, C.c_int(threads)), "msckf_b200_batch_update")
        return [{"m": reps[i].m, "rank": reps[i].rank, "accepted": accs[i][:batches[i].n_tracks]} for i in range(n)]

    def kernel_times(self):
        ms = (C.c_float * 32)()
        names = (C.c_char_p * 32)()
        n = check(lib().msckf_b200_batch_kernel_times(self.h, ms, names, C.c_int(32)), "msckf_b200_batch_kernel_times")
        return [(names[i].decode(), ms[i]) for i in range(n)]

    def launch_count(self):
        return int(lib().msckf_b200_batch_launch_count(self.h))


def update_batch(engines, mode, batches, threads=8):
    """msckf_b200_update_batch: one update per engine (independent filters), host work on `threads` threads.
    Returns the per-engine (m, rank, accepted) reports."""
    n = len(engines)
    assert n == len(batches)
    hs = (C.c_void_p * n)(*[e.h for e in engines])
    trs = (Tracks * n)(*[b.c for b in batches])
    reps = (Report * n)()
    accs = []
    for i, b in enumerate(batches):
        acc = np.zeros(max(b.n_tracks, 1), dtype=np.int32)
        reps[i].accepted = acc.ctypes.data_as(C.POINTER(C.c_int))
        accs.append(acc)
    check(lib().msckf_b200_update_batch(hs, C.c_int(n), C.c_int(mode), trs, reps, C.c_int(int(threads))), "msckf_b200_update_batch")
    return [{"m": reps[i].m, "rank": reps[i].rank, "accepted": accs[i][:batches[i].n_tracks]} for i in range(n)]


class Engine:
    """owning wrapper of a msckf_b200_engine*; `borrowed` wraps a handle owned by somebody else."""

    def __init__(self, dtype=np.float32, device=0, max_clones=40, max_tracks=512, max_obs=512 * 30, borrowed=None):
        self.dtype = np.dtype(dtype)
        self.owned = borrowed is None
        if borrowed is not None:
            self.h = C.c_void_p(borrowed)
        else:
            cfg = Config(0 if self.dtype == np.float32 else 1, device, max_clones, max_tracks, max_obs)
            self.h = C.c_void_p()
            check(lib().msckf_b200_create(C.byref(cfg), C.byref(self.h)), "msckf_b200_create")

    def close(self):
        if self.owned and self.h:
            lib().msckf_b200_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def copy_state_from(self, other):
        check(lib().msckf_b200_copy_state(self.h, other.h), "msckf_b200_copy_state")

    def stage(self, mode, batch):
        check(lib().msckf_b200_stage(self.h, C.c_int(mode), C.byref(batch.c)), "msckf_b200_stage")

    def launch(self):
        check(lib().msckf_b200_launch(self.h), "msckf_b200_launch")

    def launch_timed(self):
        ms = C.c_float()
        check(lib().msckf_b200_launch_timed(self.h, C.byref(ms)), "msckf_b200_launch_timed")
        return ms.value

    def fetch(self, n_tracks=0):
        rep = Report()
        acc = np.zeros(max(n_tracks, 1), dtype=np.int32)
        rep.accepted = acc.ctypes.data_as(C.POINTER(C.c_int))
        check(lib().msckf_b200_fetch(self.h, C.byref(rep)), "msckf_b200_fetch")
        return {"m": rep.m, "rank": rep.rank, "accepted": acc[:n_tracks]}

    def synchronize(self):
        check(lib().msckf_b200_synchronize(self.h), "msckf_b200_synchronize")

    def propagate_n(self, readings):
        r = np.ascontiguousarray(readings, dtype=self.dtype).reshape(-1, 7)
        check(lib().msckf_b200_propagate_n(self.h, r.ctypes.data_as(C.c_void_p), C.c_int(len(r))), "msckf_b200_propagate_n")

    def augment(self):
        check(lib().msckf_b200_augment(self.h), "msckf_b200_augment")

    def prune(self, keep):
        k = np.ascontiguousarray(keep, dtype=np.int32)
        check(lib().msckf_b200_prune(self.h, k.ctypes.data_as(C.POINTER(C.c_int)), C.c_int(len(k))), "msckf_b200_prune")

    def update(self, mode, batch):
        rep = Report()
        acc = np.zeros(max(batch.n_tracks, 1), dtype=np.int32)
        rep.accepted = acc.ctypes.data_as(C.POINTER(C.c_int))
        check(lib().msckf_b200_update(self.h, C.c_int(mode), C.byref(batch.c), C.byref(rep)), "msckf_b200_update")
        return {"m": rep.m, "rank": rep.rank, "accepted": acc[:batch.n_tracks]}

    def rank_pivots(self):
        buf = (C.c_double * 2048)()
        n = check(lib().msckf_b200_rank_pivots(self.h, buf, C.c_int(2048)), "msckf_b200_rank_pivots")
        return np.array(buf[:n])

    def set_option(self, key, value):
        check(lib().msckf_b200_set_option(self.h, C.c_int(key), C.c_double(value)), "msckf_b200_set_option")

    def kernel_times(self):
        ms = (C.c_float * 32)()
        names = (C.c_char_p * 32)()
        n = check(lib().msckf_b200_kernel_times(self.h, ms, names, C.c_int(32)), "msckf_b200_kernel_times")
        return [(names[i].decode(), ms[i]) for i in range(n)]

    def launch_count(self):
        return int(lib().msckf_b200_launch_count(self.h))

    def num_clones(self):
        return lib().msckf_b200_num_clones(self.h)

    def covariance(self):
        n = 15 + 6 * self.num_clones()
        out = np.zeros((n, n), dtype=self.dtype)
        check(lib().msckf_b200_get_covariance(self.h, out.ctypes.data_as(C.c_void_p)), "msckf_b200_get_covariance")
        return out

    def state(self):
        """(IMU state: the 29 scalars of msckf_b200_get_state, clone poses [M, 7]: p, q)"""
        imu = np.zeros(29, dtype=self.dtype)
        poses = np.zeros((self.num_clones(), 7), dtype=self.dtype)
        check(lib().msckf_b200_get_state(self.h, imu.ctypes.data_as(C.c_void_p), poses.ctypes.data_as(C.c_void_p)), "msckf_b200_get_state")
        return imu, poses

    def set_covariance(self, P):
        P = np.ascontiguousarray(P, dtype=self.dtype)
        check(lib().msckf_b200_set_covariance(self.h, P.ctypes.data_as(C.c_void_p)), "msckf_b200_set_covariance")

    def poison_covariance(self):
        """test hook: a NaN in the IMU block (exercises MSCKF_B200_ERR_NUMERIC)"""
        P = self.covariance()
        P[0, 0] = np.nan
        self.set_covariance(P)

    def delta_x(self):
        out = np.zeros(15 + 6 * 128)
        n = check(lib().msckf_b200_last_delta_x(self.h, out.ctypes.data_as(C.POINTER(C.c_double)), C.c_int(len(out))), "last_delta_x")
        return out[:n].copy()
