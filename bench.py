#!/usr/bin/env python
"""bench.py -- MSCKF updates/sec on the B200 engine (and the reference arm / CPU baseline beside it).

A "step" is one pass of the hot path over one batch of synthetic input.  The unit of work is BASELINE.json configs[1]:
ONE marginalize() (msckf.h:336-449 -> measurementUpdate :1325-1423) on 300 feature tracks x 30 camera clones, float32,
produced through the public MSCKF<_S> surface (SURVEY.md 8d) so that the update processes exactly 300 x 30.
Per-rank work of a step = FILTERS_PER_GPU (8) such updates on 8 independent filters, run as ONE device batch
(msckf_b200_batch_*: one launch per kernel, filter index in blockIdx.z, one CUDA graph, one packed copy each way) -- the
shape of BASELINE configs[3] (64 independent sequences, 8 per GPU, on 8 GPUs), used at every N so that the driver's
1/2/4/8-GPU curve is that configuration and N=1 is consistent with it.  One filter alone (configs[1] literally: latency of
a single update()) is the `single` sub-record.

  value        whole-job updates/s: N GPUs x 8 filters / device time of a step (CUDA events on the batch's stream around the
               kernels, inputs resident in HBM, states restored and L2 flushed between steps, max over ranks)
  e2e          the same step through the C-ABI call msckf_b200_batch_update with HOST buffers: packing into pinned memory,
               one H2D copy, all kernels, one D2H copy of the reports, report unpacking (host wall clock)
  single       one filter: device-timed update, end to end through the drop-in class (marginalize() + getImuState()),
               per-kernel table
  stress       BASELINE configs[4]: 2000 x 60 float64, one filter: ms per update, per-kernel table, flop figures
  stream       BASELINE configs[2] stand-in (E-sim, SURVEY 8d): 200 frames of propagate + update through the class, float32:
               frames/s, updates/s, trajectory RMS vs the oracle on the same inputs, the oracle's own frames/s beside it
  parity       engine vs oracle on the config-B workload in THIS run: dx relative differences (fp32 direct, fp64 clean,
               fp64 faithful) and accept/reject flips
  roofline     dominant kernel of the step: SURVEY 8d algorithmic bytes of the updates one launch processes / that
               kernel's mean device time (CUDA events between the kernels), against the measured HBM peak
  cpu_baseline the oracle (CPU restatement of the reference's Eigen path) timed on this box's host, 1 core

Every rank runs the same per-GPU work (weak scaling; independent filters shard with no collective on the data path, NCCL is
only used for the barrier / max-over-ranks).  `--impl reference` times the CPU oracle instead.
"""
import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

N_FEAT, N_CLONES = 300, 30
DTYPE = np.float32
FILTERS_PER_GPU = 8


def algorithmic_bytes(nf, nc, b):
    """SURVEY.md 8d: 2*b*m*6L (H_o non-zero columns written + read) + 2*b*m (r_o) + 3*b*n^2 (P) + inputs."""
    L = M = nc
    m = nf * (2 * L - 3)
    n = 15 + 6 * M
    return 2 * b * m * 6 * L + 2 * b * m + 3 * b * n * n + nf * L * 2 * b + M * 7 * b


def algorithmic_flops(nf, nc):
    """SURVEY.md 8d reference-path flops (projection + gating + QR + R_n + n^3 tail)."""
    L = M = nc
    rho, n, c = 2 * L - 3, 15 + 6 * M, 6 * M
    m = nf * rho
    return (nf * 2 * rho * (2 * L) * (6 * L) + nf * (2 * rho * (6 * L) ** 2 + 2 * rho ** 2 * (6 * L) + rho ** 3 / 3)
            + (2 * (m - 15) * c ** 2 - 2 / 3 * c ** 3) + 2 * (nf * L) * n ** 2 + 12 * n ** 3)


def executed_flops(nf, nc):
    """flops of the path as built (DESIGN.md 4): per-feature structured gate + reflectors, Gram pair, n^3 tail."""
    L = M = nc
    rho, n, c = 2 * L - 3, 15 + 6 * M, 6 * M
    per_feat = 2 * (L * (L + 1) / 2) * (2 * 36 * 2 + 4 * 12) + 2 * (2 * L) ** 2 * 3 * 2 + rho ** 3 / 3 + 40 * 2 * L
    gram = 2 * 2 * (3 * nf) * c * c / 2 * 2  # Z^T Z and Z^T Yq + Yq^T Z, upper tiles
    tail = 2 * n ** 3 * 2 + 2 * n ** 3 / 3 + n ** 3 + n ** 3  # TP, S'', two factorisations, substitution, P - W^T W
    return nf * per_feat + gram + tail


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons sampled through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                     "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
                time.sleep(0.001)
        except Exception as e:  # pragma: no cover
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def result(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def physical_gpu_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


def ready_filter(dtype, seq, device, nf=N_FEAT, nc=N_CLONES):
    """a filter driven through the public API up to (not including) the marginalize() that processes nf x nc."""
    from msckf_mono_b200 import engine_filter, synth
    wl = synth.make_window_workload(n_features=nf, n_clones=nc, seq=seq)
    f = engine_filter(dtype, device=device, max_clones=nc + 8, max_tracks=max(512, nf + 48), max_obs=max(512, nf + 48) * nc)
    synth.drive(f, wl, marginalize_last=False)
    return f


def oracle_lib():
    lib = ROOT / "oracle" / "libmsckf_oracle.so"
    if not lib.exists():
        raise RuntimeError("oracle/libmsckf_oracle.so missing (run __graft_entry__.build())")
    return lib


def cpu_oracle_updates(seconds_target, threads, dtype):
    """time the CPU oracle's marginalize() on the same workload; returns (updates/s, n_updates, wall seconds)."""
    from concurrent.futures import ThreadPoolExecutor
    from msckf_mono_b200 import synth
    from msckf_mono_b200.cview import CFilter
    lib = oracle_lib()

    def prepare(seq):
        o = CFilter(lib, "msckf_oracle_", dtype)
        synth.drive(o, synth.make_window_workload(n_features=N_FEAT, n_clones=N_CLONES, seq=seq), marginalize_last=False)
        return o

    def one(o):
        t0 = time.perf_counter()
        o.marginalize()  # ctypes releases the GIL: threads run truly in parallel
        return time.perf_counter() - t0

    warm = prepare(0)
    t_one = one(warm)
    rounds = max(1, int(round(seconds_target / max(t_one, 1e-3))))
    done, wall = 0, 0.0
    with ThreadPoolExecutor(max_workers=threads) as ex:
        for r in range(rounds):
            filts = [prepare(1 + r * threads + i) for i in range(threads)]  # untimed: builds the pre-update state
            t0 = time.perf_counter()
            list(ex.map(one, filts))
            wall += time.perf_counter() - t0
            done += threads
    return done / wall, done, wall


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU path (here: its restatement, the reference cannot be built on
    this image) on the host cores.  The filter is single-threaded like the reference; independent filters use
    all cores (one update per core per step)."""
    if rank != 0:
        return
    # the oracle's working set (three 17100 x 195 matrices per filter) makes it memory-bandwidth bound: throughput
    # saturates around 16 concurrent filters (measured on the 128-core GPU box: 8.1/s with 128 threads vs 2.0/s with 1),
    # and a step must stay bounded, so a step = one update on each of min(cores, 16) threads
    cores = min(os.cpu_count() or 1, 16)
    from concurrent.futures import ThreadPoolExecutor
    from msckf_mono_b200 import synth
    from msckf_mono_b200.cview import CFilter
    lib = oracle_lib()

    def prepare(seq):
        o = CFilter(lib, "msckf_oracle_", DTYPE)
        synth.drive(o, synth.make_window_workload(n_features=N_FEAT, n_clones=N_CLONES, seq=seq), marginalize_last=False)
        return o

    def one(o):
        o.marginalize()

    total, wall = 0, 0.0
    with ThreadPoolExecutor(max_workers=cores) as ex:
        for step in range(args.warmup + args.steps):
            filts = [prepare(1000 + step * cores + i) for i in range(cores)]
            t0 = time.perf_counter()
            list(ex.map(one, filts))
            dt = time.perf_counter() - t0
            if step >= args.warmup:
                total += cores
                wall += dt
    val = total / wall
    line = {"impl": "reference", "metric": "msckf_updates_per_sec", "value": val, "unit": "updates/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{N_FEAT} features x {N_CLONES} clones, float32, one marginalize() per update; "
                                   f"a step = {cores} independent updates, one per host core", "n_features": N_FEAT, "n_clones": N_CLONES},
            "cpu_baseline": {"value": val, "unit": "updates/s", "cores": cores, "kind": "port",
                             "sample": f"{total} updates of the {N_FEAT}x{N_CLONES} fp32 workload, {cores} concurrent single-threaded oracle filters"},
            "e2e": {"value": val, "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "reference (Eigen 3 + Boost + ROS) is not buildable on this image; this is oracle/ (its line-by-line CPU restatement, thin-Q form; "
                    "hand-written loops at -ffp-contract=off: Eigen itself would be a few times faster, the reference as written -- dense m x m Q -- far slower)"}
    print(json.dumps(line))


DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def dump_outputs(out_dir, reps, engines, suffix=""):
    """What the last timed step handed its caller, per filter of this rank: the batch update's report and the corrected filter
    state, stacked over the filters as DIR/<name><suffix>.npy (integers as float64, the filter's own precision otherwise).
    The inputs are seeded, so two builds run with the same arguments can be compared file by file.  Filters past the
    64 MB budget are left out (the first ones are kept, the same ones in every run)."""
    fields = {k: [r[k] for r in reps] for k in ("m", "rank", "cm_ok", "tri_ok", "valid", "accepted", "gamma", "p_f_G")}
    states = [e.state() for e in engines]
    fields["imu_state"] = [s[0] for s in states]
    fields["clone_poses"] = [s[1] for s in states]
    fields["covariance"] = [e.covariance() for e in engines]
    fields["delta_x"] = [e.delta_x() for e in engines]
    per_filter = sum(8 * np.asarray(v[0]).size for v in fields.values())
    keep = max(1, min(len(engines), DUMP_LIMIT_BYTES // per_filter))
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for name, vals in fields.items():
        a = np.stack([np.asarray(v) for v in vals[:keep]])
        a = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
        np.save(out / f"{name}{suffix}.npy", a)


def kernel_table(obj, step_fn, reps=5):
    """per-kernel device times (CUDA events between the kernels: engine option 1, plain launches on one stream)"""
    per = {}
    for _ in range(reps):
        step_fn()
        for name, ms in obj.kernel_times():
            per.setdefault(name, []).append(ms)
    return {k: float(np.mean(v[1:])) for k, v in per.items()}


def single_filter_record(local_rank, flush_l2, steps, warm):
    """configs[1] literally: one filter, one update(): device time, end to end through the class, per-kernel table"""
    from msckf_mono_b200 import capi
    tmpl = ready_filter(DTYPE, seq=100, device=local_rank)
    off, obs, idx = tmpl.packQueued()
    batch = capi.TrackBatch(off, obs, idx, DTYPE)
    tmpl_eng = capi.Engine(DTYPE, borrowed=tmpl.engineHandle())
    work = capi.Engine(DTYPE, device=local_rank, max_clones=N_CLONES + 8, max_tracks=512, max_obs=512 * N_CLONES)

    def device_step():
        work.copy_state_from(tmpl_eng)
        work.stage(capi.MARGINALIZE, batch)
        work.synchronize()
        flush_l2()
        ms = work.launch_timed()
        rep = work.fetch(batch.n_tracks)
        assert rep["m"] == N_FEAT * (2 * N_CLONES - 3), rep
        return ms

    for _ in range(warm):
        device_step()
    dev = [device_step() for _ in range(steps)]
    # end to end through the drop-in class: marginalize() + getImuState(), host buffers
    filts = [ready_filter(DTYPE, seq=200 + i, device=local_rank) for i in range(steps + warm)]
    e2e, parts = [], []
    for i, f in enumerate(filts):
        flush_l2()
        t0 = time.perf_counter()
        f.marginalizeLaunch()      # marginalize() = launch (pack into the pinned block + one H2D copy + graph launch) ...
        t1 = time.perf_counter()
        f.marginalizeCollect()     # ... + collect (wait for the kernels, one D2H report copy, host bookkeeping)
        t2 = time.perf_counter()
        st = f.getImuState()       # D2H of the corrected state (the step's result)
        t3 = time.perf_counter()
        if i >= warm:
            e2e.append(t3 - t0)
            parts.append((t1 - t0, t2 - t1, t3 - t2))
    assert np.isfinite(st["p_I_G"]).all()
    work.set_option(1, 1.0)
    kern = kernel_table(work, device_step)
    work.set_option(1, 0.0)
    pl, pc_, ps = (1e6 * float(np.mean([p[j] for p in parts])) for j in range(3))
    dev_ms, e2e_ms = float(np.mean(dev)), 1e3 * float(np.mean(e2e))
    return {"workload": f"{N_FEAT} x {N_CLONES} float32, ONE filter, one update() per step (BASELINE configs[1] literally)",
            "ms_per_update_device": dev_ms, "updates_per_s_device": 1e3 / dev_ms,
            "ms_per_update_e2e": e2e_ms, "updates_per_s_e2e": 1e3 / e2e_ms, "e2e_over_device": e2e_ms / dev_ms,
            "e2e_path": "msckf_mono::MSCKF<float>::marginalize() + getImuState() via the C view, host wall clock",
            "e2e_breakdown_us": {"launch (pack into pinned + H2D + graph launch)": pl, "collect (kernels + D2H + bookkeeping)": pc_, "getImuState": ps},
            "kernel_us": {k: round(1e3 * v, 1) for k, v in kern.items()}}, kern


def stress_record(local_rank, flush_l2):
    """BASELINE configs[4]: 2000 x 60 float64, one filter"""
    from msckf_mono_b200 import capi
    nf, nc = 2000, 60
    tmpl = ready_filter(np.float64, seq=30, device=local_rank, nf=nf, nc=nc)
    off, obs, idx = tmpl.packQueued()
    batch = capi.TrackBatch(off, obs, idx, np.float64)
    tmpl_eng = capi.Engine(np.float64, borrowed=tmpl.engineHandle())
    work = capi.Engine(np.float64, device=local_rank, max_clones=nc + 8, max_tracks=nf + 48, max_obs=(nf + 48) * nc)

    def device_step():
        work.copy_state_from(tmpl_eng)
        work.stage(capi.MARGINALIZE, batch)
        work.synchronize()
        flush_l2()
        ms = work.launch_timed()
        rep = work.fetch(batch.n_tracks)
        assert rep["m"] == nf * (2 * nc - 3) and rep["accepted"].all(), rep["m"]
        return ms, rep

    for _ in range(3):
        device_step()
    dev = [device_step()[0] for _ in range(6)]
    rep = device_step()[1]
    work.set_option(1, 1.0)
    kern = kernel_table(work, lambda: device_step())
    work.set_option(1, 0.0)
    ms = float(np.mean(dev))
    dom = max(kern, key=kern.get)
    fl_ref, fl_exec = algorithmic_flops(nf, nc), executed_flops(nf, nc)
    return {"workload": f"{nf} x {nc} float64, one filter, one update() per step (BASELINE configs[4]); m = {nf * (2 * nc - 3)}, n = {15 + 6 * nc}",
            "ms_per_update_device": ms, "updates_per_s_device": 1e3 / ms, "accepted": int(rep["accepted"].sum()), "rank": int(rep["rank"]),
            "kernel_us": {k: round(1e3 * v, 1) for k, v in kern.items()}, "dominant_kernel": dom,
            "reference_path_gflop": fl_ref / 1e9, "executed_gflop_estimate": fl_exec / 1e9,
            "reference_path_tflops_equivalent": fl_ref / (ms * 1e-3) / 1e12, "executed_tflops_fp64": fl_exec / (ms * 1e-3) / 1e12,
            "algorithmic_bytes": algorithmic_bytes(nf, nc, 8), "algorithmic_gbs": algorithmic_bytes(nf, nc, 8) / (ms * 1e-3) / 1e9,
            "parity": "tests/test_engine_gpu.py::test_config_s_full_2000x60_fp64_vs_oracle_fixture (zero flips; numbers in tests/golden/parity_measured.json)"}


def stream_record(local_rank):
    """BASELINE configs[2] stand-in: E-sim stream, float32, propagate + update per frame through the class"""
    from msckf_mono_b200 import engine_filter, synth
    from msckf_mono_b200.cview import CFilter
    wl = synth.make_stream_workload(n_frames=200, seq=8, max_features=60, max_track_length=20, max_cam_states=20)
    wl["noise"] = synth.euroc_noise(tuned=True)
    n_imu = sum(len(fr["imu"]) for fr in wl["frames"])
    best = None
    pg = []
    for rep in range(3):  # first pass warms kernels / graphs
        g = engine_filter(DTYPE, device=local_rank)
        pg = []
        t0 = time.perf_counter()
        synth.drive(g, wl, on_frame=lambda k, f: pg.append(f.getImuState()["p_I_G"].copy()))
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
        n_upd = g.counters()["n_updates"]
    o = CFilter(oracle_lib(), "msckf_oracle_", DTYPE)
    po = []
    t0 = time.perf_counter()
    synth.drive(o, wl, on_frame=lambda k, f: po.append(f.getImuState()["p_I_G"].copy()))
    dt_o = time.perf_counter() - t0
    d = np.array(pg) - np.array(po)
    return {"workload": "E-sim (stands in for EuRoC MH_03, not on this box): 200 frames at 20 Hz, 10 IMU readings per frame, <= 60 features, "
                        "window 20 clones, float32, through MSCKF<float> (propagate x10, augmentState, update, addFeatures, marginalize, "
                        "pruneEmptyStates, getImuState per frame)",
            "frames_per_s": 200 / best, "imu_readings_per_s": n_imu / best, "updates_per_s": n_upd / best, "n_updates": int(n_upd),
            "oracle_frames_per_s": 200 / dt_o, "speedup_vs_oracle_1core": dt_o / best,
            "traj_rms_vs_oracle_m": float(np.sqrt((d ** 2).sum(axis=1).mean())), "traj_max_vs_oracle_m": float(np.abs(d).max())}


def parity_record(local_rank):
    """engine vs oracle on the config-B workload, computed in this run (test infrastructure used as the checker)"""
    from tests import parity_cases as pc
    out = {}
    for key, name in (("f32", "f32_direct_300x30"), ("f64_clean", "f64_clean_300x30"), ("f64_faithful", "f64_faithful_300x30")):
        r = pc.run_case(name)  # asserts zero accept / reject flips and bit-exact bookkeeping inside
        out[f"dx_rel_{key}"] = r["dx"]
        out[f"P_rel_{key}"] = r["P"]
    out["flips"] = 0
    out["workload"] = "300 x 30, seq 0; oracle = oracle/libmsckf_oracle.so (fp32 vs the fp32 engine directly; fp64 exact-subspace and reference-literal modes)"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--filters", type=int, default=FILTERS_PER_GPU, help="independent filters per GPU in the device batch")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--skip-extras", action="store_true", help="profiling aid: only the device-timed steps (use under ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3

    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from msckf_mono_b200 import capi, shard

    K, W, F = args.steps, args.warmup, args.filters
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")  # > 126 MB L2

    def flush_l2():
        flush.add_(1.0)
        torch.cuda.synchronize()

    def barrier():
        shard.barrier()
        torch.cuda.synchronize()

    # ---------------------------------------------------------------- setup (untimed): F filters per GPU, one device batch
    tmpl, tmpl_eng, batches, work = [], [], [], []
    for i in range(F):
        f = ready_filter(DTYPE, seq=(rank * F + i) % 24, device=local_rank)
        off, obs, idx = f.packQueued()
        batches.append(capi.TrackBatch(off, obs, idx, DTYPE))
        tmpl.append(f)
        tmpl_eng.append(capi.Engine(DTYPE, borrowed=f.engineHandle()))
        work.append(capi.Engine(DTYPE, device=local_rank, max_clones=N_CLONES + 8, max_tracks=512, max_obs=512 * N_CLONES))
    grp = capi.Batch(work)
    host_threads = max(1, min(4, (os.cpu_count() or 1)))

    def restore():
        for w, t in zip(work, tmpl_eng):
            w.copy_state_from(t)

    def device_step(full_report=False):
        restore()
        grp.stage(capi.MARGINALIZE, batches, threads=host_threads)
        work[0].synchronize()
        flush_l2()
        ms = grp.launch_timed()
        reps = grp.fetch(batches, full=full_report)
        return ms, reps

    def e2e_step():
        restore()
        work[0].synchronize()
        flush_l2()
        t0 = time.perf_counter()
        reps = grp.update(capi.MARGINALIZE, batches, threads=host_threads)  # host buffers in, reports out
        return time.perf_counter() - t0, reps

    # ---------------------------------------------------------------- device-timed steps
    for _ in range(W):
        device_step()
    sampler = ClockSampler(physical_gpu_index(local_rank))
    sampler.start()
    barrier()
    l0 = grp.launch_count()
    t_wall0 = time.perf_counter()
    times = []
    for k in range(K):
        ms, reps = device_step(full_report=args.dump_outputs is not None and k == K - 1)
        times.append(ms)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches_timed = grp.launch_count() - l0
    assert all(r["m"] == N_FEAT * (2 * N_CLONES - 3) for r in reps), [r["m"] for r in reps]
    if args.dump_outputs is not None:
        dump_outputs(args.dump_outputs, reps, work, suffix=f"_rank{rank}" if world > 1 else "")
    dev_ms = float(np.sum(times))
    if args.skip_extras:
        sampler.stop_flag = True
        if rank == 0:
            print(json.dumps({"profiling_only": True, "ms_per_step": dev_ms / K, "gpu_launches": int(launches_timed), "filters": F}))
        return
    # ---------------------------------------------------------------- end to end through the C-ABI batch call, host buffers
    for _ in range(W):
        e2e_step()
    e2e_times = []
    for _ in range(K):
        dt, reps = e2e_step()
        e2e_times.append(dt)
    e2e_s = float(np.sum(e2e_times))
    sampler.stop_flag = True
    sampler.join(timeout=2)
    up16 = lambda x: (x + 15) & ~15
    up256 = lambda x: (x + 255) & ~255
    rep_bytes = F * up256(16 + 5 * up16(4 * N_FEAT) + up16(4 * 3 * N_FEAT) + up16(4 * N_FEAT))
    h2d_bytes = sum(b.h2d_bytes() for b in batches) + up256(F * 416)  # + the UpdArgs array (sizeof(UpdArgs<float>) = 416)
    # ---------------------------------------------------------------- per-kernel profile of the batch step
    work[0].set_option(1, 1.0)
    kern_ms = kernel_table(grp, device_step)
    work[0].set_option(1, 0.0)
    dom = max(kern_ms, key=kern_ms.get)
    # 32 filters per GPU (side number)
    side32 = None
    if rank == 0 and F != 32:
        w32 = [capi.Engine(DTYPE, device=local_rank, max_clones=N_CLONES + 8, max_tracks=512, max_obs=512 * N_CLONES) for _ in range(32)]
        g32 = capi.Batch(w32)
        b32 = [batches[i % F] for i in range(32)]
        ts = []
        for r in range(7):
            for i, w in enumerate(w32):
                w.copy_state_from(tmpl_eng[i % F])
            g32.stage(capi.MARGINALIZE, b32, threads=host_threads)
            w32[0].synchronize()
            flush_l2()
            ts.append(g32.launch_timed())
            g32.fetch(b32)
        side32 = 32 / (float(np.mean(ts[2:])) * 1e-3)
        g32.close()

    # ---------------------------------------------------------------- reduce over ranks
    dev_ms, e2e_s = shard.max_over_ranks([dev_ms, e2e_s], device="cuda")
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    single, single_kern = single_filter_record(local_rank, flush_l2, steps=min(K, 20), warm=W)
    stress = stress_record(local_rank, flush_l2)
    stream = stream_record(local_rank)
    parity = parity_record(local_rank)

    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    peak_src = "of measured (MEASURED_PEAKS.json hbm_gbs, burst copy)" if "hbm_gbs" in peaks else "of fallback (6.65 TB/s)"
    bytes_alg = algorithmic_bytes(N_FEAT, N_CLONES, 4)
    achieved = F * bytes_alg / (kern_ms[dom] * 1e-3) / 1e9
    traffic = None
    try:
        traffic = json.loads((ROOT / "profiles" / "traffic.json").read_text()).get(dom)
    except Exception:
        pass
    cpu_val, cpu_n, cpu_wall = cpu_oracle_updates(args.cpu_seconds, 1, DTYPE)

    value = world * F * K / (dev_ms * 1e-3)
    line = {
        "metric": "msckf_updates_per_sec", "value": value, "unit": "updates/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{F} independent filters per GPU, each ONE update() (= one marginalize(): triangulation + Jacobian/null-space + gating + "
                               f"compression + Kalman/covariance update) on {N_FEAT} features x {N_CLONES} camera clones, float32 (BASELINE configs[1] x {F} = the "
                               f"per-GPU share of configs[3], 64 sequences on 8 GPUs), one device batch per step; states restored and L2 flushed (256 MiB "
                               "write) between timed steps; one filter alone: see `single`",
                   "filters_per_gpu": F, "updates_per_step_per_gpu": F, "n_features": N_FEAT, "n_clones": N_CLONES,
                   "stacked_rows_m": N_FEAT * (2 * N_CLONES - 3), "state_dim_n": 15 + 6 * N_CLONES,
                   "timing": "CUDA events on the batch's stream around the update's kernels, summed over steps, max over ranks",
                   "l2": "flushed between timed iterations", "parallelism": f"independent filters, {world} GPU(s) x {F}, no data-path collective"},
        "clocks": sampler.result(),
        "e2e": {"value": world * F * K / e2e_s, "unit": "updates/s", "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": int(rep_bytes),
                "ms_per_step": 1e3 * e2e_s / K, "e2e_over_device": (e2e_s / K) / (dev_ms * 1e-3 / K),
                "path": "msckf_b200_batch_update (C-ABI) with host buffers: pack into pinned, one H2D, kernels, one D2H, unpack; host wall clock"},
        "gpu_launches": int(launches_timed),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic,
                     "kernel": dom, "kernel_ms": kern_ms[dom], "peak_source": peak_src, "algorithmic_bytes_per_update": bytes_alg,
                     "updates_per_launch": F, "whole_step_gbs": F * bytes_alg / (dev_ms / K * 1e-3) / 1e9,
                     "whole_step_frac": F * bytes_alg / (dev_ms / K * 1e-3) / 1e9 / hbm_peak,
                     "single_filter_frac": bytes_alg / (single_kern[max(single_kern, key=single_kern.get)] * 1e-3) / 1e9 / hbm_peak,
                     "reference_path_gflop_per_update": algorithmic_flops(N_FEAT, N_CLONES) / 1e9,
                     "note": "the path moves < 8 MB per update inside L2 and executes ~0.25 GFLOP: it is latency-bound, see DESIGN.md 6",
                     "kernel_ms_all": kern_ms},
        "cpu_baseline": {"value": cpu_val, "unit": "updates/s", "cores": 1, "kind": "port",
                         "sample": f"{cpu_n} marginalize() calls of the same {N_FEAT}x{N_CLONES} fp32 workload in {cpu_wall:.1f} s, "
                                   "oracle/ (CPU restatement of the reference's Eigen path, thin-Q form), single thread like the reference"},
        "single": single, "stress": stress, "stream": stream, "parity": parity,
        "batch64": {"filters_per_gpu": F, "value": value, "unit": "updates/s", "value_32_filters_per_gpu": side32,
                    "note": f"`value` IS this configuration: {F} filters per GPU x {world} GPU(s) ({F * world} sequences)"},
        "wall_s_timed_region": t_wall,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
