"""ASL / EuRoC folder round trip (no GPU): `asl.write_mav0` -> files -> the C++ player's parsers (`asl_player --dry-run`).

The reference has no tests for its readers (datasets/asl_readers.cpp); these pin ours: every number written is read
back (checksums over all IMU readings, track rows and ids), the camera block and the filter parameters survive the
YAML subset, and the layout is the EuRoC one."""
import os

import numpy as np
import pytest

from msckf_mono_b200 import asl, synth


@pytest.fixture(scope="module")
def mav0(tmp_path_factory):
    wl = synth.make_stream_workload(n_frames=15, seq=3, max_features=40)
    root = tmp_path_factory.mktemp("asl")
    return wl, asl.write_mav0(wl, str(root))


def test_layout_is_euroc(mav0, engine_lib):
    _, m = mav0
    for rel in ("imu0/data.csv", "cam0/data.csv", "cam0/sensor.yaml", "cam0/tracks.csv", "state_groundtruth_estimate0/data.csv", "msckf.yaml"):
        assert os.path.exists(os.path.join(m, rel)), rel
    with open(os.path.join(m, "imu0/data.csv")) as f:
        assert f.readline().startswith("#timestamp [ns],w_RS_S_x")
    with open(os.path.join(m, "state_groundtruth_estimate0/data.csv")) as f:
        assert f.readline().startswith("#timestamp,p_RS_R_x")


def test_player_reads_back_every_number(mav0, engine_lib):
    wl, m = mav0
    r = asl.run_player(m, dry_run=True)
    frames = wl["frames"]
    assert r["frames"] == len(frames) and r["groundtruth"] == len(frames)
    assert r["imu"] == sum(len(fr["imu"]) for fr in frames)
    rows = sum(len(fr[k][1]) for fr in frames for k in ("update", "add"))
    assert r["track_rows"] == rows
    imu_sum = sum(float(np.sum(om) + np.sum(a)) for fr in frames for (om, a, _) in fr["imu"])
    assert abs(r["imu_checksum"] - imu_sum) <= 1e-9 * max(1.0, abs(imu_sum))
    tr_sum = sum(float(np.sum(fr[k][0])) for fr in frames for k in ("update", "add"))
    assert abs(r["track_checksum"] - tr_sum) <= 1e-9 * max(1.0, abs(tr_sum))
    assert r["id_checksum"] == sum(int(np.sum(fr[k][1])) for fr in frames for k in ("update", "add"))
    assert r["fu"] == wl["camera"]["f_u"] and r["fv"] == wl["camera"]["f_v"]
    assert r["T_BS_03"] == pytest.approx(wl["camera"]["p_C_I"][0], abs=0)
    assert r["max_track_length"] == wl["params"]["max_track_length"] and r["feature_cov"] == 7.0


def test_timestamps_are_ordered_and_imu_precedes_its_frame(mav0):
    wl, m = mav0
    imu = np.loadtxt(os.path.join(m, "imu0/data.csv"), delimiter=",", comments="#")
    cam_t = [int(l.split(",")[0]) for l in open(os.path.join(m, "cam0/data.csv")) if not l.startswith("#")]
    t = imu[:, 0].astype(np.int64)
    assert np.all(np.diff(t) == 5_000_000)  # 200 Hz
    assert np.all(np.diff(cam_t) == 50_000_000)  # 20 Hz
    assert t[0] == cam_t[0] + 5_000_000 and t[-1] == cam_t[-1]
    tr = np.loadtxt(os.path.join(m, "cam0/tracks.csv"), delimiter=",", comments="#")
    assert set(tr[:, 0].astype(np.int64)) <= set(cam_t)


def test_player_rejects_missing_folder(engine_lib, tmp_path):
    with pytest.raises(RuntimeError):
        asl.run_player(str(tmp_path / "missing" / "mav0"), dry_run=True)


def test_player_call_sequence_on_cpu_against_the_oracle(mav0, oracle_lib, tmp_path):
    """The compiled player's host logic without a GPU: asl_player.cpp linked against tests/stub/stub_engine.cpp (a fake
    of the C-ABI with no numerics) must hand the class the same frames, IMU readings and tracked / new feature split as
    `synth.drive` hands the oracle: the clone-window size per frame (update / addFeatures / pruneEmptyStates bookkeeping)
    is then identical.  pruneRedundantStates is off here: its decisions depend on poses, which the fake does not compute."""
    import subprocess
    from tests.common import ROOT, make_oracle
    wl, m = mav0
    exe = ROOT / "tests" / "stub" / "asl_player_stub"
    src = [ROOT / "msckf_mono_b200" / "asl" / "asl_player.cpp", ROOT / "tests" / "stub" / "stub_engine.cpp",
           ROOT / "msckf_mono_b200" / "asl" / "asl_io.hpp", ROOT / "include" / "msckf_mono" / "msckf.h"]
    if (not exe.exists()) or any(s.stat().st_mtime > exe.stat().st_mtime for s in src):
        subprocess.check_call(["g++", "-O1", "-std=c++17", f"-I{ROOT / 'include'}", f"-I{ROOT / 'msckf_mono_b200' / 'asl'}",
                               str(src[0]), str(src[1]), "-o", str(exe)])
    out = tmp_path / "traj_stub.csv"
    r = subprocess.run([str(exe), "--mav0", m, "--dtype", "f64", "--out", str(out), "--prune-redundant", "0", "--state-id", "frame"],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    import json
    summary = json.loads(r.stdout.strip().splitlines()[-1])
    frames = wl["frames"]
    assert summary["frames"] == len(frames) and summary["imu_readings"] == sum(len(fr["imu"]) for fr in frames)
    tr = asl.read_trajectory(str(out))
    o = make_oracle(oracle_lib, np.float64)
    ncl = []
    synth.drive(o, wl, prune_redundant=False, on_frame=lambda k, f: ncl.append(f.getNumCamStates()))
    assert np.array_equal(tr["n_clones"], np.array(ncl))
    assert np.array_equal(tr["t_ns"], np.array([int(l.split(",")[0]) for l in open(os.path.join(m, "cam0/data.csv")) if not l.startswith("#")]))
