import sys
from pathlib import Path
import numpy as np
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from msckf_mono_b200 import capi, synth
from tests.parity_cases import make_engine
wl = synth.make_window_workload(n_features=300, n_clones=30, seq=0)
for thr in (1e-13, 1e-12, 0.25e-11, 0.5e-11, 1e-11, 2e-11, 4e-11, 1e-10, 1e-9):
    f = make_engine(np.float64, max_clones=40, max_tracks=512, max_obs=512 * 30)
    synth.drive(f, wl, marginalize_last=False)
    capi.Engine(np.float64, borrowed=f.engineHandle()).set_option(0, thr)
    f.marginalize()
    print(thr, f.counters()["rows_kept"], f.counters()["m"])
    if thr == 1e-11:
        pv = capi.Engine(np.float64, borrowed=f.engineHandle()).rank_pivots()
        o = np.argsort(pv)
        print("   smallest pivot ratios:", [(int(i), float("%.3g" % pv[i])) for i in o[:14]])
