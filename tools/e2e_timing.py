"""Tuning aid: wall time of the pipelined end-to-end solve (pvio_b200_batch_solve_host) for a library variant
named by PVIO_B200_TUNE_LIB."""
import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from synthetic import synth
from pvio_b200.bundle_adjustor import BundleAdjustor
W = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
w, st, _ = synth.make_cfg2()
ba = BundleAdjustor(max_windows=W, max_frames=10, max_landmarks=512, max_obs=4608)
ba.batch_set(0, w, st); ba.batch_replicate(W)
fr = np.zeros((W, w.N * 16)); rh = np.zeros((W, w.M))
devnull = os.open(os.devnull, os.O_WRONLY); err = os.dup(2)
os.dup2(devnull, 2)
ts = []
for _ in range(6):
    t = time.perf_counter(); _, _, sm = ba.batch_solve_host(W, w.N, w.M, frames=fr, rho=rh); ts.append(time.perf_counter() - t)
os.dup2(err, 2)
its = sum(x.iterations for x in sm)
best = min(ts[1:])
print(f"{os.environ.get('PVIO_B200_TUNE_LIB', 'shipped')}: {best * 1e3:.2f} ms  {its / best:.0f} window-iterations/s")
