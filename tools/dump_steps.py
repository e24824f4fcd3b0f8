"""Developer helper (GPU box): integrator step counts of the bench batch, for the queue-order study."""
import os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
from metrotrpl_b200 import trial_move_evaluation as tme

ini, t = bench.workload_inputs()
vals, uncs = bench.workload_measurement()
sf = bench.make_shared_fields(ini, t, vals, uncs)
states = bench.draw_states(4096, seed=20261018)
res = tme.eval_trial_moves(states, np.ones((4096, 3)), {"TRPL": 1.0}, sf)
np.savez(os.path.join(ROOT, "gpurun_out", "steps.npz"), states=states, nsteps=res.nsteps, status=res.status,
         logll=res.per_meas)
print("mean steps", res.nsteps[..., 0].mean())
