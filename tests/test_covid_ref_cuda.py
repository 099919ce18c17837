"""The reference's OWN COVID-19 CUDA kernels on the same GPU (BASELINE config 4).

oracle/_ref/libref_covid_cuda.so is built by oracle/build_ref_covid.py from the reference's sources where they are present
(nothing copied).  Here:

  * the reference CUDA path replays the golden trace recorded from the reference's PYTHON path (the comparison the
    reference's tests/run_covid19_cpu_gpu_consistency_checks.py makes through WarpDrive's EnvironmentCPUvsGPU, with
    num_envs = 3), and
  * aie_covid_step_kernel replays the same trace next to it: both against the golden, and against each other.  Where
    the library is not built, the reference CUDA path's values recorded from it stand in for it
    (tests/golden/reference_tapes/covid_ref_cuda.*, oracle/ref_tape.py; AIE_RECORD_REFERENCE=1 records them again where
    the library is built), so the comparison with ours runs everywhere.

Tolerances.  The reference's CUDA path is a float32 re-implementation of a Python path that promotes to float64 in
places, so the two differ in the last digits (that is why WarpDrive's checker compares with a tolerance rather than
exactly); REF_RTOL / REF_ATOL below are what the reference's own CUDA path needs against its own Python path on this
trace (measured maxima are printed).  aie_covid_step_kernel follows the Python path and keeps the suite's 1e-6.
"""
import json
import os

import numpy as np
import pytest

from ai_economist_b200.foundation.covid19 import build_covid_params
from oracle import build_ref_covid
from oracle import ref_tape

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden_covid")
OBS_KEYS = ["agent_state", "postsubsidy", "lagged", "policy_ind", "scalars"]
REF_RTOL, REF_ATOL = 2e-3, 2e-4   # reference CUDA (float32) vs reference Python (float64 promotions), see module docstring
RTOL, ATOL = 1e-6, 1e-9           # aie_covid_step_kernel vs reference Python

pytestmark = pytest.mark.gpu
needs_library = pytest.mark.skipif(not build_ref_covid.available(),
                                   reason="oracle/_ref/libref_covid_cuda.so not built (needs the reference's sources)")


def _load(name="covid_seed3.npz"):
    z = np.load(os.path.join(GOLDEN_DIR, name))
    meta = json.loads(str(z["meta_json"]))
    return z, meta, build_covid_params(**meta["kwargs"])


def _maxdev(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b) / (np.abs(b) + 1e-3))) if a.size else 0.0


def test_reference_cuda_kernels_replay_the_python_golden_trace_next_to_ours():
    import torch
    from ai_economist_b200.covid_stepper import CudaCovidStepper

    z, meta, p = _load()
    E = 3
    # the reference's kernels run wherever the library is built; elsewhere their recorded values stand in for them
    live = build_ref_covid.available() and not ref_tape.recording()
    tape = (ref_tape.Tape(available=build_ref_covid.available) if live else
            ref_tape.Tape("covid_ref_cuda", "covid_seed3", available=build_ref_covid.available))
    if tape.live:
        from oracle.ref_covid_cuda import RefCovidCuda
        ref = RefCovidCuda(p, E)
    ours = CudaCovidStepper(p, E, auto_reset=False)
    ours.reset()
    worst = {}
    for t in range(1, meta["n_steps"] + 1):
        a = torch.as_tensor(z["act_a"][t - 1].astype(np.int32), device="cuda")
        pl = int(z["act_p"][t - 1])
        if tape.live:
            ref.t["actions_a"][:] = a; ref.t["actions_p"][:] = pl
            ref.step()
        ours.buf["actions_agent"][:] = a; ours.buf["actions_planner"][:] = pl
        ours.step()
        if t % 7 and t < meta["n_steps"] - 2 and t > 3:
            continue   # full comparison on a subset of days (every day costs two D2H round trips per field)
        for e in (0, E - 1):
            r, o = (ref.read_obs(e) if tape.live else {}), ours.read_obs(e)
            where = "ours vs reference CUDA, day %d" % t
            for k in OBS_KEYS + ["rew_a"]:
                g = z[k][t] if k != "rew_a" else z["rew_a"][t - 1]
                if tape.live:
                    worst[k] = max(worst.get(k, 0.0), _maxdev(r[k], g))
                    assert np.allclose(r[k], g, rtol=REF_RTOL, atol=REF_ATOL), "reference CUDA vs Python golden, day %d: %s" % (t, k)
                assert np.allclose(o[k], g, rtol=RTOL, atol=ATOL), "ours vs Python golden, day %d: %s" % (t, k)
                tape.close(k, r.get(k), o[k], rtol=REF_RTOL, atol=REF_ATOL, where=where)
            if tape.live:
                worst["rew_p"] = max(worst.get("rew_p", 0.0), _maxdev(r["rew_p"], z["rew_p"][t - 1]))
                assert np.isclose(float(r["rew_p"]), float(z["rew_p"][t - 1]), rtol=REF_RTOL, atol=REF_ATOL), "day %d: rew_p" % t
            assert np.isclose(float(o["rew_p"]), float(z["rew_p"][t - 1]), rtol=RTOL, atol=ATOL)
            tape.close("rew_p", r.get("rew_p"), float(o["rew_p"]), rtol=REF_RTOL, atol=REF_ATOL, where=where)
            # masks are exact in all three
            if tape.live:
                assert np.array_equal(r["mask_a"], z["mask_a"][t]) and np.array_equal(r["mask_p"], z["mask_p"][t]), "day %d: masks" % t
            assert np.array_equal(o["mask_a"], z["mask_a"][t]) and np.array_equal(o["mask_p"], z["mask_p"][t])
            for k in ("mask_a", "mask_p"):
                tape.equal(k, r.get(k), o[k], where)
            assert int(z["done"][t - 1]) == int(o["done"])
            tape.equal("done", int(r["done"]) if tape.live else None, int(o["done"]), where)
    tape.finish()
    if tape.live:
        print("max relative deviation of the reference CUDA path from its Python path:", {k: "%.2e" % v for k, v in worst.items()})


@needs_library
def test_reference_cuda_reset_restores_the_saved_arrays():
    import torch
    from oracle.ref_covid_cuda import RefCovidCuda

    z, meta, p = _load()
    ref = RefCovidCuda(p, 2)
    first = None
    for ep in range(2):
        for t in range(1, 31):
            ref.t["actions_a"][:] = torch.as_tensor(z["act_a"][t - 1].astype(np.int32), device="cuda")
            ref.t["actions_p"][:] = int(z["act_p"][t - 1])
            ref.step()
        snap = {k: v.copy() for k, v in ref.read_obs(1).items()}
        if first is None:
            first = snap
        else:
            for k in first:
                assert np.array_equal(first[k], snap[k]), k
        ref.reset()
