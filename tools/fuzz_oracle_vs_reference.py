"""Randomised configuration fuzz (build container only): the C oracle against the LIVE imported reference on
configurations drawn by tools/fuzz_emu_vs_oracle.random_config.  python tools/fuzz_oracle_vs_reference.py [n] [seed]"""
import sys, traceback
import os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tools'))
import numpy as np
from oracle import configs
from oracle import ref_tape
from oracle.validate_vs_reference import run
import fuzz_emu_vs_oracle as fz
rng = np.random.RandomState(int(sys.argv[2]) if len(sys.argv) > 2 else 5)
n = int(sys.argv[1]) if len(sys.argv) > 1 else 30
bad = 0
for i in range(n):
    name, kw = fz.random_config(rng)
    cfg = dict(kw, scenario_name=name)
    configs.CONFIGS["_fuzz"] = cfg
    try:
        run("_fuzz", 100 + i, min(80, kw["episode_length"]), verbose=False)
    except ref_tape.Mismatch as ex:
        bad += 1; print("[%d] MISMATCH %r\n    %s" % (i, cfg, str(ex)[:300]))
    except Exception as ex:
        msg = "".join(traceback.format_exception_only(type(ex), ex)).strip()[:300]
        print("[%d] exception (reference or harness): %s | %s" % (i, msg, {k: cfg[k] for k in ("scenario_name",)}))
print(n, "configs,", bad, "mismatches")
