"""Randomised fuzz (build container only): adapters.ReferenceApiEnv (explicit resets, nested numpy dictionaries) against
the LIVE reference on configurations from tools/fuzz_emu_vs_oracle.random_config, three short episodes each, with random
flatten_observations / flatten_masks.   python tools/fuzz_reference_api_vs_reference.py [n] [seed]"""
import os
import sys
import traceback

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import fuzz_emu_vs_oracle as fz  # noqa: E402
from ai_economist_b200 import foundation  # noqa: E402
from oracle import ref_harness as rh  # noqa: E402
from oracle import ref_tape  # noqa: E402
from tests.emu.emu_stepper import emu_factory  # noqa: E402


def pick(env, obs, rng):
    """A random unmasked action per agent from either mask layout (flat vector or {subspace: mask})."""
    acts = {}
    for idx, o in obs.items():
        ag, m = env.get_agent(idx), o["action_mask"]
        names = [n for n in ag._action_names if n != "PassiveAgentPlaceholder"]
        if not names:                      # passive multi-action planner: one placeholder subspace, always NO-OP
            acts[idx] = [0] if ag.multi_action_mode else 0
            continue
        if isinstance(m, dict):
            parts = [np.asarray(m[n], np.float64).reshape(-1) for n in names]
        else:
            m = np.asarray(m, np.float64)
            if ag.multi_action_mode:
                dims = [int(ag.action_dim[n]) for n in names]
                parts = [m[sum(dims[:i]) + 1:sum(dims[:i + 1])] for i in range(len(dims))]
            else:
                parts, off = [], 1
                for n in names:
                    k = int(ag.action_dim[n]); parts.append(m[off:off + k]); off += k
        if ag.multi_action_mode:
            acts[idx] = [int(rng.choice(len(p) + 1, p=np.r_[1.0, p] / (1.0 + p.sum()))) for p in parts]
        else:
            flat = np.r_[1.0, np.concatenate(parts)] if parts else np.ones(1)
            acts[idx] = int(rng.choice(len(flat), p=flat / flat.sum()))
    return acts


def run_one(name, kw, seed, tape=None):
    """tape (oracle/ref_tape.py): None compares with the live reference, a replaying tape with its recorded digests.
    The actions are picked from the facade's observations (equal to the reference's, which every check compares)."""
    import json
    from oracle.ref_tape import same_log, same_metrics, same_tree

    tape = tape or ref_tape.Tape()
    cfg = dict(kw, scenario_name=name, flatten_observations=bool(seed % 2), flatten_masks=bool((seed // 2) % 2),
               episode_length=12, dense_log_frequency=1, world_dense_log_frequency=5)
    if tape.live:
        f = rh.load_reference_foundation()
        ref = f.make_env_instance(**cfg)
    mine = foundation.make_env_instance(**cfg, reference_api=True, stepper_factory=emu_factory)
    if tape.live:
        ref.seed(seed)
    mine.seed(seed)
    o1 = r1 = d1 = p1 = m1 = log1 = None
    for ep in range(3):
        rng = np.random.RandomState(seed * 10 + ep)
        if tape.live:
            o1 = ref.reset()
        o2 = mine.reset()
        same_tree(tape, "obs", o1, o2, "ep %d reset" % ep)
        if ep > 0:   # previous_episode_metrics: what _finalize_logs stored when the last episode ended
            with np.errstate(all="ignore"):
                p1 = ref.previous_episode_metrics if tape.live else None
                same_metrics(tape, "previous metrics", p1, mine.previous_episode_metrics, "ep %d" % ep)
        for t in range(12):
            a = pick(mine, o2, rng)
            if tape.live:
                o1, r1, d1, _ = ref.step(a)
            o2, r2, d2, _ = mine.step(a)
            same_tree(tape, "obs", o1, o2, "ep %d t %d obs" % (ep, t))
            same_tree(tape, "rew", r1, r2, "ep %d t %d rew" % (ep, t))
            tape.equal("done", ref_tape.flags(d1) if tape.live else None, ref_tape.flags(d2), "ep %d t %d" % (ep, t))
        tape.equal("completions", int(ref._completions) if tape.live else None, mine._completions, "ep %d" % ep)
        # the dense log of the episode that just ended (world / states / actions / rewards + every component's log)
        if tape.live:
            log1 = json.loads(json.dumps(ref.previous_episode_dense_log))
        same_log(tape, "dense log", log1, json.loads(json.dumps(mine.previous_episode_dense_log)), "ep %d dense log" % ep)
        # env.metrics at the end of the episode (scenario + every component's get_metrics)
        with np.errstate(all="ignore"):
            m1 = ref.metrics if tape.live else None
            same_metrics(tape, "metrics", m1, mine.metrics, "ep %d" % ep)
    tape.finish()


if __name__ == "__main__":
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 30
    rng = np.random.RandomState(int(sys.argv[2]) if len(sys.argv) > 2 else 0)
    bad = 0
    for i in range(n):
        name, kw = fz.random_config(rng)
        try:
            run_one(name, kw, seed=700 + i)
        except Exception as ex:  # noqa: BLE001
            bad += 1
            print("[%d] FAILED %s %r\n    %s" % (i, name, kw, "".join(traceback.format_exception_only(type(ex), ex)).strip()[:500]))
    print("%d configs x 3 episodes, %d failures" % (n, bad))
