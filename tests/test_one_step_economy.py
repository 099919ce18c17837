"""SimpleLabor + the one-step-economy scenario (SURVEY §8f row 3; reference: components/simple_labor.py:16-134,
scenarios/one_step_economy/one_step_economy.py:15-336).

Golden traces recorded from the unmodified reference (oracle/gen_golden_one_step.py -> tests/golden_one_step/): five
episodes each with env.reset() in between, replayed here through the public API with auto_reset on - on the 1-lane
emulation of the device source (CPU) and on the CUDA build (-m gpu).  Masks and the numpy stream bit-exact; observations,
rewards, coin / labor / production within 1e-6 relative; the metrics of every finished episode.  The reset of this scenario
draws nothing, so the device's snapshot restore is the reference's reset.
tests/test_fuzz_subsets.py adds random configurations against the live reference.
"""
import glob
import json
import os

import numpy as np
import pytest

from ai_economist_b200 import foundation

FILES = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden_one_step", "*.npz")))


def _replay(path, factory):
    z = np.load(path)
    meta = json.loads(str(z["meta_json"]))
    kw = dict(meta["reference_kwargs"])
    name = kw.pop("scenario_name")
    kw["components"] = [tuple(c) for c in kw["components"]]
    extra = dict(stepper_factory=factory) if factory else dict(device="cuda:0")
    seed = meta["seed"]
    env = foundation.make_env_instance(name, n_envs=3, auto_reset=True, seeds=[seed] * 3, **kw, **extra)
    env.seed([seed + 1] * 3)
    env.reset()
    s = env.stepper
    assert s.buf["obs_agent_map"].shape[-1] == 0 and "obs_planner_map" not in s.buf   # nothing spatial in this scenario

    def check(t, e):
        o, st = s.read_obs(e), s.read_state(e)
        for k in ("a_mask", "p_mask"):
            assert np.array_equal(z[k][t], np.asarray(o[k]).reshape(z[k][t].shape)), "t=%d: %s" % (t, k)
        for k in ("a_flat", "p_flat", "p_agents", "time"):
            assert np.allclose(z[k][t], np.asarray(o[k]).reshape(z[k][t].shape), rtol=1e-6, atol=1e-7), "t=%d: %s" % (t, k)
        assert np.array_equal(z["mt_key"][t], st["mt_key"]) and int(z["mt_pos"][t]) == int(st["mt_pos"][0]), "t=%d: numpy stream" % t
        for k, mine in (("coin", "coin"), ("labor", "labor"), ("production", "build_payment")):
            assert np.allclose(z[k][t], st[mine], rtol=1e-6, atol=1e-9), "t=%d: %s" % (t, k)

    check(0, 2)
    n_done = 0
    for t in range(1, int(meta["n_steps"]) + 1):
        aa = np.repeat(z["act_a"][t - 1][None], 3, axis=0).astype(np.int32)
        ap = np.repeat(z["act_p"][t - 1][None], 3, axis=0).astype(np.int32) if z["act_p"].shape[1] else None
        env.step((aa, ap))
        got = s.to_numpy(s.buf["reward"])
        assert np.allclose(z["rew"][t - 1], got[2], rtol=1e-6, atol=1e-9), "t=%d: rewards" % t
        assert np.array_equal(got[0], got[2])   # replicas with the same seeds agree (env indexing)
        assert int(z["done"][t - 1]) == int(s.to_numpy(s.buf["done"])[2])
        if z["done"][t - 1]:
            n_done += 1
            want, have = meta["metrics"][str(t)], env.previous_episode_metrics_of(2)
            assert set(want) == set(have), sorted(set(want) ^ set(have))[:5]
            for k, v in want.items():
                a, b = float(v), float(have[k])
                assert (np.isnan(a) and np.isnan(b)) or abs(a - b) <= 1e-6 * max(1.0, abs(a)), "t=%d metric %s: %r vs %r" % (t, k, a, b)
        check(t, 2)
    assert n_done >= 4


@pytest.mark.parametrize("path", FILES, ids=lambda p: os.path.basename(p))
def test_emulated_one_step_economy_matches_reference_golden_trace(path):
    from tests.emu.emu_stepper import emu_factory
    _replay(path, emu_factory)


@pytest.mark.gpu
@pytest.mark.parametrize("path", FILES, ids=lambda p: os.path.basename(p))
def test_cuda_one_step_economy_matches_reference_golden_trace(path):
    _replay(path, None)


def test_one_step_economy_rejects_what_the_reference_rejects():
    from tests.emu.emu_stepper import emu_factory
    base = dict(n_agents=3, world_size=[1, 1], episode_length=2, stepper_factory=emu_factory, n_envs=1, seed=1)
    with pytest.raises(NotImplementedError):   # planner reward outside the scenario's two (one_step_economy.py:331-334)
        foundation.make_env_instance("one-step-economy", components=[("SimpleLabor", {})],
                                     planner_reward_type="inv_income_weighted_coin_endowments", **base)
    with pytest.raises(NotImplementedError):   # the scenario is defined for SimpleLabor (+ PeriodicBracketTax)
        foundation.make_env_instance("one-step-economy", components=[("SimpleLabor", {}), ("Gather", {})], **base)
    with pytest.raises(AssertionError):
        foundation.make_env_instance("one-step-economy", components=[("SimpleLabor", {})], labor_exponent=1.0, **base)


def test_reference_api_facade_runs_the_one_step_economy_like_the_reference():
    """reference_api=True: the reference's single-env interface (nested dicts, named fields) over replica 0, side by side with
    the reference through three episodes: observations, rewards, done, metrics (the reference's values as recorded,
    oracle/ref_tape.py)."""
    from oracle import ref_harness as rh
    from oracle import ref_tape
    from oracle.ref_tape import same_metrics, same_tree
    from tests.emu.emu_stepper import emu_factory
    cfg = dict(components=[("SimpleLabor", dict(mask_first_step=True, payment_max_skill_multiplier=3)),
                           ("PeriodicBracketTax", dict(bracket_spacing="us-federal", period=2, tax_model="model_wrapper", rate_disc=0.05))],
               n_agents=6, world_size=[1, 1], episode_length=2, flatten_observations=False, flatten_masks=True)
    env = foundation.make_env_instance("one-step-economy", reference_api=True, stepper_factory=emu_factory, seed=5, **cfg)
    env.seed(7)
    tape = ref_tape.Tape("one_step_economy_facade", 0)
    if tape.live:
        f = rh.load_reference_foundation()
        np.random.seed(5)
        ref = f.make_env_instance(scenario_name="one-step-economy", **cfg)
        ref.seed(7)

    rng = np.random.RandomState(1)
    o1 = r1 = d1 = m1 = None
    for ep in range(3):
        if tape.live:
            o1 = ref.reset()
        o2 = env.reset()
        same_tree(tape, "obs", o1, o2, "ep %d reset" % ep)
        for t in range(2):
            acts = {str(i): int(rng.choice(np.flatnonzero(np.asarray(o2[str(i)]["action_mask"])))) for i in range(6)}
            pm = np.asarray(o2["p"]["action_mask"]).reshape(7, -1)
            acts["p"] = [int(rng.choice(np.flatnonzero(pm[b]))) for b in range(7)]
            if tape.live:
                o1, r1, d1, _ = ref.step(acts)
            o2, r2, d2, _ = env.step(acts)
            same_tree(tape, "obs", o1, o2, "ep %d t %d obs" % (ep, t))
            same_tree(tape, "rew", r1, r2, "ep %d t %d rew" % (ep, t))
            tape.equal("done", ref_tape.flags(d1) if tape.live else None, ref_tape.flags(d2), "ep %d t %d" % (ep, t))
        with np.errstate(all="ignore"):
            m1 = ref.metrics if tape.live else None
            same_metrics(tape, "metrics", m1, env.metrics, "ep %d" % ep)
    tape.finish()
