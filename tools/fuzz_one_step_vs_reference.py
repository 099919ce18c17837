"""Randomised fuzz (build container only): the one-step-economy scenario with SimpleLabor (+ PeriodicBracketTax) on the
1-lane emulation of the device source against the LIVE reference: observations, masks, rewards, the numpy stream, and the
metrics of every finished episode, across auto-resets.   python tools/fuzz_one_step_vs_reference.py [n] [seed]"""
import os
import sys
import traceback

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ai_economist_b200 import foundation  # noqa: E402
from oracle import ref_harness as rh  # noqa: E402
from oracle import ref_tape  # noqa: E402
from tests.emu.emu_stepper import emu_factory  # noqa: E402


def random_config(rng):
    A = int(rng.choice([2, 3, 6, 10, 31, 40]))
    comps = [("SimpleLabor", dict(mask_first_step=bool(rng.rand() < 0.8), payment_max_skill_multiplier=float(rng.choice([1.5, 3, 5])),
                                  pareto_param=4.0))]
    if rng.rand() < 0.85:
        model = str(rng.choice(["model_wrapper", "model_wrapper", "us-federal-single-filer-2018-scaled"]))
        comps.append(("PeriodicBracketTax", dict(bracket_spacing="us-federal", period=int(rng.choice([1, 2, 3])), tax_model=model,
                                                 rate_disc=float(rng.choice([0.05, 0.1])), usd_scaling=float(rng.choice([1000.0, 50.0])))))
    if rng.rand() < 0.3:
        comps = comps[::-1]
    reward = str(rng.choice(["coin_minus_labor_cost", "isoelastic_coin_minus_labor"]))
    return dict(scenario_name="one-step-economy", components=comps, n_agents=A, world_size=[1, 1],
                episode_length=int(rng.choice([2, 2, 3, 5])), multi_action_mode_agents=bool(rng.rand() < 0.3),
                multi_action_mode_planner=bool(rng.rand() < 0.8), flatten_observations=True, flatten_masks=True,
                allow_observation_scaling=bool(rng.rand() < 0.8), agent_reward_type=reward,
                isoelastic_eta=float(rng.choice([0.0, 0.23, 0.5])), labor_exponent=float(rng.choice([2.0, 1.5, 3.0])),
                labor_cost=float(rng.choice([1.0, 0.01, 0.2])),
                planner_reward_type=str(rng.choice(["inv_income_weighted_utility", "coin_eq_times_productivity"])),
                mixing_weight_gini_vs_coin=float(rng.choice([0.0, 0.4])))


def reference_arrays(ref, obs):
    A = ref.n_agents
    out = dict(a_flat=np.stack([obs[str(i)]["flat"] for i in range(A)]).astype(np.float32),
               a_mask=np.stack([obs[str(i)]["action_mask"] for i in range(A)]).astype(np.float32),
               p_flat=np.asarray(obs["p"]["flat"], np.float32), p_mask=np.asarray(obs["p"]["action_mask"], np.float32),
               p_agents=(np.stack([obs["p"]["p%d" % i] for i in range(A)]).astype(np.float32) if "p0" in obs["p"]
                         else np.zeros((A, 0), np.float32)),
               time=np.asarray(obs["p"]["time"], np.float32))
    key = np.random.get_state()
    out["mt_key"], out["mt_pos"] = np.array(key[1], np.uint32), int(key[2])
    ag = ref.world.agents
    out["coin"] = np.array([a.state["inventory"]["Coin"] for a in ag], np.float64)
    out["labor"] = np.array([a.state["endogenous"]["Labor"] for a in ag], np.float64)
    out["production"] = np.array([a.state["production"] for a in ag], np.float64)
    return out


def compare(tape, want, s, e, label):
    o, st = s.read_obs(e), s.read_state(e)
    want = want or {}
    for k in ("a_mask", "p_mask"):
        tape.equal(k, want.get(k), o[k], label)
    for k in ("a_flat", "p_flat", "p_agents", "time"):
        tape.close(k, want.get(k), o[k], rtol=1e-6, atol=1e-7, where=label)
    tape.equal("mt_key", want.get("mt_key"), st["mt_key"], label + ": numpy stream")
    tape.equal("mt_pos", want.get("mt_pos"), int(st["mt_pos"][0]), label + ": numpy stream")
    for k, mine in (("coin", "coin"), ("labor", "labor"), ("production", "build_payment")):
        tape.close(k, want.get(k), st[mine], rtol=1e-9, atol=1e-9, where=label + ": state")


def run_one(cfg, seed, episodes=4, tape=None):
    """tape (oracle/ref_tape.py): None compares with the live reference, a replaying tape with its recorded digests.
    The actions are drawn from the product's masks (equal to the reference's, which every check compares)."""
    tape = tape or ref_tape.Tape()
    if tape.live:
        f = rh.load_reference_foundation()
        np.random.seed(seed)   # the constructor draws the SimpleLabor skill table from the global stream
        ref = f.make_env_instance(**cfg)
        ref.seed(seed + 1)
        obs = ref.reset()
    kw = dict(cfg)
    name = kw.pop("scenario_name")
    env = foundation.make_env_instance(name, n_envs=2, stepper_factory=emu_factory, auto_reset=True, seeds=[seed, seed], **kw)
    env.seed([seed + 1, seed + 1])
    env.reset()
    s = env.stepper
    compare(tape, reference_arrays(ref, obs) if tape.live else None, s, 1, "reset")
    arng = np.random.RandomState(seed + 2)
    A, T = cfg["n_agents"], cfg["episode_length"]
    for t in range(1, episodes * T + 1):
        po = s.read_obs(1)
        actions, a_act, p_act = rh.sample_actions_from_masks(env, po["a_mask"], po["p_mask"], arng)
        if tape.live:
            obs, rew, done, _ = ref.step(actions)
        env.step((np.repeat(a_act[None], 2, axis=0), np.repeat(p_act[None], 2, axis=0) if p_act.size else None))
        want_rew = np.array([rew[str(i)] for i in range(A)] + [rew["p"]]) if tape.live else None
        tape.close("rew", want_rew, s.to_numpy(s.buf["reward"])[1], rtol=1e-6, atol=1e-9, where="t=%d rewards" % t)
        ended = bool(int(s.to_numpy(s.buf["done"])[1]))
        tape.equal("done", bool(done["__all__"]) if tape.live else None, ended, "t=%d" % t)
        if ended:
            m_ref = None
            if tape.live:
                with np.errstate(all="ignore"):
                    m_ref = ref.metrics
                obs = ref.reset()
            with np.errstate(all="ignore"):
                ref_tape.same_metrics(tape, "finished episode", m_ref, env.previous_episode_metrics_of(1), "t=%d" % t)
        compare(tape, reference_arrays(ref, obs) if tape.live else None, s, 1, "t=%d" % t)
    tape.finish()


if __name__ == "__main__":
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 30
    rng = np.random.RandomState(int(sys.argv[2]) if len(sys.argv) > 2 else 0)
    bad = 0
    for i in range(n):
        cfg = random_config(rng)
        try:
            run_one(cfg, seed=300 + i)
        except Exception as ex:  # noqa: BLE001
            bad += 1
            print("[%d] FAILED %r\n    %s" % (i, cfg, "".join(traceback.format_exception_only(type(ex), ex)).strip()[:600]))
    print("%d configs x 4 episodes, %d failures" % (n, bad))
