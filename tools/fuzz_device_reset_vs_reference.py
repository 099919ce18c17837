"""Randomised multi-episode fuzz (build container only): the device-side reference-exact reset (auto_reset, 1-lane
emulation of the device source) against the LIVE reference, which calls env.reset() between episodes on one continuing
global numpy stream.  layout_from_file configurations with skill_dist in {none, pareto, lognormal}, with / without
fixed_four_skill_and_loc; with --dynamic: uniform / quadrant scenarios (device-side layout generation); with --saez: the Saez
tax model (device / host hybrid, foundation/saez.py) over enough episodes to fill its 500-sample buffer and run the formula,
with and without a tax_annealing_schedule.
python tools/fuzz_device_reset_vs_reference.py [n] [seed] [--dynamic | --multi-zone | --saez]"""
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

LAYOUTS = {(15, 15): "env-pure_and_mixed-15x15.txt", (25, 25): "quadrant_25x25_20each_30clump.txt",
           (40, 40): "quadrant_40x40_50each.txt"}


def random_config(rng):
    size = list(LAYOUTS)[rng.randint(len(LAYOUTS))]
    fixed_four = bool(rng.rand() < 0.4)
    A = int(rng.choice([2, 3, 4, 6, 9, 12]))
    comps = [("Build", dict(skill_dist="pareto" if fixed_four else str(rng.choice(["none", "pareto", "lognormal"], p=[0.2, 0.6, 0.2])),
                            payment_max_skill_multiplier=int(rng.randint(1, 4)))),
             ("ContinuousDoubleAuction", dict(max_num_orders=int(rng.choice([1, 3, 5])), order_duration=int(rng.choice([2, 50])))),
             ("Gather", dict(skill_dist=str(rng.choice(["none", "pareto", "lognormal"]))))]
    if rng.rand() < 0.5:
        tkw = dict(period=int(rng.choice([3, 10])), bracket_spacing="us-federal",
                   tax_model=str(rng.choice(["model_wrapper", "us-federal-single-filer-2018-scaled"])))
        if rng.rand() < 0.6:
            tkw["tax_annealing_schedule"] = [int(rng.choice([-2, 0, 1])), float(rng.choice([0.25, 0.5]))]
        comps.append(("PeriodicBracketTax", tkw))
    split = (not fixed_four) and comps[0][1]["skill_dist"] == "pareto" and rng.rand() < 0.7
    if split:   # split_layout: constructor-time skill table (needs a constructor seed), ranks above the water row
        n_top = int(rng.randint(1, A))
        extra = dict(seed=int(rng.randint(1, 1000)), skill_rank_of_top_agents=[int(x) for x in rng.choice(A, n_top, replace=False)])
        return dict(scenario_name="split_layout/simple_wood_and_stone", components=comps, n_agents=A,
                    world_size=list(size), env_layout_file=LAYOUTS[size], episode_length=int(rng.choice([8, 15])),
                    starting_agent_coin=float(rng.choice([0, 10])), multi_action_mode_agents=bool(rng.rand() < 0.3),
                    multi_action_mode_planner=True, flatten_observations=True, flatten_masks=True, **extra)
    return dict(scenario_name="layout_from_file/simple_wood_and_stone", components=comps, n_agents=A,
                world_size=list(size), env_layout_file=LAYOUTS[size], episode_length=int(rng.choice([8, 15, 30])),
                fixed_four_skill_and_loc=fixed_four, starting_agent_coin=float(rng.choice([0, 10])),
                multi_action_mode_agents=bool(rng.rand() < 0.3), multi_action_mode_planner=True,
                flatten_observations=True, flatten_masks=True,
                energy_warmup_constant=float(rng.choice([0, 4])), energy_warmup_method="decay")


FAMILIES = ["uniform", "quadrant"]   # tests/test_fuzz_subsets.py: the multi_zone subset sets ["multi_zone"]


def random_dynamic_config(rng):
    """uniform/... and quadrant/... : every reset generates a new clumped layout on the device (dynamic_layout.py:313-429)."""
    fam = str(rng.choice(FAMILIES))
    H = int(rng.randint(9, 27)); W = H if fam == "quadrant" else int(rng.randint(9, 27))
    A = int(rng.choice([2, 3, 5, 8]))
    comps = [("Build", dict(skill_dist=str(rng.choice(["none", "pareto", "lognormal"])), payment_max_skill_multiplier=int(rng.randint(1, 4)))),
             ("ContinuousDoubleAuction", dict(max_num_orders=int(rng.choice([1, 5])))),
             ("Gather", dict(skill_dist=str(rng.choice(["none", "pareto", "lognormal"]))))]
    return dict(scenario_name=fam + "/simple_wood_and_stone", components=comps, n_agents=A, world_size=[H, W],
                episode_length=int(rng.choice([6, 12])), starting_agent_coin=float(rng.choice([0, 10])),
                multi_action_mode_agents=bool(rng.rand() < 0.3), multi_action_mode_planner=True,
                flatten_observations=True, flatten_masks=True,
                starting_wood_coverage=float(rng.choice([0.05, 0.1, 0.15])), starting_stone_coverage=float(rng.choice([0.05, 0.1])),
                wood_clumpiness=float(rng.choice([0.0, 0.35, 0.8])), stone_clumpiness=float(rng.choice([0.2, 0.5, 1.0])),
                gradient_steepness=float(rng.choice([1, 4, 8])), checker_source_blocks=bool(rng.rand() < 0.3),
                wood_regen_weight=float(rng.choice([0.05, 0.5])), stone_regen_weight=float(rng.choice([0.05, 0.5])),
                **(dict(num_partitions_row=int(rng.choice([3, 4])), num_partitions_col=int(rng.choice([2, 3, 5])),   # >= 6 regions >= 5 zones
                        num_wood_zones=int(rng.choice([1, 2])), num_stone_zones=int(rng.choice([1, 2])),
                        num_wood_and_stone_zones=int(rng.choice([0, 1]))) if fam == "multi_zone" else {}))


def random_saez_config(rng):
    """PeriodicBracketTax(tax_model="saez") (redistribution.py:437-823): warm-up draws, sample buffer, elasticity regression,
    binned welfare weights, bracketisation, running average across resets - and curr_rate_max under annealing."""
    size = list(LAYOUTS)[rng.randint(len(LAYOUTS))]
    A = int(rng.choice([5, 8, 10, 12]))
    spacing = str(rng.choice(["us-federal", "linear", "log"]))
    tkw = dict(tax_model="saez", period=int(rng.choice([2, 5])), bracket_spacing=spacing,
               usd_scaling=float(rng.choice([1000.0, 10000.0])), pareto_weight_type=str(rng.choice(["inverse_income", "uniform"])),
               rate_min=float(rng.choice([0.0, 0.1])), rate_max=float(rng.choice([1.0, 0.8])))
    if spacing != "us-federal":
        tkw.update(n_brackets=int(rng.choice([3, 5, 7])), top_bracket_cutoff=float(rng.choice([20, 100])))
    if rng.rand() < 0.3:
        tkw["saez_fixed_elas"] = float(rng.choice([0.0, 0.4, 1.0]))
    if rng.rand() < 0.6:
        tkw["tax_annealing_schedule"] = [int(rng.choice([-2, 0, 1])), float(rng.choice([0.15, 0.3, 0.6]))]
    comps = [("Build", dict(skill_dist="pareto", payment_max_skill_multiplier=int(rng.randint(1, 4)))),
             ("ContinuousDoubleAuction", dict(max_num_orders=int(rng.choice([1, 3, 5])), order_duration=int(rng.choice([2, 50])))),
             ("Gather", dict(skill_dist=str(rng.choice(["none", "pareto"])))), ("PeriodicBracketTax", tkw)]
    return dict(scenario_name="layout_from_file/simple_wood_and_stone", components=comps, n_agents=A,
                world_size=list(size), env_layout_file=LAYOUTS[size], episode_length=int(rng.choice([40, 60])),
                fixed_four_skill_and_loc=False, starting_agent_coin=float(rng.choice([5, 20])),
                multi_action_mode_agents=bool(rng.rand() < 0.3), multi_action_mode_planner=True,
                flatten_observations=True, flatten_masks=True)


def saez_episodes(cfg):
    """episodes until the 500-sample buffer has been full for at least two more episodes (one tax day = n_agents samples)"""
    tax = [kw for name, kw in cfg["components"] if name == "PeriodicBracketTax"][0]
    per_episode = (cfg["episode_length"] // tax["period"]) * cfg["n_agents"]
    return -(-500 // per_episode) + 2


def run_one(cfg, seed, episodes=4, tape=None):
    """tape (oracle/ref_tape.py): None compares with the live reference, a replaying tape with its recorded digests.
    The actions are drawn from the product's masks (equal to the reference's, which every check compares)."""
    tape = tape or ref_tape.Tape()
    if tape.live:
        f = rh.load_reference_foundation()
        ref = f.make_env_instance(**cfg)
        ref.seed(seed)
        obs = ref.reset()
    kw = dict(cfg)
    name = kw.pop("scenario_name")
    if "seed" in kw:
        kw["seeds"] = [kw.pop("seed")] * 2
    env = foundation.make_env_instance(name, n_envs=2, stepper_factory=emu_factory, auto_reset=True, **kw)
    assert env.spec["reset_mode"] == 1
    env.seed([seed, seed])
    env.reset()
    s = env.stepper
    arng = np.random.RandomState(seed + 1)
    T = cfg["episode_length"]

    def compare(label):
        ro = rs = {}
        if tape.live:
            ro = rh.obs_arrays_from_reference(ref, obs)
            rs = rh.state_arrays_from_reference(ref)
        po, ps = s.read_obs(1), s.read_state(1)
        for k in tape.keys("state", ["cell", "owner", "loc", "inv", "esc", "mt_key", "mt_pos", "n_orders"], rs):
            tape.equal(k, rs.get(k), ps[k], label + ": state")
        for k in ["coin", "labor"]:
            tape.close(k, rs.get(k), ps[k], rtol=1e-9, atol=1e-9, where=label + ": state")
        for k in ["a_map", "a_idx", "a_mask", "p_mask"]:
            tape.equal(k, ro.get(k), po[k], label + ": obs")
        for k in ["a_flat", "p_flat", "p_agents"]:
            tape.close(k, ro.get(k), po[k], rtol=1e-6, atol=1e-7, where=label + ": obs")

    compare("reset")
    for t in range(1, episodes * T + 1):
        po = s.read_obs(1)
        actions, a_act, p_act = rh.sample_actions_from_masks(env, po["a_mask"], po["p_mask"], arng)
        if tape.live:
            obs, rew, done, _ = ref.step(actions)
        env.step((np.repeat(a_act[None], 2, axis=0), np.repeat(p_act[None], 2, axis=0) if p_act.size else None))
        got_rew = s.to_numpy(s.buf["reward"])[1]
        want_rew = np.array([rew[str(i)] for i in range(ref.n_agents)] + [rew["p"]]) if tape.live else None
        tape.close("rew", want_rew, got_rew, rtol=1e-6, atol=1e-9, where="t=%d rewards" % t)
        ended = bool(int(s.to_numpy(s.buf["done"])[1]))
        tape.equal("done", bool(done["__all__"]) if tape.live else None, ended, "t=%d" % t)
        if ended:
            if tape.live:
                obs = ref.reset()
            with np.errstate(all="ignore"):   # the finished episode's metrics: _finalize_logs vs the device's end-of-episode snapshot
                p1 = ref.previous_episode_metrics if tape.live else None
                ref_tape.same_metrics(tape, "previous metrics", p1, env.previous_episode_metrics_of(1), "t=%d" % t)
        compare("t=%d%s" % (t, " (after reset)" if ended else ""))
    tape.finish()


if __name__ == "__main__":
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    n = int(args[0]) if len(args) > 0 else 30
    rng = np.random.RandomState(int(args[1]) if len(args) > 1 else 0)
    bad, kinds = 0, {}
    dynamic = "--dynamic" in sys.argv or "--multi-zone" in sys.argv
    saez = "--saez" in sys.argv
    if "--multi-zone" in sys.argv:
        FAMILIES[:] = ["multi_zone"]
    for i in range(n):
        cfg = (random_saez_config if saez else random_dynamic_config if dynamic else random_config)(rng)
        kind = "saez" + ("+annealing" if "tax_annealing_schedule" in cfg["components"][-1][1] else "") if saez else cfg["scenario_name"].split("/")[0]
        kinds[kind] = kinds.get(kind, 0) + 1
        try:
            run_one(cfg, seed=500 + i, **(dict(episodes=saez_episodes(cfg)) if saez else {}))
        except Exception as ex:  # noqa: BLE001
            bad += 1
            print("[%d] FAILED %r\n    %s" % (i, cfg, "".join(traceback.format_exception_only(type(ex), ex)).strip()[:500]))
    print("%d configs x %s episodes, %d failures" % (n, "enough" if saez else "4", bad), kinds)
