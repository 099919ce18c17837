"""TEST INFRASTRUCTURE ONLY — imports the *unmodified* reference from /root/reference.

Used (a) to validate the C restatement in oracle/ and (b) to generate the golden
fixtures committed under tests/golden/ (including the recorded digests of
oracle/ref_tape.py).  The reference is not part of the repository, so nothing under
`-m gpu`, smoke() or bench.py may load it (load_reference_foundation).

Recipe follows SURVEY.md Appendix C: stub the absent third-party modules the
reference imports at module scope (lz4, Crypto, GPUtil), restore `np.int`.
"""
import os
import sys
import types

import numpy as np

REFERENCE_ROOT = os.environ.get("AIE_REFERENCE_ROOT", "/root/reference")


def reference_available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "ai_economist"))


_foundation = None


def load_reference_foundation():
    """Import `ai_economist.foundation` from the read-only reference tree."""
    global _foundation
    if _foundation is not None:
        return _foundation
    if not reference_available():
        raise RuntimeError("reference tree not present at %s" % REFERENCE_ROOT)
    for name in ["lz4", "lz4.frame", "Crypto", "Crypto.PublicKey",
                 "Crypto.PublicKey.RSA", "GPUtil"]:
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["lz4"].frame = sys.modules["lz4.frame"]
    sys.modules["Crypto"].PublicKey = sys.modules["Crypto.PublicKey"]
    sys.modules["Crypto.PublicKey"].RSA = sys.modules["Crypto.PublicKey.RSA"]
    sys.modules["GPUtil"].getAvailable = lambda *a, **k: []
    if not hasattr(np, "int"):
        np.int = int  # layout_from_file.py:212-213 uses the removed alias
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    from ai_economist import foundation  # noqa: E402

    mod = sys.modules.get("ai_economist.foundation.scenarios.covid19.covid19_env")
    if mod is not None:
        mod.verify_activation_code = lambda: None
    _foundation = foundation
    return foundation


# --------------------------------------------------------------------------- #
# Converters: reference env object  ->  plain arrays in the oracle/product layout
# --------------------------------------------------------------------------- #

COMPONENT_NAMES = ["Build", "ContinuousDoubleAuction", "Gather", "PeriodicBracketTax", "WealthRedistribution"]


def spec_from_reference_env(env):
    """Read a flat config dict (the oracle's orc_config fields) off a constructed reference env."""
    comps = [c.name for c in env._components]
    for c in comps:
        assert c in COMPONENT_NAMES, "component %s is outside the hot-path scope" % c
    spec = dict(
        components=comps,
        n_agents=env.n_agents, height=env.world_size[0], width=env.world_size[1],
        episode_length=env.episode_length,
        multi_action_agents=int(env.multi_action_mode_agents),
        has_water=int("Water" in env.world.maps.keys()),
        obs_range=env._mobile_agent_observation_range,
        planner_gets_spatial_info=int(env._planner_gets_spatial_info),
        allow_observation_scaling=int(env._allow_observation_scaling),
        regen_weight=[env.layout_specs["Stone"]["regen_weight"], env.layout_specs["Wood"]["regen_weight"]],
        isoelastic_eta=env.isoelastic_eta, energy_cost=env.energy_cost,
        energy_warmup_constant=env.energy_warmup_constant,
        energy_warmup_auto=int(env.energy_warmup_method == "auto"),
        planner_reward_type={"coin_eq_times_productivity": 0, "inv_income_weighted_coin_endowments": 1,
                             "inv_income_weighted_utility": 2}[env.planner_reward_type],
        mixing_weight_gini_vs_coin=env.mixing_weight_gini_vs_coin,
        build_payment=10.0, build_labor=10.0, move_labor=1.0, collect_labor=1.0,
        max_bid_ask=10, order_duration=50, max_num_orders=50, order_labor=0.25,
        tax_model=0, disable_taxes=0, period=100, n_brackets=0, n_disc_rates=0,
        bracket_cutoffs=[], disc_rates=[], fixed_rates=[],
        tax_annealing=0, annealing_warmup=0.0, annealing_slope=0.0, rate_max=1.0,
    )
    for r in ("Stone", "Wood"):
        assert env.layout_specs[r]["max_health"] == 1
    hw = [int(env.layout_specs[r]["regen_halfwidth"]) for r in ("Stone", "Wood")]
    if any(hw):
        spec["regen_halfwidth"] = hw
    if not env.multi_action_mode_planner:
        spec["single_action_planner"] = 1
    if env._full_observability:
        spec["full_observability"] = 1
    for c in env._components:
        if c.name == "Build":
            spec.update(build_payment=float(c.payment), build_labor=c.build_labor)
        elif c.name == "Gather":
            spec.update(move_labor=c.move_labor, collect_labor=c.collect_labor)
        elif c.name == "ContinuousDoubleAuction":
            spec.update(max_bid_ask=c.max_bid_ask, order_duration=c.order_duration,
                        max_num_orders=c.max_num_orders, order_labor=c.order_labor)
        elif c.name == "PeriodicBracketTax":
            assert c.tax_model in ("model_wrapper", "us-federal-single-filer-2018-scaled", "fixed-bracket-rates", "saez")
            spec.update(
                tax_model={"model_wrapper": 0, "saez": 2}.get(c.tax_model, 1), rate_min=float(c.rate_min),
                disable_taxes=int(c.disable_taxes), period=c.period, n_brackets=c.n_brackets,
                n_disc_rates=c.n_disc_rates, bracket_cutoffs=[float(x) for x in c.bracket_cutoffs],
                disc_rates=[] if c.disc_rates is None else [float(x) for x in c.disc_rates],
                # fixed schedules: the schedule clipped by rate_max; a tax_annealing_schedule clips it further per episode
                fixed_rates=([0.0] * c.n_brackets if c.tax_model in ("model_wrapper", "saez") else
                             [float(x) for x in np.minimum(np.array(c.us_federal_single_filer_2018_scaled
                                                                    if c.tax_model == "us-federal-single-filer-2018-scaled"
                                                                    else c.fixed_bracket_rates), c.rate_max)]),
                tax_annealing=int(c.tax_annealing_schedule is not None),
                annealing_warmup=float(c._annealing_warmup or 0.0),
                annealing_slope=float(c._annealing_slope or 0.0), rate_max=float(c.rate_max),
            )
    return spec


def state_from_reference_env(env):
    """Post-reset host snapshot (call right after env.reset())."""
    maps = env.world.maps
    A = env.n_agents
    H, W = env.world_size
    water = maps.get("Water") if "Water" in maps.keys() else np.zeros((H, W))
    key = np.random.get_state()
    st = dict(
        stone=(maps.get("Stone") > 0).astype(np.uint8), wood=(maps.get("Wood") > 0).astype(np.uint8),
        stone_src=(maps.get("StoneSourceBlock") > 0).astype(np.uint8),
        wood_src=(maps.get("WoodSourceBlock") > 0).astype(np.uint8),
        water=(water > 0).astype(np.uint8),
        loc=np.array([[int(a.loc[0]), int(a.loc[1])] for a in env.world.agents], np.int16),
        coin=np.array([a.state["inventory"]["Coin"] for a in env.world.agents], np.float64),
        inv_stone=np.array([a.state["inventory"]["Stone"] for a in env.world.agents], np.int32),
        inv_wood=np.array([a.state["inventory"]["Wood"] for a in env.world.agents], np.int32),
        build_payment=np.array([a.state.get("build_payment", 0.0) for a in env.world.agents], np.float64),
        build_skill=np.array([a.state.get("build_skill", 0.0) for a in env.world.agents], np.float64),
        bonus_gather_prob=np.array([a.state.get("bonus_gather_prob", 0.0) for a in env.world.agents], np.float64),
        mt_key=np.array(key[1], np.uint32), mt_pos=int(key[2]),
        completions=int(env._completions),
    )
    if "Build" in env._components_dict:
        bm = env.get_component("Build")
        st["build_skill"] = np.array([bm.sampled_skills[i] for i in range(A)], np.float64)
    assert np.all(maps.get("House") == 0)
    return st


def obs_arrays_from_reference(env, obs, rew=None, done=None):
    """Reference obs dict (flatten_observations=True, flatten_masks=True) -> oracle-layout arrays."""
    A = env.n_agents
    out = dict(
        a_map=np.stack([obs[str(i)]["world-map"] for i in range(A)]).astype(np.float32),
        a_idx=np.stack([obs[str(i)]["world-idx_map"] for i in range(A)]).astype(np.int16),
        a_flat=np.stack([obs[str(i)]["flat"] for i in range(A)]).astype(np.float32),
        a_mask=np.stack([obs[str(i)]["action_mask"] for i in range(A)]).astype(np.float32),
        p_flat=np.asarray(obs["p"]["flat"], np.float32),
        p_agents=(np.stack([obs["p"]["p%d" % i] for i in range(A)]).astype(np.float32) if "p0" in obs["p"]
                  else np.zeros((A, 0), np.float32)),   # full_observability without a tax component: no p<i> at all
        p_mask=np.asarray(obs["p"]["action_mask"], np.float32),
        time=np.asarray(obs["p"]["time"], np.float32),
    )
    if "world-map" in obs["p"]:
        out["p_map"] = np.asarray(obs["p"]["world-map"], np.float32)
        out["p_idx"] = np.asarray(obs["p"]["world-idx_map"], np.int16)
    if rew is not None:
        out["rew"] = np.array([rew[str(i)] for i in range(A)] + [rew["p"]], np.float64)
    if done is not None:
        out["done"] = np.array([int(done["__all__"])], np.int32)
    return out


def state_arrays_from_reference(env):
    """Full mid-episode state of the reference env in the oracle's orc_get_state layout."""
    maps = env.world.maps
    A = env.n_agents
    H, W = env.world_size
    water = maps.get("Water") if "Water" in maps.keys() else np.zeros((H, W))
    cell = ((maps.get("Stone") > 0).astype(np.uint8) | ((maps.get("Wood") > 0).astype(np.uint8) << 1)
            | ((maps.get("StoneSourceBlock") > 0).astype(np.uint8) << 2)
            | ((maps.get("WoodSourceBlock") > 0).astype(np.uint8) << 3)
            | ((water > 0).astype(np.uint8) << 4) | ((maps.get("House") > 0).astype(np.uint8) << 5))
    ag = env.world.agents
    key = np.random.get_state()
    out = dict(
        cell=cell, owner=maps.get("House", owner=True).astype(np.int8),
        loc=np.array([[int(a.loc[0]), int(a.loc[1])] for a in ag], np.int16),
        coin=np.array([a.state["inventory"]["Coin"] for a in ag], np.float64),
        esc_coin=np.array([a.state["escrow"]["Coin"] for a in ag], np.float64),
        labor=np.array([a.state["endogenous"]["Labor"] for a in ag], np.float64),
        inv=np.array([[a.state["inventory"]["Stone"], a.state["inventory"]["Wood"]] for a in ag], np.int32),
        esc=np.array([[a.state["escrow"]["Stone"], a.state["escrow"]["Wood"]] for a in ag], np.int32),
        mt_key=np.array(key[1], np.uint32), mt_pos=np.array([key[2]], np.int32),
        t=np.array([env.world.timestep], np.int32),
    )
    if "ContinuousDoubleAuction" in env._components_dict:
        c = env.get_component("ContinuousDoubleAuction")
        out["n_orders"] = np.array([[c.n_orders[r][i] for i in range(A)] for r in c.commodities], np.int32)
        out["bid_hist"] = np.array([[c.bid_hists[r][i] for i in range(A)] for r in c.commodities]).astype(np.int32)
        out["ask_hist"] = np.array([[c.ask_hists[r][i] for i in range(A)] for r in c.commodities]).astype(np.int32)
        out["price_hist"] = np.array([[c.price_history[r][i] for i in range(A)] for r in c.commodities], np.float64)
        out["book"] = {
            (ci, 0): np.array([[b["buyer"], b["bid"], b["bid_lifetime"]] for b in c.bids[r]], np.int32).reshape(-1, 3)
            for ci, r in enumerate(c.commodities)}
        out["book"].update({
            (ci, 1): np.array([[a["seller"], a["ask"], a["ask_lifetime"]] for a in c.asks[r]], np.int32).reshape(-1, 3)
            for ci, r in enumerate(c.commodities)})
    if "PeriodicBracketTax" in env._components_dict:
        t = env.get_component("PeriodicBracketTax")
        out["tax_pos"] = np.array([t.tax_cycle_pos], np.int32)
        out["rate_idx"] = np.array(t.curr_rate_indices, np.int32)
        out["last_coin"] = np.array(t.last_coin, np.float64)
        out["last_income"] = np.array(t.last_income, np.float64)
        out["last_marg"] = np.array(t.last_marginal_rate, np.float64)
    return out


def sample_actions(env, obs, rng):
    """Uniform over unmasked actions (tutorial semantics), drawn from a *separate* RandomState so the
    env's own global-stream tape is not perturbed.  Returns (reference action dict, a_act [A,n], p_act [B])."""
    A = env.n_agents
    actions = {}
    a_rows = []
    for i in range(A):
        mask = np.asarray(obs[str(i)]["action_mask"])
        ag = env.get_agent(i)
        if ag.multi_action_mode:
            dims = [ag.action_dim[k] for k in ag._action_names]
            row, off = [], 0
            for d in dims:
                m = mask[off:off + d]
                p = m / m.sum()
                row.append(int(rng.choice(d, p=p)))
                off += d
            actions[str(i)] = row
            a_rows.append(row)
        else:
            p = mask / mask.sum()
            a = int(rng.choice(len(mask), p=p))
            actions[str(i)] = a
            a_rows.append([a])
    pl = env.get_agent("p")
    pmask = np.asarray(obs["p"]["action_mask"])
    p_row = []
    if len(pmask) > 1 and not pl.multi_action_mode:   # one index over [NO-OP] ++ every bracket's rates
        p_row = [int(rng.choice(len(pmask), p=pmask / pmask.sum()))]
        actions["p"] = p_row[0]
    elif len(pmask) > 1:
        dims = [pl.action_dim[k] for k in pl._action_names]
        off = 0
        for d in dims:
            m = pmask[off:off + d]
            p_row.append(int(rng.choice(d, p=m / m.sum())))
            off += d
        actions["p"] = p_row
    return actions, np.array(a_rows, np.int32), np.array(p_row, np.int32)


def sample_actions_from_masks(env, a_mask, p_mask, rng):
    """sample_actions on masks held as arrays (a_mask [A, L], p_mask [L]) with the agents of a product env: the same
    draws as sample_actions on the reference's observation wherever the masks are equal."""
    obs = {str(i): {"action_mask": np.asarray(a_mask[i])} for i in range(env.n_agents)}
    obs["p"] = {"action_mask": np.asarray(p_mask).reshape(-1)}
    return sample_actions(env, obs, rng)
