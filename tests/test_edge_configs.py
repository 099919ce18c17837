"""Edge-of-range configurations (oracle/configs.py: EDGE_CONFIGS): two agents, 1x1 and wider-than-world windows, one
order slot, 32 price levels, no auction / no build component, tax every step, disabled taxes, linear / log brackets,
eta near 1, unscaled observations, a non-square world with 33 agents.

  * the C oracle and the product's host-side reset against the reference (its recorded values, oracle/ref_tape.py);
  * everywhere: the device source (1-lane emulation) against the oracle through the public API;
  * `-m gpu`: the CUDA build against the oracle, same harness (ordered last, see tests/conftest.py).
"""
import numpy as np
import pytest

from oracle import configs
from oracle import ref_harness as rh
from oracle import ref_tape

EDGE = sorted(configs.EDGE_CONFIGS)


def _all_configs():
    configs.CONFIGS.update(configs.EDGE_CONFIGS)


def make_product_env(cfg, n_envs, stepper_factory, seed, **extra):
    from ai_economist_b200 import foundation
    kw = dict(configs.EDGE_CONFIGS[cfg])
    name = kw.pop("scenario_name")
    return foundation.make_env_instance(name, n_envs=n_envs, stepper_factory=stepper_factory, auto_reset=False,
                                        seed=seed, **kw, **extra)


def run_against_oracle(env, steps, check_every):
    from oracle.oracle import OracleBatch
    from tests import batch_utils as bu
    host = env.host_reset_arrays()
    env.load_host_state(host)
    orc = OracleBatch(env.spec, env.n_envs)
    for e in range(env.n_envs):
        orc.load_env(e, {k: v[e] for k, v in host.items()})
    for e in range(env.n_envs):
        bu.compare_env(orc, env.stepper, e, "reset", spatial=bool(env.spec["planner_gets_spatial_info"]))
    bu.run_pair(env, orc, steps, np.random.RandomState(17), check_every=check_every)


@pytest.mark.parametrize("cfg", EDGE)
def test_emulated_device_code_matches_oracle_on_edge_config(cfg):
    from tests.emu.emu_stepper import emu_factory
    run_against_oracle(make_product_env(cfg, 3, emu_factory, seed=900), steps=40, check_every=10)


@pytest.mark.parametrize("cfg", EDGE)
def test_oracle_and_host_reset_track_live_reference_on_edge_config(cfg):
    from oracle.validate_vs_reference import run
    _all_configs()
    assert run(cfg, 501, 40, verbose=False, tape=ref_tape.Tape("edge_oracle", cfg))
    # the product's host-side reset: same spec, same post-reset state, same stream position
    tape = ref_tape.Tape("edge_host_reset", cfg)
    want_spec = want = {}
    if tape.live:
        f = rh.load_reference_foundation()
        ref = f.make_env_instance(**configs.EDGE_CONFIGS[cfg])
        ref.seed(77)
        ref.reset()
        want_spec, want = rh.spec_from_reference_env(ref), rh.state_from_reference_env(ref)
    env = make_product_env(cfg, 1, lambda *a, **k: None, seed=None)
    env.seed(77)
    got = env.host_reset_arrays()
    assert set(want_spec) <= set(env.spec), sorted(set(want_spec) - set(env.spec))
    for k in tape.keys("spec", [k for k in sorted(env.spec) if k != "components"], want_spec):
        tape.equal(k, want_spec.get(k), env.spec[k])
    for k in ["stone", "wood", "stone_src", "wood_src", "water", "loc", "mt_key", "coin", "build_payment",
              "build_skill", "bonus_gather_prob"]:
        tape.equal(k, want.get(k), np.asarray(got[k][0]))
    tape.equal("mt_pos", int(want["mt_pos"]) if tape.live else None, int(got["mt_pos"][0]))
    tape.finish()


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", EDGE)
def test_cuda_matches_oracle_on_edge_config(cfg):
    run_against_oracle(make_product_env(cfg, 24, None, seed=900, device="cuda:0"), steps=40, check_every=20)


def test_mean_agent_reward_sign_follows_numpys_pairwise_sum():
    """layout_from_file.py:552 / dynamic_layout.py:615: `np.mean([rew ...]) > 0` feeds the automatic energy warm-up.  In a
    step of trades only the agents' rewards cancel to rounding noise and the *order* of the sum decides the sign: numpy's
    pairwise order gives exactly 0.0 at t = 24 of this run (found by tools/fuzz_emu_vs_oracle.py 4000 1777, case 1329), a
    left-to-right sum 4.4e-17.  Device code and oracle must both take numpy's order (10 agents: the 8-accumulator path)."""
    import numpy as np
    from ai_economist_b200 import foundation
    from oracle.oracle import OracleBatch
    from tests import batch_utils as bu
    from tests.emu.emu_stepper import emu_factory

    kw = {'components': [('Build', {'skill_dist': 'lognormal', 'payment_max_skill_multiplier': 1, 'build_labor': 2.5}),
                         ('ContinuousDoubleAuction', {'max_num_orders': 2, 'order_duration': 3, 'max_bid_ask': 17, 'order_labor': 0.25}),
                         ('Gather', {'skill_dist': 'lognormal', 'move_labor': 0.5}),
                         ('PeriodicBracketTax', {'period': 10, 'tax_model': 'us-federal-single-filer-2018-scaled',
                                                 'bracket_spacing': 'us-federal'})],
          'n_agents': 10, 'episode_length': 30, 'multi_action_mode_agents': False, 'multi_action_mode_planner': True,
          'flatten_observations': True, 'flatten_masks': True, 'starting_agent_coin': 5.0, 'mobile_agent_observation_range': 2,
          'planner_gets_spatial_info': True, 'full_observability': False, 'allow_observation_scaling': True,
          'isoelastic_eta': 0.0, 'energy_cost': 1.0, 'energy_warmup_constant': 3.0, 'energy_warmup_method': 'auto',
          'planner_reward_type': 'inv_income_weighted_utility', 'mixing_weight_gini_vs_coin': 0.0, 'world_size': [24, 24],
          'starting_wood_coverage': 0.1, 'starting_stone_coverage': 0.1, 'wood_regen_weight': 0.01, 'stone_regen_weight': 0.01,
          'wood_regen_halfwidth': 0, 'stone_regen_halfwidth': 0}
    seed = 1330
    env = foundation.make_env_instance("quadrant/simple_wood_and_stone", n_envs=2, stepper_factory=emu_factory,
                                       auto_reset=False, seed=seed, **kw)
    host = env.host_reset_arrays()
    env.load_host_state(host)
    orc = OracleBatch(env.spec, 2)   # two replicas as in the fuzz run: the action sampler's stream covers both
    for e in range(2):
        orc.load_env(e, {k: v[e] for k, v in host.items()})
    st, rng = env.stepper, np.random.RandomState(seed)
    seg_a, seg_p = bu.segments(env.spec, "a"), bu.segments(env.spec, "p")
    hit = False
    for t in range(1, 31):
        aa = bu.sample_from_masks(st.to_numpy(st.buf["mask_agent"]), seg_a, rng)
        ap = bu.sample_from_masks(st.to_numpy(st.buf["mask_planner"]), seg_p, rng)
        env.step((aa, ap))
        orc.step(aa, ap)
        rew = [float(x) for x in st.to_numpy(st.buf["reward"])[0][:-1]]
        seq = 0.0
        for x in rew:
            seq += x
        hit |= (np.mean(rew) > 0) != (seq > 0)
        assert np.allclose(orc.state(0)["util_prev"], st.read_state(0)["util_prev"], rtol=1e-9, atol=1e-12), t
    assert hit, "the run no longer contains a step where the summation order decides the sign"
