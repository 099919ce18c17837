"""Seeded, bounded subsets of the randomised configuration fuzzers in tools/fuzz_*.py as collected test cases.

The fuzzers draw configurations from the whole supported option space (scenario families, component subsets and orders,
both action modes, tax models incl. annealing, WealthRedistribution, view radius, full observability, regen halfwidths,
social welfare functions, skill distributions).  Unbounded runs are a tool (`python tools/fuzz_*.py N SEED`, logs under
profiles/); here every fuzzer contributes N_CASES configurations drawn from a fixed seed, one test case each:

  * emu vs oracle            CPU, always            the device source (1-lane emulation) against the C oracle
  * cuda vs oracle           -m gpu                 the same configurations on the CUDA build (through the C-ABI)
  * oracle vs reference      CPU, always            the C oracle against the reference
  * device reset vs ref.     CPU, always            reference-exact auto-reset across 4 episodes against env.reset()
  * reference API vs ref.    CPU, always            ReferenceApiEnv against the reference: obs, rewards, metrics, dense logs
  * dynamic layouts vs ref.  CPU, always            uniform / quadrant: device-side layout generation at every auto-reset
  * one-step-economy vs ref. CPU, always            SimpleLabor + one-step-economy incl. finished-episode metrics
  * Saez hybrid vs reference CPU, always            the Saez tax model (device / host), with and without tax annealing
  * COVID vs reference       CPU, always            COVID device code (scan and change list) under parameter variants

The cases against the reference compare with its values as recorded from the unmodified reference
(tests/golden/reference_tapes/, oracle/ref_tape.py; AIE_RECORD_REFERENCE=1 records them again where the reference is
importable).  A case whose configuration the reference itself refused when it was recorded is skipped.
"""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import fuzz_emu_vs_oracle as fz  # noqa: E402
from oracle import ref_tape  # noqa: E402

N_CASES = 20


def _configs(seed, n=N_CASES, draw=None):
    rng = np.random.RandomState(seed)
    return [(draw or fz.random_config)(rng) for _ in range(n)]


def _against_reference(family, case, fn, refusals=(), when=lambda ex: True):
    """fn(tape) against the recorded reference (the live one while recording); `refusals`: exceptions by which the
    reference refuses a configuration (recorded; the case is then skipped)."""
    try:
        tape = ref_tape.Tape(family, case)
        with tape.refusals(refusals, when):
            fn(tape)
    except ref_tape.Refused as ex:
        pytest.skip("the reference refused the configuration: %s" % ex)


def _skip_unsupported(fn, *a, **k):
    """Configurations the product rejects loudly or that the reference itself cannot build
    (layout coverage asserts) are skipped, like the tools do."""
    try:
        fn(*a, **k)
    except (NotImplementedError, TimeoutError) as ex:
        pytest.skip("unsupported / unbuildable configuration: %r" % (ex,))


EMU_CASES = _configs(20260923)


@pytest.mark.parametrize("i", range(N_CASES))
def test_fuzz_emulated_device_code_matches_oracle(i):
    name, kw = EMU_CASES[i]
    _skip_unsupported(fz.run_one, name, kw, seed=1 + i, steps=60)


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(N_CASES))
def test_fuzz_cuda_matches_oracle(i):
    """GPU twin of the case above: same configurations, the CUDA build through the C-ABI (incl. the EXT kernels)."""
    from ai_economist_b200 import foundation
    from oracle.oracle import OracleBatch
    from tests import batch_utils as bu

    name, kw = EMU_CASES[i]
    E = 3
    env = foundation.make_env_instance(name, n_envs=E, device="cuda:0", auto_reset=False, seed=1 + i, **kw)
    host = env.host_reset_arrays()
    env.load_host_state(host)
    orc = OracleBatch(env.spec, E)
    for e in range(E):
        orc.load_env(e, {k: v[e] for k, v in host.items()})
    for e in range(E):
        bu.compare_env(orc, env.stepper, e, "reset", spatial=bool(env.spec["planner_gets_spatial_info"]))
    bu.run_pair(env, orc, min(60, kw["episode_length"]), np.random.RandomState(1 + i), check_every=15)


@pytest.mark.parametrize("i", range(N_CASES))
def test_fuzz_oracle_matches_live_reference(i):
    from oracle import configs
    from oracle.validate_vs_reference import run

    name, kw = _configs(5)[i]
    configs.CONFIGS["_fuzz"] = dict(kw, scenario_name=name)
    _against_reference("fuzz_oracle", i, lambda tape: run("_fuzz", 100 + i, min(60, kw["episode_length"]), verbose=False, tape=tape),
                       (AssertionError, NotImplementedError, TimeoutError))   # the reference refusing its own configuration


@pytest.mark.parametrize("i", range(N_CASES))
def test_fuzz_device_reset_matches_live_reference(i):
    import fuzz_device_reset_vs_reference as fr

    cfg = _configs(0, draw=fr.random_config)[i]
    _against_reference("fuzz_device_reset", i, lambda tape: fr.run_one(cfg, seed=500 + i, episodes=3, tape=tape))


@pytest.mark.parametrize("i", range(N_CASES))
def test_fuzz_dynamic_layout_device_reset_matches_live_reference(i):
    """uniform / quadrant: the device generates a new clumped layout at every auto-reset (rand thinning, randn + convolve2d
    growth, coverage retries, checkering, water lines) and must land on the reference's maps, placements and stream."""
    import fuzz_device_reset_vs_reference as fr

    cfg = _configs(11, draw=fr.random_dynamic_config)[i]
    _against_reference("fuzz_dynamic_layout", i, lambda tape: fr.run_one(cfg, seed=600 + i, episodes=3, tape=tape),
                       (TimeoutError,))   # the reference's own placement loop giving up on a crowded map


@pytest.mark.parametrize("i", range(10))
def test_fuzz_multi_zone_device_reset_matches_live_reference(i, monkeypatch):
    """multi_zone: np.random.shuffle of the region -> zone-type vector on the device before every layout."""
    import fuzz_device_reset_vs_reference as fr

    monkeypatch.setattr(fr, "FAMILIES", ["multi_zone"])
    cfg = _configs(21, n=10, draw=fr.random_dynamic_config)[i]
    # the reference refusing its own configuration: placement timeouts, its coverage / world asserts
    _against_reference("fuzz_multi_zone", i, lambda tape: fr.run_one(cfg, seed=650 + i, episodes=3, tape=tape),
                       (TimeoutError, AssertionError),
                       lambda ex: not isinstance(ex, AssertionError) or "coverage" in str(ex) or "World" in str(ex))


@pytest.mark.parametrize("i", range(10))
def test_fuzz_saez_hybrid_matches_live_reference(i):
    """PeriodicBracketTax(tax_model="saez"): warm-up draws on the device, buffer / regression / formula on the host, rates in
    force and observed across resets - random bracket layouts, weights, fixed elasticities, rate bounds, with and without a
    tax_annealing_schedule, over enough episodes to run the formula for two of them."""
    import fuzz_device_reset_vs_reference as fr

    cfg = _configs(31, n=10, draw=fr.random_saez_config)[i]
    _against_reference("fuzz_saez", i, lambda tape: fr.run_one(cfg, seed=800 + i, episodes=fr.saez_episodes(cfg), tape=tape))


@pytest.mark.parametrize("i", range(N_CASES))
def test_fuzz_reference_api_matches_live_reference(i):
    import fuzz_reference_api_vs_reference as fa

    name, kw = _configs(0)[i]
    _against_reference("fuzz_reference_api", i, lambda tape: fa.run_one(name, kw, seed=700 + i, tape=tape),
                       (NotImplementedError, TimeoutError))   # unsupported / unbuildable configurations


@pytest.mark.parametrize("i", range(N_CASES))
def test_fuzz_one_step_economy_matches_live_reference(i):
    """SimpleLabor + one-step-economy (components/simple_labor.py, scenarios/one_step_economy): observations, masks, rewards,
    numpy stream and finished-episode metrics across auto-resets, random reward types / tax settings / populations."""
    import fuzz_one_step_vs_reference as fo

    cfg = _configs(3, draw=fo.random_config)[i]
    _against_reference("fuzz_one_step_economy", i, lambda tape: fo.run_one(cfg, seed=300 + i, episodes=3, tape=tape))


@pytest.mark.parametrize("i", range(8))
def test_fuzz_covid_matches_live_reference(i):
    import fuzz_covid_vs_reference as fc

    kw = _configs(0, n=8, draw=fc.random_kwargs)[i]
    _against_reference("fuzz_covid", i, lambda tape: fc.run_one(kw, 900 + i, tape=tape))
