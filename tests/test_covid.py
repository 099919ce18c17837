"""COVID-19 + economy scenario (BASELINE config 4).

CPU: (1) the host-side parameter derivation against constants read off the reference (when present);
(2) oracle/covid_oracle.py (numpy restatement) against the golden trace recorded from the unmodified reference;
(3) the device source compiled for the host (tests/emu) against the same trace.
GPU: the CUDA kernel through the C-ABI against the golden trace and against the numpy oracle on batches.

Tolerance: float32 fields <= 1e-6 relative (atol 1e-9); masks / integer state exact.  In practice all float32
observations are bit-identical; the tolerance covers powf/exp/log ulp differences between device and glibc.
"""
import json
import os

import numpy as np
import pytest

from ai_economist_b200.foundation.covid19 import build_covid_params
from oracle.covid_oracle import CovidOracleEnv

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden_covid", "covid_seed3.npz")
OBS_KEYS = ["agent_state", "postsubsidy", "lagged", "policy_ind", "scalars", "mask_a", "mask_p"]
RTOL, ATOL = 1e-6, 1e-9


VARIANTS = ["covid_seed3.npz", "covid_cooldown1_seed11.npz", "covid_cooldown7_seed12.npz"]   # cooldown 28 / 1 / 7, own action seeds


def load(name=None):
    z = np.load(GOLDEN if name is None else os.path.join(os.path.dirname(GOLDEN), name))
    meta = json.loads(str(z["meta_json"]))
    return z, meta, build_covid_params(**meta["kwargs"])


def check(z, t, obs, label):
    for k in OBS_KEYS:
        assert np.allclose(z[k][t], obs[k], rtol=RTOL, atol=ATOL), "%s step %d: %s" % (label, t, k)
    assert np.array_equal(z["mask_a"][t], obs["mask_a"]) and np.array_equal(z["mask_p"][t], obs["mask_p"])
    if t > 0:
        assert np.allclose(z["rew_a"][t - 1], obs["rew_a"], rtol=RTOL, atol=ATOL), "%s step %d: rew_a" % (label, t)
        assert np.isclose(float(z["rew_p"][t - 1]), float(obs["rew_p"]), rtol=RTOL, atol=ATOL), "%s step %d: rew_p" % (label, t)
        assert int(z["done"][t - 1]) == int(obs["done"])


def replay(stepper_step, stepper_obs, z, n, label):
    check(z, 0, stepper_obs(), label)
    for t in range(1, n + 1):
        stepper_step(z["act_a"][t - 1].astype(np.int32), np.int32(z["act_p"][t - 1]))
        check(z, t, stepper_obs(), label)


@pytest.mark.parametrize("name", VARIANTS)
def test_covid_oracle_matches_reference_golden_trace(name):
    z, meta, p = load(name)
    env = CovidOracleEnv(p)
    replay(lambda a, pl: env.step(a, pl), env.obs, z, meta["n_steps"], "oracle")


def _drive(stepper, e=0):
    def step(a, pl):
        ba, bp = stepper.buf["actions_agent"], stepper.buf["actions_planner"]
        if isinstance(ba, np.ndarray):
            ba[e] = a; bp[e] = pl
        else:
            import torch
            ba[e] = torch.as_tensor(a, device=ba.device); bp[e] = int(pl)
        stepper.step()
    return step, (lambda: stepper.read_obs(e))


@pytest.mark.parametrize("name", VARIANTS)
@pytest.mark.parametrize("change_list", [False, True], ids=["scan", "change_list"])
def test_covid_emulated_device_code_matches_reference_golden_trace(change_list, name):
    from tests.emu.emu_stepper import EmuCovidStepper
    z, meta, p = load(name)
    s = EmuCovidStepper(p, 2, change_list=change_list)
    s.reset()
    step, obs = _drive(s, e=1)
    replay(step, obs, z, meta["n_steps"], "emu")
    st = s.read_state(1)
    assert np.allclose(st["susceptible"], z["st_susceptible"][-1], rtol=RTOL) and np.allclose(st["deaths"], z["st_deaths"][-1], rtol=RTOL)
    assert np.array_equal(st["stringency"], z["st_stringency"][-1])


@pytest.mark.parametrize("cooldown,steps", [(None, 130), (1, 90)], ids=["default_cooldown", "cooldown_1_overflows_the_list"])
def test_covid_emulated_change_list_equals_history_scan(cooldown, steps):
    """The O(changes) unemployment response against the O(filter_len) scan under random policies, across an auto-reset;
    with a 1-day cooldown the 32-entry lists overflow and those states fall back to scanning."""
    from tests.emu.emu_stepper import EmuCovidStepper
    from ai_economist_b200 import foundation
    from oracle.gen_golden_covid import COVID_KWARGS, reference_config
    cfg = reference_config(COVID_KWARGS)
    name = cfg.pop("scenario_name")
    cfg["episode_length"] = 60
    if cooldown is not None:
        pairs = [list(c.items())[0] if isinstance(c, dict) else tuple(c) for c in cfg["components"]]
        cfg["components"] = [(n, dict(k, action_cooldown_period=cooldown) if n == "ControlUSStateOpenCloseStatus" else k)
                             for n, k in pairs]
    envs = [foundation.make_env_instance(name, n_envs=2, auto_reset=True,
                                         stepper_factory=lambda params, n, ar, cl=cl: EmuCovidStepper(params, n, ar, change_list=cl),
                                         **cfg) for cl in (False, True)]
    a, b = envs[0].stepper, envs[1].stepper
    a.reset(); b.reset()
    rng = np.random.RandomState(5)
    for t in range(steps):
        ma, mp = a.to_numpy(a.buf["mask_agent"]), a.to_numpy(a.buf["mask_planner"])
        aa = np.argmax(ma * (rng.random_sample(ma.shape) + 1e-3), axis=1).astype(np.int32)
        ap = np.argmax(mp * (rng.random_sample(mp.shape) + 1e-3), axis=1).astype(np.int32)
        for s in (a, b):
            s.buf["actions_agent"][...] = aa
            s.buf["actions_planner"][...] = ap
            s.step()
        for e in range(2):
            oa, ob = a.read_obs(e), b.read_obs(e)
            for k in OBS_KEYS + ["rew_a"]:
                assert np.allclose(oa[k], ob[k], rtol=RTOL, atol=ATOL), (t, e, k)
            assert np.isclose(float(oa["rew_p"]), float(ob["rew_p"]), rtol=RTOL, atol=ATOL) and int(oa["done"]) == int(ob["done"])
    counts = (b.buf["changes"][:, 0, :] >> 8) & 0xFF
    assert (counts == 255).any() == (cooldown == 1), counts.max()


@pytest.mark.parametrize("change_list", [False, True], ids=["scan", "change_list"])
def test_covid_emulated_auto_reset_starts_a_fresh_episode(change_list):
    from tests.emu.emu_stepper import EmuCovidStepper
    z, meta, _ = load()
    kw = dict(meta["kwargs"], episode_length=12)
    p = build_covid_params(**kw)
    s = EmuCovidStepper(p, 1, auto_reset=True, change_list=change_list)
    s.reset()
    first = s.read_obs(0)
    step, obs = _drive(s)
    for t in range(12):
        step(np.zeros(51, np.int32), np.int32(0))
    o = obs()
    assert int(o["done"]) == 1 and s.read_state(0)["t"] == 0 and s.read_state(0)["episodes"] == 1
    for k in OBS_KEYS:
        assert np.array_equal(o[k], first[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("name", VARIANTS)
@pytest.mark.parametrize("change_list", [False, True], ids=["scan", "change_list"])
def test_covid_cuda_matches_reference_golden_trace(change_list, name):
    from ai_economist_b200.covid_stepper import CudaCovidStepper
    z, meta, p = load(name)
    s = CudaCovidStepper(p, 3, auto_reset=False, change_list=change_list)
    s.reset()
    step, obs = _drive(s, e=2)
    replay(step, obs, z, meta["n_steps"], "cuda")


@pytest.mark.gpu
@pytest.mark.parametrize("change_list", [False, True], ids=["scan", "change_list"])
def test_covid_cuda_batch_matches_numpy_oracle(change_list):
    import torch
    from ai_economist_b200.covid_stepper import CudaCovidStepper
    z, meta, p = load()
    E, steps = 12, 200
    s = CudaCovidStepper(p, E, auto_reset=False, change_list=change_list)
    s.reset()
    envs = [CovidOracleEnv(p) for _ in range(E)]
    rng = np.random.RandomState(11)
    for t in range(steps):
        ma = s.to_numpy(s.buf["mask_agent"])      # [E, 11, S]
        mp = s.to_numpy(s.buf["mask_planner"])    # [E, 21]
        aa = np.argmax(ma * (rng.random_sample(ma.shape) + 1e-3), axis=1).astype(np.int32)
        ap = np.argmax(mp * (rng.random_sample(mp.shape) + 1e-3), axis=1).astype(np.int32)
        s.buf["actions_agent"].copy_(torch.as_tensor(aa)); s.buf["actions_planner"].copy_(torch.as_tensor(ap))
        s.step()
        for e in range(E):
            envs[e].step(aa[e], ap[e])
        if (t + 1) % 50 == 0:
            for e in range(E):
                got, ref = s.read_obs(e), envs[e].obs()
                for k in OBS_KEYS + ["rew_a"]:
                    assert np.allclose(ref[k], got[k], rtol=RTOL, atol=ATOL), (t, e, k)
                assert np.isclose(float(ref["rew_p"]), float(got["rew_p"]), rtol=RTOL, atol=ATOL)


@pytest.mark.gpu
def test_covid_cuda_full_size_sample_vs_oracle_and_invariants():
    """BASELINE config 4 at full size (4 096 replicas): device random policy, a sample of replicas replayed through the
    numpy oracle with the actions the device drew, state invariants on the whole batch, run-to-run determinism."""
    import torch
    from ai_economist_b200.covid_stepper import CudaCovidStepper
    z, meta, p = load()
    E, steps = 4096, 60
    sample = list(range(0, E, 455))

    def run():
        s = CudaCovidStepper(p, E, auto_reset=False)
        s.reset()
        envs = {e: CovidOracleEnv(p) for e in sample}
        for t in range(steps):
            s.sample_random_actions(seed=900 + t)
            aa, ap = s.to_numpy(s.buf["actions_agent"]), s.to_numpy(s.buf["actions_planner"])
            ma, mp = s.to_numpy(s.buf["mask_agent"]), s.to_numpy(s.buf["mask_planner"])
            assert np.all(np.take_along_axis(ma, aa[:, None, :], axis=1) == 1.0)          # drawn actions are unmasked
            assert np.all(np.take_along_axis(mp, ap[:, None], axis=1) == 1.0)
            s.step()
            for e in sample:
                envs[e].step(aa[e], ap[e])
        for e in sample:
            got, ref = s.read_obs(e), envs[e].obs()
            for k in OBS_KEYS + ["rew_a"]:
                assert np.allclose(ref[k], got[k], rtol=RTOL, atol=ATOL), (e, k)
        return s

    s = run()
    st = s.to_numpy(s.buf["state"])                      # [E, 9, S]
    assert np.isfinite(st).all() and (st[:, :6] >= 0).all()                                   # S, I, R, D, V, U >= 0
    assert (st[:, 6] >= 1).all() and (st[:, 6] <= p["num_stringency_levels"]).all()           # stringency level in range
    pop = np.asarray(p["population"], np.float64)[None]
    assert np.all(np.abs(st[:, 0] + st[:, 1] + st[:, 2] - pop) <= 1e-3 * pop)                 # S + I + R stays the population
    assert int(s.to_numpy(s.buf["hdr"])[:, 0].min()) == steps == int(s.to_numpy(s.buf["hdr"])[:, 0].max())
    s2 = run()
    assert torch.equal(s.buf["state"], s2.buf["state"]) and torch.equal(s.buf["obs_agent_state"], s2.buf["obs_agent_state"])


def test_covid_env_api_through_make_env_instance():
    """Same call as the reference (tests/run_covid19_cpu_gpu_consistency_checks.py:44-81 config)."""
    from ai_economist_b200 import foundation
    from oracle.gen_golden_covid import COVID_KWARGS, reference_config
    from tests.emu.emu_stepper import EmuCovidStepper
    z, meta, p = load()
    cfg = reference_config(COVID_KWARGS)
    name = cfg.pop("scenario_name")
    env = foundation.make_env_instance(name, n_envs=2, auto_reset=False,
                                       stepper_factory=lambda params, n, ar: EmuCovidStepper(params, n, ar), **cfg)
    assert foundation.scenarios.has("CovidAndEconomySimulation") and foundation.components.has("VaccinationCampaign")
    obs = env.reset()
    assert set(obs.keys()) == {"a", "p"}
    assert obs["a"]["world-agent_state"].shape == (2, 6, 51) and obs["a"]["action_mask"].shape == (2, 11, 51)
    assert obs["p"]["action_mask"].shape == (2, 21) and obs["a"]["time"].shape == (2, 51)
    for t in range(1, 40):
        a = np.repeat(z["act_a"][t - 1][None].astype(np.int32), 2, axis=0)
        pl = np.repeat(np.int32(z["act_p"][t - 1]), 2)
        obs, rew, done, info = env.step({"a": a, "p": pl})
        check(z, t, env.stepper.read_obs(1), "api")
    assert rew["a"].shape == (2, 51) and rew["p"].shape == (2,) and "__all__" in done


@pytest.mark.parametrize("variant", range(4))
def test_covid_observe_rate_matches_live_reference(variant):
    """VaccinationCampaign(observe_rate=True) (covid19_components.py:629-661): `next_vaccination_rate` for agents and planner is
    a function of the timestep alone; the facade serves it by table lookup after every step / reset.  Variants: deliveries from
    the start, a delivery interval that shifts the first delivery, unscaled time observations, deliveries that never begin.
    The reference's values are the ones recorded from the unmodified reference (oracle/ref_tape.py)."""
    import contextlib
    import io

    from ai_economist_b200 import foundation
    from oracle import gen_golden_covid as gg
    from oracle import ref_harness as rh
    from oracle import ref_tape
    from tests.emu.emu_stepper import EmuCovidStepper

    kw = dict(gg.COVID_KWARGS)
    kw.update(episode_length=60, start_date=["2020-03-22", "2020-12-01", "2020-12-20", "2020-06-01"][variant],
              delivery_interval=[1, 7, 3, 7][variant],
              vaccine_delivery_start_date=["2020-04-15", "2020-12-22", "2021-01-05", "2021-06-01"][variant],
              allow_observation_scaling=variant != 2)
    cfg = gg.reference_config(kw)
    for c in cfg["components"]:
        if "VaccinationCampaign" in c:
            c["VaccinationCampaign"]["observe_rate"] = True
    tape = ref_tape.Tape("covid_observe_rate", variant)
    obs = None
    if tape.live:
        f = rh.load_reference_foundation()
        with contextlib.redirect_stdout(io.StringIO()):
            ref = f.make_env_instance(**cfg)
            obs = ref.reset()
    ours = dict(cfg)
    env = foundation.make_env_instance(ours.pop("scenario_name"), n_envs=2, auto_reset=False,
                                       stepper_factory=lambda p, n, ar: EmuCovidStepper(p, n, auto_reset=ar), **ours)
    o = env.reset()
    rng, seen, key = np.random.RandomState(variant), set(), "VaccinationCampaign-next_vaccination_rate"
    for t in range(kw["episode_length"] + 1):
        tape.equal("a", np.asarray(obs["a"][key], np.float32) if tape.live else None, np.asarray(o["a"][key])[1], t)
        tape.equal("p", np.float32(obs["p"][key]) if tape.live else None, np.asarray(o["p"][key])[1], t)
        seen.add(float(np.asarray(o["p"][key])[1]))
        if t == kw["episode_length"]:
            break
        act_a, act_p = gg.sample({w: {"action_mask": np.asarray(o[w]["action_mask"])[1]} for w in ("a", "p")}, rng)
        actions = {str(i): int(act_a[i]) for i in range(51)}
        actions["p"] = int(act_p)
        if tape.live:
            obs, _, _, _ = ref.step(actions)
        o, _, _, _ = env.step((np.repeat(act_a[None], 2, 0), np.repeat(np.asarray(act_p)[None], 2, 0)))
    tape.finish()
    assert len(seen) == (1 if variant == 3 else 2)


def test_covid_observe_rate_torch_and_numpy_lookups_agree():
    """the facade's table lookup has a numpy (emulation) and a torch (CUDA buffers) branch: same values from the same scalars"""
    import torch

    from ai_economist_b200 import foundation
    from ai_economist_b200.workloads import COVID_KWARGS, covid_reference_config
    from tests.emu.emu_stepper import EmuCovidStepper

    kw = dict(COVID_KWARGS, episode_length=40, start_date="2020-12-01", delivery_interval=7, vaccine_delivery_start_date="2020-12-15")
    cfg = covid_reference_config(kw)
    for c in cfg["components"]:
        if "VaccinationCampaign" in c:
            c["VaccinationCampaign"]["observe_rate"] = True
    env = foundation.make_env_instance(cfg.pop("scenario_name"), n_envs=3, auto_reset=False,
                                       stepper_factory=lambda p, n, ar: EmuCovidStepper(p, n, auto_reset=ar), **cfg)
    env.reset()
    key = "VaccinationCampaign-next_vaccination_rate"
    want = []
    for t in range(30):
        env.step(None)
        want.append((np.array(env.obs["a"][key]), np.array(env.obs["p"][key]), np.array(env.stepper.buf["obs_scalars"])))
    # the same lookups through the torch branch: scalars as (CPU) torch tensors
    sc = torch.zeros(tuple(env.stepper.buf["obs_scalars"].shape), dtype=torch.float32)
    env._stepper.buf = dict(env._stepper.buf, obs_scalars=sc)
    env._build_rate_observation()
    for a, p, scalars in want:
        sc.copy_(torch.from_numpy(scalars))
        env._refresh_rate_observation()
        assert np.array_equal(a, env.obs["a"][key].numpy()) and np.array_equal(p, env.obs["p"][key].numpy())
    assert len({float(p[0]) for _, p, _ in want}) == 2
