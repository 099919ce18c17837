"""flatten_observations=False / flatten_masks=False (the setting of the reference's basic and advanced tutorials and of
tests/test_env.py): named observation fields and per-subspace masks as slices of the flat device tensors."""
import numpy as np
import pytest

from ai_economist_b200 import foundation
from oracle import ref_harness as rh
from oracle import ref_tape
from oracle.configs import CONFIGS
from tests.emu.emu_stepper import emu_factory


def _product(cfg, **over):
    kw = dict(CONFIGS[cfg])
    kw.update(over)
    name = kw.pop("scenario_name")
    return foundation.make_env_instance(name, n_envs=2, stepper_factory=emu_factory, auto_reset=False, **kw)


@pytest.mark.parametrize("cfg", ["c1_tutorial", "c3_short_period", "tax_us_federal", "full_obs_tax"])
def test_named_fields_are_slices_of_the_flat_vectors(cfg):
    flat = _product(cfg)
    named = _product(cfg, flatten_observations=False, flatten_masks=False)
    for env in (flat, named):
        env.seed(3)
        env.reset()
        env.step(None)
    st = named.stepper
    for which, key, buf in (("agent", "0", "obs_agent_flat"), ("planner", "p", "obs_planner_flat")):
        lay = st.flat_layout(which)
        assert [k for k, _, _ in lay] == sorted(k for k, _, _ in lay)            # sorted-key concatenation
        assert sum(n for _, _, n in lay) == st.buf[buf].shape[-1]               # ... covering the whole vector
        for k, off, n in lay:
            if k == "time":
                continue
            got = np.asarray(named.obs[key][k])
            want = np.asarray(flat.obs[key]["flat"])[..., off:off + n]
            assert np.array_equal(got.reshape(want.shape), want), k
            assert np.shares_memory(got, st.buf[buf])                           # a view, not a copy
    assert "flat" not in named.obs["0"] and "flat" not in named.obs["p"]
    assert isinstance(named.obs["p"]["p0"], dict) and isinstance(named.obs["0"]["action_mask"], dict)
    # per-subspace masks: the flat mask minus its NO-OP entries, in registration order
    ag = named.get_agent(0)
    m = named.obs["0"]["action_mask"]
    assert [k for k in m if np.asarray(m[k]).shape[-1]] == list(ag._action_names)   # (+ the reference's empty entries)
    total = sum(np.asarray(v).shape[-1] for v in m.values())
    n_noop = len(ag._action_names) if ag.multi_action_mode else 1
    assert total + n_noop == np.asarray(flat.obs["0"]["action_mask"]).shape[-1]


@pytest.mark.parametrize("cfg", ["c1_tutorial", "c3_short_period", "tax_us_federal", "full_obs_tax"])
def test_unflattened_observations_match_live_reference(cfg):
    """The named fields and per-subspace masks against the reference's (its values as recorded, oracle/ref_tape.py)."""
    tape = ref_tape.Tape("unflattened_views", cfg)
    ref_obs = None
    if tape.live:
        f = rh.load_reference_foundation()
        kw = dict(CONFIGS[cfg])
        kw.update(flatten_observations=False, flatten_masks=False)
        ref = f.make_env_instance(**kw)
        ref.seed(21)
        ref_obs = ref.reset()
    env = _product(cfg, flatten_observations=False, flatten_masks=False)
    env.seed([21, 22])
    obs = env.reset()
    rng = np.random.RandomState(4)

    def compare(ro, po, key, label):
        tape.equal(key + "/", sorted(ro) if tape.live else None, sorted(po), label)
        for k in sorted(po):
            if isinstance(po[k], dict) or (tape.live and isinstance(ro[k], dict)):
                compare(ro[k] if tape.live else None, po[k], key + "/" + k, label)
                continue
            got = np.asarray(po[k])[0]
            want = np.asarray(ro[k], dtype=np.float64).reshape(got.shape) if tape.live else None
            tape.close(key + "/" + k, want, got, rtol=1e-6, atol=1e-7, where=label)

    for t in range(25):
        tape.equal("agents", sorted(ref_obs) if tape.live else None, sorted(obs), "t=%d" % t)
        for idx in sorted(obs):
            compare(ref_obs[idx] if tape.live else None, obs[idx], idx, "t=%d agent %s" % (t, idx))
        actions, a_act, p_act = {}, [], None
        for i in range(env.n_agents):          # a random unmasked action per agent, from the mask dict
            ag = env.get_agent(i)
            mask = {n: np.asarray(obs[str(i)]["action_mask"][n], float)[0] for n in ag._action_names}
            if ag.multi_action_mode:
                row = [int(rng.choice(len(m) + 1, p=np.r_[1, m] / (1 + np.sum(m)))) for m in (mask[n] for n in ag._action_names)]
                actions[str(i)] = row
            else:
                flat_m = np.r_[1.0, np.concatenate([mask[n] for n in ag._action_names])]
                row = [int(rng.choice(len(flat_m), p=flat_m / flat_m.sum()))]
                actions[str(i)] = row[0]
            a_act.append(row)
        if tape.live:
            ref_obs, _, _, _ = ref.step(actions)
        aa = np.asarray(a_act, np.int32)[None].repeat(2, axis=0)
        obs, _, _, _ = env.step((aa, None))
    tape.finish()
