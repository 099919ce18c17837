"""adapters.ReferenceApiEnv: the reference's single-env interface over replica 0, so code written for
ai_economist.foundation runs unchanged.  The loop below is the one of tutorials/economic_simulation_basic.ipynb
(cells 11-39: env_config, sample_random_actions, play an episode with dense logging)."""
import numpy as np
import pytest

from ai_economist_b200 import foundation
from oracle import ref_harness as rh
from oracle import ref_tape
from oracle.ref_tape import same_tree
from tests.emu.emu_stepper import emu_factory

# tutorials/economic_simulation_basic.ipynb cell 11, verbatim apart from a shorter episode
ENV_CONFIG = {
    'scenario_name': 'layout_from_file/simple_wood_and_stone',
    'components': [
        ('Build', {'skill_dist': "pareto", 'payment_max_skill_multiplier': 3}),
        ('ContinuousDoubleAuction', {'max_num_orders': 5}),
        ('Gather', {}),
    ],
    'env_layout_file': 'quadrant_25x25_20each_30clump.txt',
    'starting_agent_coin': 10,
    'fixed_four_skill_and_loc': True,
    'n_agents': 4,
    'world_size': [25, 25],
    'episode_length': 60,
    'multi_action_mode_agents': False,
    'multi_action_mode_planner': True,
    'flatten_observations': False,
    'flatten_masks': True,
}


def sample_random_action(agent, mask, rng):   # cell 18 (with an explicit generator instead of np.random)
    if agent.multi_action_mode:
        split_masks = np.split(mask, agent.action_spaces.cumsum()[:-1])
        return [rng.choice(np.arange(len(m_)), p=m_ / m_.sum()) for m_ in split_masks]
    return rng.choice(np.arange(agent.action_spaces), p=mask / mask.sum())


def sample_random_actions(env, obs, rng):
    return {a_idx: sample_random_action(env.get_agent(a_idx), a_obs['action_mask'], rng) for a_idx, a_obs in obs.items()}


def play(env, rng, dense):
    obs = env.reset(force_dense_logging=dense)
    trace = [obs]
    for t in range(env.episode_length):
        obs, rew, done, info = env.step(sample_random_actions(env, obs, rng))
        trace.append((obs, rew, done))
    return trace


def test_tutorial_loop_runs_unchanged_on_the_reference_api():
    env = foundation.make_env_instance(**ENV_CONFIG, reference_api=True, stepper_factory=emu_factory,
                                       dense_log_frequency=1)
    env.seed(5)
    assert env.get_agent(0).action_spaces == 50 and env.episode_length == 60
    trace = play(env, np.random.RandomState(0), dense=True)
    obs, rew, done = trace[-1]
    assert set(obs.keys()) == {"0", "1", "2", "3", "p"} and done["__all__"] is True
    assert isinstance(rew["0"], float) and isinstance(obs["0"]["world-inventory-Coin"], float)
    assert obs["0"]["world-map"].shape == (7, 11, 11) and obs["0"]["action_mask"].shape == (50,)
    assert set(obs["p"]["p0"].keys()) == {"world-inventory-Coin", "world-inventory-Stone", "world-inventory-Wood",
                                          "world-loc-row", "world-loc-col"}
    assert env._completions == 1 and isinstance(env._completions, int)   # counted on the step that ended the episode
    log = env.previous_episode_dense_log
    assert len(log["states"]) == 61 and len(log["actions"]) == 60 and set(log) >= {"world", "Build", "Gather", "Trade"}
    env.reset()
    m = env.previous_episode_metrics
    assert m is not None and "social/productivity" in m


@pytest.mark.parametrize("flags", [dict(flatten_observations=False, flatten_masks=True),
                                   dict(flatten_observations=True, flatten_masks=True),
                                   # schedules that live across resets: the "auto" warm-up integrator, completions
                                   dict(energy_warmup_constant=3, energy_warmup_method="auto", episode_length=30),
                                   dict(energy_warmup_constant=2, energy_warmup_method="decay", episode_length=30)],
                         ids=["named_fields", "flat", "auto_warmup", "decay_warmup"])
def test_reference_api_tracks_the_live_reference(flags, request):
    """Same config, same seed, same caller code on both: identical observation structure and values, two episodes (the
    reference's values as recorded, oracle/ref_tape.py)."""
    cfg = dict(ENV_CONFIG)
    cfg.update(flags)
    tape = ref_tape.Tape("reference_api", request.node.callspec.id)
    if tape.live:
        f = rh.load_reference_foundation()
        ref = f.make_env_instance(**cfg)
    mine = foundation.make_env_instance(**cfg, reference_api=True, stepper_factory=emu_factory)
    if tape.live:
        ref.seed(9)
    mine.seed(9)

    def leaf_types(b, label):
        if isinstance(b, dict):
            for k in b:
                leaf_types(b[k], label + "/" + str(k))
        else:
            assert type(b) in (float, list, np.ndarray, bool), (label, type(b))

    o1 = r1 = d1 = None
    for episode in range(3):
        ra, rb = np.random.RandomState(episode), np.random.RandomState(episode)
        if tape.live:
            o1 = ref.reset()
        o2 = mine.reset()
        leaf_types(o2, "reset %d" % episode)
        same_tree(tape, "obs", o1, o2, "reset %d" % episode)
        for t in range(mine.episode_length):
            a2 = sample_random_actions(mine, o2, rb)
            if tape.live:
                a1 = sample_random_actions(ref, o1, ra)
            agents = sorted(k for k in a2 if k != "p")
            tape.equal("actions", [int(a1[k]) for k in agents] if tape.live else None, [int(a2[k]) for k in agents], "ep %d t %d" % (episode, t))
            if tape.live:
                o1, r1, d1, _ = ref.step(a1)
            o2, r2, d2, _ = mine.step(a2)
            leaf_types(o2, "ep %d t %d obs" % (episode, t)); leaf_types(r2, "ep %d t %d rew" % (episode, t))
            same_tree(tape, "obs", o1, o2, "ep %d t %d obs" % (episode, t))
            same_tree(tape, "rew", r1, r2, "ep %d t %d rew" % (episode, t))
            tape.equal("done", ref_tape.flags(d1) if tape.live else None, ref_tape.flags(d2), "ep %d t %d" % (episode, t))
    tape.equal("metric keys", sorted(ref.metrics) if tape.live else None, sorted(mine.metrics))
    tape.finish()


@pytest.mark.gpu
def test_reference_api_cuda_matches_the_emulated_facade():
    """The facade over the CUDA stepper: same nested outputs as over the emulation, same caller code, two episodes."""
    cfg = dict(ENV_CONFIG, episode_length=25, flatten_observations=False, flatten_masks=True)
    cuda = foundation.make_env_instance(**cfg, reference_api=True, device="cuda:0")
    emu = foundation.make_env_instance(**cfg, reference_api=True, stepper_factory=emu_factory)
    cuda.seed(4); emu.seed(4)

    def same(a, b, label):
        if isinstance(a, dict):
            assert set(a) == set(b), label
            for k in a:
                same(a[k], b[k], label + "/" + str(k))
        else:
            assert np.allclose(np.asarray(a, np.float64), np.asarray(b, np.float64), rtol=1e-6, atol=1e-7), label

    for episode in range(2):
        ra, rb = np.random.RandomState(episode), np.random.RandomState(episode)
        o1, o2 = cuda.reset(), emu.reset()
        same(o1, o2, "reset")
        for t in range(25):
            (o1, r1, d1, _), (o2, r2, d2, _) = cuda.step(sample_random_actions(cuda, o1, ra)), emu.step(sample_random_actions(emu, o2, rb))
            same(o1, o2, "obs t=%d" % t); same(r1, r2, "rew t=%d" % t)
            assert d1 == d2
    assert cuda._completions == emu._completions == 2


def _final_state(env):
    d = env.stepper.read_state(0)
    return {k: np.array(d[k]) for k in ["cell", "owner", "loc", "inv", "esc", "coin", "labor", "mt_key", "mt_pos"]}


def test_replay_log_reproduces_an_episode():
    """previous_episode_replay_log (base_env.py:455-471): reset(**log["reset"]) + step(**s) for every logged step
    reproduces the episode exactly - state, metrics and dense log - whatever the env's stream did in between."""
    env = foundation.make_env_instance(**ENV_CONFIG, reference_api=True, stepper_factory=emu_factory, dense_log_frequency=1)
    env.seed(12)
    play(env, np.random.RandomState(0), dense=True)
    want_state, want_metrics, want_log = _final_state(env), env.metrics, env.previous_episode_dense_log
    log = env.previous_episode_replay_log
    assert len(log["step"]) == env.episode_length and len(log["reset"]["seed_state"]) == 5
    play(env, np.random.RandomState(99), dense=False)          # something else in between: the stream has moved on
    obs = env.reset(force_dense_logging=True, **log["reset"])
    for s in log["step"]:
        obs, rew, done, info = env.step(**s)
    got = _final_state(env)
    for k in want_state:
        assert np.array_equal(want_state[k], got[k]), k
    got_metrics = env.metrics
    assert set(got_metrics) == set(want_metrics)
    # (the auto warm-up integrator counts steps over the env's whole life, in the reference too)
    assert all(np.array_equal(got_metrics[k], want_metrics[k], equal_nan=True) for k in want_metrics if k != "labor/warmup_integrator")
    assert env.previous_episode_dense_log["states"] == want_log["states"]
    assert env.previous_episode_dense_log["Trade"] == want_log["Trade"]


def _log_text(log):
    """A replay log as canonical text (numpy scalars and arrays as numbers and lists)."""
    import json
    return json.dumps(log, sort_keys=True, default=lambda o: o.tolist() if hasattr(o, "tolist") else str(o))


def test_a_replay_log_recorded_by_the_reference_replays_here():
    """Cross-implementation replay: the unmodified reference plays an episode and hands over its replay log; replaying
    that log through the facade ends in the reference's final state and metrics (and the other way round).  The
    reference's log, end states and metrics are the ones recorded from it (oracle/ref_tape.py); the log the facade
    writes for the same play must be the reference's."""
    tape = ref_tape.Tape("reference_api_replay_log", 0)
    here = foundation.make_env_instance(**ENV_CONFIG, reference_api=True, stepper_factory=emu_factory)
    here.seed(5)
    play(here, np.random.RandomState(3), dense=False)
    log = here.previous_episode_replay_log
    want = {}
    if tape.live:
        f = rh.load_reference_foundation()
        ref = f.make_env_instance(**ENV_CONFIG)
        ref.seed(5)
        play(ref, np.random.RandomState(3), dense=False)
        tape.equal("log", _log_text(ref.previous_episode_replay_log), _log_text(log))
        log = ref.previous_episode_replay_log
        want = rh.state_arrays_from_reference(ref)
    else:
        tape.equal("log", None, _log_text(log))
    mine = foundation.make_env_instance(**ENV_CONFIG, reference_api=True, stepper_factory=emu_factory)
    mine.reset(**log["reset"])
    for s in log["step"]:
        mine.step(**s)
    got = _final_state(mine)
    for k in ["cell", "owner", "loc", "inv", "esc", "mt_key"]:
        tape.equal(k, want.get(k), got[k])
    tape.close("coin", want.get("coin"), got["coin"], rtol=1e-9, atol=1e-8)
    tape.close("labor", want.get("labor"), got["labor"], rtol=1e-9, atol=1e-8)
    m_mine = mine.metrics
    m_ref = ref.metrics if tape.live else {}
    tape.equal("metric keys", sorted(m_ref) if tape.live else None, sorted(m_mine))
    for k in sorted(m_mine):
        tape.close("metric/" + k, m_ref.get(k), float(m_mine[k]), rtol=1e-6, atol=1e-9, equal_nan=True)
    # ... and a log recorded here drives the reference to the same end state
    mine.seed(8)
    play(mine, np.random.RandomState(4), dense=False)
    log2, want2 = mine.previous_episode_replay_log, _final_state(mine)
    got2 = {}
    if tape.live:
        ref.reset(**log2["reset"])
        for s in log2["step"]:
            ref.step(**s)
        got2 = rh.state_arrays_from_reference(ref)
    for k in ["cell", "owner", "loc", "inv", "esc", "mt_key"]:
        tape.equal("replayed/" + k, got2.get(k), want2[k])
    tape.finish()
