"""oracle/ref_tape.py on a synthetic case: what replay lets through and what it rejects.  A recorded 'reference' (per-agent
rewards as an array and as named entries, a metric, an exact flag) is replayed against perturbed copies of itself."""
import zlib

import numpy as np
import pytest

from oracle import ref_tape

STEPS, AGENTS, RTOL, ATOL = 64, 5, 1e-6, 1e-9
REF = np.random.RandomState(3).uniform(0.5, 2.0, (STEPS, AGENTS))


def play(tape, rew):
    for t in range(STEPS):
        live = tape.live
        tape.close("rew", REF[t] if live else None, rew[t], rtol=RTOL, atol=ATOL, where="t=%d" % t)
        ref_tape.same_tree(tape, "named", {str(a): REF[t, a] for a in range(AGENTS)} if live else None,
                           {str(a): rew[t, a] for a in range(AGENTS)}, "t=%d" % t, rtol=RTOL, atol=ATOL)
        tape.metric("total", REF[t].sum() if live else None, rew[t].sum(), "t=%d" % t)
        tape.equal("done", t == STEPS - 1 if live else None, t == STEPS - 1, "t=%d" % t)
    tape.finish()


@pytest.fixture
def recorded(tmp_path, monkeypatch):
    monkeypatch.setattr(ref_tape, "TAPE_DIR", str(tmp_path))
    monkeypatch.setattr(ref_tape, "_FILES", {})
    monkeypatch.setattr(ref_tape, "_VALUES", {})
    monkeypatch.setenv("AIE_RECORD_REFERENCE", "1")
    play(ref_tape.Tape("synthetic", 0, available=lambda: True), REF)
    monkeypatch.setenv("AIE_RECORD_REFERENCE", "0")
    monkeypatch.setattr(ref_tape, "_FILES", {})
    monkeypatch.setattr(ref_tape, "_VALUES", {})
    return lambda rew: play(ref_tape.Tape("synthetic", 0), rew)


def sampled(key, i):
    return (i + zlib.crc32(key.encode())) % ref_tape.STRIDE == 0


def test_replay_accepts_the_reference_and_anything_within_the_tolerance(recorded):
    recorded(REF.copy())
    recorded(REF * (1 + 0.9 * RTOL * np.where(np.arange(REF.size).reshape(REF.shape) % 2, 1, -1)))


@pytest.mark.parametrize("steps", ["all", "one"])
def test_replay_rejects_values_swapped_between_agents(recorded, steps):
    rew = REF.copy()
    rows = slice(None) if steps == "all" else [next(i for i in range(STEPS) if not sampled("rew", i))]   # outside the sample
    rew[rows, [0, 1]] = rew[rows, [1, 0]]
    with pytest.raises(ref_tape.Mismatch):
        recorded(rew)


def test_replay_rejects_one_element_off_by_more_than_its_tolerance_in_a_sampled_check(recorded):
    rew = REF.copy()
    t = next(i for i in range(STEPS) if sampled("named/3", i))
    rew[t, 3] *= 1 + 3 * RTOL   # 3x the element's own tolerance, no other value touched
    with pytest.raises(ref_tape.Mismatch, match="named/3"):
        recorded(rew)


def test_replay_rejects_one_element_off_by_more_than_its_tolerance_at_every_step(recorded):
    rew = REF.copy()
    rew[:, 2] *= 1 + 3 * RTOL
    with pytest.raises(ref_tape.Mismatch):
        recorded(rew)


def test_replay_rejects_a_single_deviation_above_the_summed_tolerance_outside_the_sample(recorded):
    rew = REF.copy()
    t = next(i for i in range(STEPS) if not any(sampled(k, i) for k in ("rew", "named/4", "total")))
    rew[t, 4] += 1e-3
    with pytest.raises(ref_tape.Mismatch):
        recorded(rew)
