"""CPU: the C oracle against the reference, step by step.  Shorter than the golden traces; different seeds.  The
reference's values are the ones recorded from the unmodified reference (tests/golden/reference_tapes/, oracle/ref_tape.py)."""
import pytest

from oracle import ref_tape


@pytest.mark.parametrize("cfg,seed,steps", [
    ("c1_tutorial", 31, 150), ("c3_short_period", 32, 120), ("c5_small", 33, 40), ("ref_unit_test", 34, 60),
])
def test_oracle_tracks_live_reference(cfg, seed, steps):
    from oracle.validate_vs_reference import run
    assert run(cfg, seed, steps, verbose=False, tape=ref_tape.Tape("oracle_vs_reference", "%s-%d-%d" % (cfg, seed, steps)))
