"""Randomised fuzz (build container only): the COVID-19 device code (1-lane emulation; history scan and persistent change
list) against the LIVE reference under random unmasked policies, over scenario / component parameter variants.
python tools/fuzz_covid_vs_reference.py [n] [seed]"""
import contextlib
import io
import os
import sys
import traceback

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ai_economist_b200.foundation.covid19 import build_covid_params  # noqa: E402
from oracle import gen_golden_covid as gg  # noqa: E402
from oracle import ref_harness as rh  # noqa: E402
from oracle import ref_tape  # noqa: E402
from tests.emu.emu_stepper import EmuCovidStepper  # noqa: E402

KEYS = ["agent_state", "postsubsidy", "lagged", "policy_ind", "scalars", "mask_a", "mask_p"]


def random_kwargs(rng):
    kw = dict(gg.COVID_KWARGS)
    kw.update(episode_length=int(rng.choice([40, 90])), action_cooldown_period=int(rng.choice([1, 7, 28])),
              subsidy_interval=int(rng.choice([1, 30, 90])), num_subsidy_levels=int(rng.choice([5, 20])),
              start_date=str(rng.choice(["2020-03-22", "2020-06-01", "2020-10-15"])),
              economic_reward_crra_eta=float(rng.choice([0.5, 2.0, 3.0])),   # (eta = 1 is 0 / 0 in the reference)
              health_priority_scaling_agents=float(rng.choice([0.3, 1.0])),
              health_priority_scaling_planner=float(rng.choice([0.45, 2.0])), delivery_interval=int(rng.choice([1, 7])),
              vaccine_delivery_start_date=str(rng.choice(["2021-01-12", "2020-07-01"])),
              daily_vaccines_per_million_people=int(rng.choice([3000, 10000])))
    return kw


def run_one(kw, seed, tape=None):
    """tape (oracle/ref_tape.py): None compares with the live reference, a replaying tape with its recorded digests.
    The actions are drawn from the emulation's masks (equal to the reference's, which every check compares)."""
    tape = tape or ref_tape.Tape()
    if tape.live:
        f = rh.load_reference_foundation()
        with contextlib.redirect_stdout(io.StringIO()):
            ref = f.make_env_instance(**gg.reference_config(kw))
            obs = ref.reset()
    p = build_covid_params(**kw)
    emus = [EmuCovidStepper(p, 1, auto_reset=False, change_list=cl) for cl in (False, True)]
    for s in emus:
        s.reset()
    rng = np.random.RandomState(seed)

    # Rewards go through float32 x ** (1 - eta) and a min-max normalisation.  For the default eta = 2 that is a reciprocal
    # and the float32 rewards come out bit-identical; for other eta numpy's SIMD float32 power and libm's powf differ in
    # the last place, which the normalisation turns into an ABSOLUTE error of one or two float32 ulps of the O(1) terms the
    # reward is the difference of (measured over 400 configurations: <= 2.4e-7 absolute; relative to a reward that
    # happens to be near zero that was up to 8e-5, hence the absolute bound).
    rew_tol, rew_atol = (1e-6, 1e-9) if kw["economic_reward_crra_eta"] == 2.0 else (1e-5, 1e-6)

    def check(t, ra):
        ra = ra or {}
        for s in emus:
            o = s.read_obs(0)
            where = "t=%d (change_list=%s)" % (t, s.change_list)
            for k in KEYS:
                tape.close(k, ra.get(k), o[k], rtol=1e-6, atol=1e-9, where=where)
            if t:
                tape.close("rew_a", ra.get("rew_a"), o["rew_a"], rtol=rew_tol, atol=rew_atol, where=where)
                tape.close("rew_p", ra.get("rew_p"), float(o["rew_p"]), rtol=rew_tol, atol=rew_atol, where=where)
                tape.equal("done", int(ra["done"]) if tape.live else None, int(o["done"]), where)

    check(0, gg.ref_arrays(ref, obs) if tape.live else None)
    for t in range(1, kw["episode_length"] + 1):
        o = emus[0].read_obs(0)
        act_a, act_p = gg.sample({"a": {"action_mask": o["mask_a"]}, "p": {"action_mask": o["mask_p"]}}, rng)
        actions = {str(i): int(act_a[i]) for i in range(51)}
        actions["p"] = int(act_p)
        if tape.live:
            obs, rew, done, _ = ref.step(actions)
        for s in emus:
            s.buf["actions_agent"][0] = act_a
            s.buf["actions_planner"][0] = act_p
            s.step()
        check(t, gg.ref_arrays(ref, obs, rew, done) if tape.live else None)
    tape.finish()


if __name__ == "__main__":
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 10
    rng = np.random.RandomState(int(sys.argv[2]) if len(sys.argv) > 2 else 0)
    bad = 0
    for i in range(n):
        kw = random_kwargs(rng)
        try:
            run_one(kw, 900 + i)
        except Exception as ex:  # noqa: BLE001
            bad += 1
            print("[%d] FAILED %r\n    %s" % (i, kw, "".join(traceback.format_exception_only(type(ex), ex)).strip()[:400]))
    print("%d configs, %d failures" % (n, bad))
