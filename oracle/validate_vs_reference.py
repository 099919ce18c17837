"""TEST INFRASTRUCTURE: step the imported reference and the C oracle side by side.

Usage: python oracle/validate_vs_reference.py [config ...] [--steps N] [--seeds a,b]
"""
import argparse
import sys
import os

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import ref_harness as rh  # noqa: E402
from oracle import ref_tape  # noqa: E402
from oracle.oracle import OracleBatch  # noqa: E402
from oracle.configs import CONFIGS  # noqa: E402


EXACT_STATE = ["cell", "owner", "loc", "inv", "esc", "n_orders", "bid_hist", "ask_hist", "tax_pos", "rate_idx",
               "mt_key", "mt_pos", "t"]
CLOSE_STATE = ["coin", "esc_coin", "labor", "price_hist", "last_coin", "last_income", "last_marg"]
EXACT_OBS = ["a_map", "a_idx", "a_mask", "p_map", "p_idx", "p_mask", "done"]
CLOSE_OBS = ["a_flat", "p_flat", "p_agents", "time", "rew"]


def product_env(cfg, seed):
    """The product's host-side reset of a reference configuration (spec and post-reset state for the oracle)."""
    from ai_economist_b200 import foundation
    kw = dict(cfg)
    name = kw.pop("scenario_name")
    env = foundation.make_env_instance(name, n_envs=1, stepper_factory=lambda *a, **k: None, auto_reset=False, seed=None, **kw)
    env.seed(seed)
    return env, {k: v[0] for k, v in env.host_reset_arrays().items()}


RESET_KEYS = ["stone", "wood", "stone_src", "wood_src", "water", "loc", "mt_key", "mt_pos", "coin", "build_payment",
              "build_skill", "bonus_gather_prob"]


def run(cfg_name, seed, steps, verbose=True, tape=None):
    """The C oracle against the reference, step by step.  tape (oracle/ref_tape.py): None compares with the live reference;
    a replaying tape compares with its recorded digests, the oracle then starting from the product's host-side reset
    (which recording checks against the reference's post-reset state) and drawing the same actions from its own masks."""
    tape = tape or ref_tape.Tape()
    cfg = dict(CONFIGS[cfg_name])
    prod, host = product_env(cfg, seed)
    if tape.live:
        f = rh.load_reference_foundation()
        env = f.make_env_instance(**cfg)
        env.seed(seed)
        obs = env.reset()
        spec = rh.spec_from_reference_env(env)
        state = rh.state_from_reference_env(env)
    else:
        spec, state = prod.spec, host
    if tape.live and not set(spec) <= set(prod.spec):
        raise RuntimeError("spec keys the product lacks: %s" % sorted(set(spec) - set(prod.spec)))
    for k in tape.keys("spec", [k for k in sorted(prod.spec) if k != "components"], spec if tape.live else ()):
        tape.equal("spec/" + k, spec[k] if tape.live else None, prod.spec[k])
    for k in RESET_KEYS:
        tape.equal("reset/" + k, state[k] if tape.live else None, host[k])
    orc = OracleBatch(spec, 1)
    orc.load_env(0, state)
    arng = np.random.RandomState(seed + 7919)

    def check(t, obs=None, rew=None, done=None):
        ro = rs = {}
        if tape.live:
            ro = rh.obs_arrays_from_reference(env, obs, rew, done)
            rs = rh.state_arrays_from_reference(env)
        oo = orc.obs(0)
        os_ = orc.state(0)
        where = "[%s seed %d] step %d:" % (cfg_name, seed, t)
        for k in tape.keys("exact_obs%d" % bool(t), EXACT_OBS, ro):
            tape.equal(k, ro.get(k), oo[k], where, shape=True)
        for k in tape.keys("close_obs%d" % bool(t), CLOSE_OBS, ro):
            tape.close(k, ro.get(k), oo[k], rtol=1e-6, atol=1e-7, where=where, shape=True)
        for k in tape.keys("exact_state", EXACT_STATE, rs):
            tape.equal(k, rs.get(k), os_[k], where, shape=True)
        for k in tape.keys("close_state", CLOSE_STATE, rs):
            tape.close(k, rs.get(k), os_[k], rtol=1e-9, atol=1e-9, where=where, shape=True)
        for c, side in tape.keys("book", [(0, 0), (0, 1), (1, 0), (1, 1)], rs.get("book", {})):
            tape.equal("book%d%d" % (c, side), rs["book"][(c, side)] if tape.live else None, orc.book(0, c, side), where, shape=True)

    check(0, obs if tape.live else None)
    for t in range(1, steps + 1):
        o = orc.obs(0)
        actions, a_act, p_act = rh.sample_actions_from_masks(prod, o["a_mask"], o["p_mask"], arng)
        if tape.live:
            obs, rew, done, _ = env.step(actions)
        orc.step(a_act[None], p_act[None] if p_act.size else None)
        check(t, *((obs, rew, done) if tape.live else ()))
        if int(orc.obs(0)["done"][0]):
            break
    tape.finish()
    if verbose and tape.live:
        m = env.metrics
        print("[%s seed %d] %d steps OK  (trades=%s, builds=%s)" % (
            cfg_name, seed, t, m.get("Trade/n_trades", m.get("ContinuousDoubleAuction/n_trades")),
            m.get("Build/total_builds")))
    return True


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("configs", nargs="*", default=list(CONFIGS))
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--seeds", default="1001,1002")
    a = ap.parse_args()
    ok = True
    for c in a.configs:
        for s in [int(x) for x in a.seeds.split(",")]:
            try:
                run(c, s, a.steps)
            except ref_tape.Mismatch as ex:
                print("[%s seed %d] %s" % (c, s, ex))
                ok = False
    sys.exit(0 if ok else 1)
