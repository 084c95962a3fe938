"""Pins the oracle against the reference EXECUTED HERE (oracle/ref_loader.py): fresh random
inputs every run-size, wider than the committed fixtures.  The reference sources are not part of
this repository: the tests that step them are skipped unless GYM_LORENZ_REFERENCE points at a
checkout of them; the reset-range test checks the oracle side everywhere."""
import numpy as np
import pytest

import helpers as H
import refcheck as RC
from oracle import ref_loader as R

needs_reference = pytest.mark.skipif(not R.available(), reason="reference tree not present")

import sys, os  # noqa: E402
sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))


@needs_reference
@pytest.mark.parametrize("seed", [11, 12])
def test_oracle_equals_verbatim_reference(oracle_api, seed):
    import make_golden as MG
    rng = np.random.default_rng(seed)
    for name, kind, ns, na, kw, (lo, hi), amp in MG.CASES:
        for _ in range(4):
            st = MG.make_ic(rng, kind, ns, lo, hi, kw)
            T = 120
            acts = rng.uniform(-amp, amp, (T, na)).astype(np.float32)
            noisy = RC.uses_noise(kind, kw)
            nz = rng.standard_normal((T, 3)) if noisy else None
            adam0 = int(rng.integers(0, 30000)) if kind == "pmsm_sync" else 0
            with np.errstate(all="ignore"):
                r = RC.drive_reference(kind, st, acts, nz, adam_step=adam0, **kw)
                o = RC.drive_oracle(kind, st, acts, nz, adam_step=adam0, **kw)
            for key in ("state", "obs", "reward"):
                assert H.same_nonfinite(o[key], r[key]), (name, key)
                assert H.max_rel(o[key], r[key]) == 0.0, (name, key)
            assert np.array_equal(o["done"], r["done"]), name


def test_reference_reset_ranges_match_oracle_reset_ranges(oracle_api):
    """Reset draws cannot be stream-identical (MT19937/PCG64 vs Philox); ranges and obs
    construction must be.  The boxes are the reference's reset() ranges; its own draws are
    checked against them where its sources are present."""
    O = oracle_api
    spec = {"lorenz3": (-30, 30), "lorenz3_pair": (-20, 20), "lorenz4_pair": (0, 5), "pmsm_classic": (-10, 10)}
    for kind, (lo, hi) in spec.items():
        env = None
        if R.available():
            env = getattr(R, kind)()
            np.random.seed(1)
            env.reset()
            s = np.asarray(env.state1, np.float64)
            assert np.all(s >= lo) and np.all(s <= hi)
        orc = O.Oracle(kind, 2048, seed=5)
        orc.reset()
        nsys = 4 if kind == "lorenz4_pair" else 3
        x = orc.state[:nsys, :2048]
        assert x.min() >= lo and x.max() < hi
        assert abs(x.mean() - (lo + hi) / 2) < 0.05 * (hi - lo)
        # reset obs of the oracle == reference's _get_observation (dynamic.py:70-72, 80-83) for the same state
        if env is not None:
            RC.inject(kind, env, orc.state[:, 0].astype(np.float64))
        if kind == "lorenz3":
            d = env.state1 if env is not None else orc.state[:3, 0].astype(np.float64)
            ref_obs = np.array([d[0], d[1], d[2], 10 * (d[1] - d[0]), 28 * d[0] - d[1] - d[0] * d[2],
                                d[0] * d[1] - (8 / 3) * d[2]])
            orc2 = O.Oracle(kind, 2048, seed=5)
            obs = orc2.reset()
            assert np.array_equal(obs[:, 0], ref_obs)


@needs_reference
def test_special_action_values_clip_like_the_reference(oracle_api):
    """NaN propagates through np.clip, +-inf saturates; the oracle's clip must agree."""
    specials = np.array([np.nan, np.inf, -np.inf, 1e30, -1e30, 0.0, -0.0, 499.99997, 500.00003, 2.0000002], np.float32)
    rng = np.random.default_rng(3)
    for kind, ns, na, kw in (("lorenz3", 4, 3, {}), ("hr_sync", 9, 2, {}), ("pmsm_sync", 9, 2, {"alpha": 0.5}),
                             ("pmsm_classic", 7, 2, {}), ("memristive4_pair", 9, 3, {})):
        import make_golden as MG
        case = [c for c in MG.CASES if c[1] == kind][0]
        st = MG.make_ic(rng, kind, ns, *case[5], kw)
        acts = np.zeros((len(specials), na), np.float32)
        acts[:, 0] = specials; acts[:, -1] = specials[::-1]
        nz = rng.standard_normal((len(specials), 3)) if RC.uses_noise(kind, kw) else None
        with np.errstate(all="ignore"):
            r = RC.drive_reference(kind, st, acts, nz, **kw)
            o = RC.drive_oracle(kind, st, acts, nz, **kw)
        for key in ("state", "obs", "reward"):
            assert H.same_nonfinite(o[key], r[key]), (kind, key)
            assert H.max_rel(o[key], r[key]) == 0.0, (kind, key)
        assert np.array_equal(o["done"], r["done"])
