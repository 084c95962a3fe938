"""Generates the committed golden vectors from the UNMODIFIED reference (needs its sources).

    GYM_LORENZ_REFERENCE=<gym-lorenz checkout> python tests/golden/make_golden.py

Outputs (tests/golden/*.npz) -- all produced by executing the reference's own env classes
through oracle/ref_loader.py, or read from the reference's own artefact
$GYM_LORENZ_REFERENCE/PMSM_Origin_Data.xlsx (written by code/lorenz_pmsm/test_evaluate.py:61-166):

  cfg1_lorenz3.npz    BASELINE.json configs[0]: dynamic.py::lorenzEnv_transient, N=1,
                      np.random.seed(0); reset(); 1000 steps with
                      default_rng(1).uniform(-.05,.05,(1000,3)).astype(f32) actions; per-step
                      action/state1/obs/reward/done/t.  Plus a 1000-step run with
                      action_space-wide U(-500,500) actions that pins inf/NaN propagation.
  parity_<case>.npz   per env class / kwargs: 8 initial conditions x 64 free-running steps
                      with injected actions (and injected standard-normal draws where the
                      env consumes noise): st0, actions, noise, state, obs, reward, done.
  pmsm_xlsx_kat.npz   float32 error trajectories e1,e2,e3 from PMSM_Origin_Data.xlsx for the
                      prefix of each alpha column that a bang-bang (+-1)^2 action replay of
                      the reference env reproduces bit-exactly, with the inferred actions.
"""
from __future__ import annotations

import os
import re
import sys
import zipfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import refcheck as RC  # noqa: E402
from oracle import ref_loader as R  # noqa: E402

CASES = [
    # name, kind, n_state, act_dim, kwargs, (lo, hi) of IC draw, action amplitude
    ("lorenz3", "lorenz3", 4, 3, {}, (-30, 30), 0.05),
    ("lorenz3_pair", "lorenz3_pair", 10, 3, {}, (-20, 20), 0.05),
    ("lorenz4_pair", "lorenz4_pair", 9, 3, {}, (0, 5), 1.0),
    ("hr_sync", "hr_sync", 9, 2, {}, (-2, 2), 1.0),
    ("hr_sync_filter", "hr_sync", 9, 2, {"add_filter": True}, (-2, 2), 1.5),
    ("hr_sync_noise", "hr_sync", 9, 2, {"add_noise": True}, (-2, 2), 1.0),
    ("hr_sync_diverge", "hr_sync", 9, 2, {}, (-60, 60), 1.0),
    ("pmsm_sync_a050", "pmsm_sync", 9, 2, {"alpha": 0.5}, (-20, 20), 1.2),
    ("pmsm_sync_a033_noise", "pmsm_sync", 9, 2, {"alpha": 1 / 3, "add_noise": True}, (-20, 20), 1.2),
    ("pmsm_sync_diverge", "pmsm_sync", 9, 2, {"alpha": 0.5}, (-600, 600), 1.0),
    ("pmsm_classic", "pmsm_classic", 7, 2, {}, (-10, 10), 2.5),
    ("pmsm_single", "pmsm_single", 4, 2, {}, (-20, 20), 0.5),
    ("memristive4_pair", "memristive4_pair", 9, 3, {}, (0, 5), 2.5),
    ("pmsm_free", "pmsm_free", 4, 2, {}, (-20, 20), 0.0),
]
ZERO_PLANES = {
    "lorenz3": [3], "lorenz3_pair": [3], "lorenz4_pair": [8], "pmsm_classic": [6], "pmsm_single": [3],
    "memristive4_pair": [8], "pmsm_free": [3],
}


def make_ic(rng, kind, ns, lo, hi, kw):
    st = rng.uniform(lo, hi, ns)
    for p in ZERO_PLANES.get(kind, []):
        st[p] = 0.0
    if kind == "hr_sync":
        st[6] = 1.3 if kw.get("add_noise") else 0.0
        st[7:9] = 0.0
    if kind == "pmsm_sync":
        st = st.astype(np.float32).astype(np.float64)
        st[6:9] = 0.0
    return st


def gen_parity(outdir):
    rng = np.random.default_rng(20261018)
    for name, kind, ns, na, kw, (lo, hi), amp in CASES:
        K, T = 8, 64
        rec = {k: [] for k in ("st0", "actions", "noise", "state", "obs", "reward", "done", "adam0")}
        for k in range(K):
            st = make_ic(rng, kind, ns, lo, hi, kw)
            acts = rng.uniform(-amp, amp, (T, na)).astype(np.float32)
            noisy = RC.uses_noise(kind, kw)
            nz = rng.standard_normal((T, 3)) if noisy else np.zeros((T, 3))
            adam0 = int(rng.integers(0, 400)) if kind == "pmsm_sync" else 0
            r = RC.drive_reference(kind, st, acts, nz if noisy else None, adam_step=adam0, **kw)
            rec["st0"].append(st); rec["actions"].append(acts); rec["noise"].append(nz)
            rec["state"].append(r["state"]); rec["obs"].append(r["obs"])
            rec["reward"].append(r["reward"]); rec["done"].append(r["done"]); rec["adam0"].append(adam0)
        np.savez_compressed(os.path.join(outdir, f"parity_{name}.npz"), kind=kind,
                            kwargs=repr(kw), **{k: np.array(v) for k, v in rec.items()})
        print("wrote parity_" + name, "done steps:", int(np.sum(np.array(rec["done"]) != 0)))


def gen_cfg1(outdir):
    out = {}
    for tag, lo, hi in (("small", -0.05, 0.05), ("wide", -500.0, 500.0)):
        env = R.lorenz3()
        np.random.seed(0)
        obs0 = env.reset()
        st0 = np.array([*env.state1, env.t], np.float64)
        acts = np.random.default_rng(1).uniform(lo, hi, (1000, 3)).astype(np.float32)
        S, OB, RW, DN, TT = [], [], [], [], []
        with np.errstate(all="ignore"):
            for a in acts:
                o, r, d, _ = env.step(a)
                S.append(np.array(env.state1, np.float64)); OB.append(np.asarray(o, np.float64))
                RW.append(float(r)); DN.append(bool(d)); TT.append(env.t)
        out.update({f"{tag}_obs0": np.asarray(obs0, np.float64), f"{tag}_st0": st0, f"{tag}_actions": acts,
                    f"{tag}_state1": np.array(S), f"{tag}_obs": np.array(OB), f"{tag}_reward": np.array(RW),
                    f"{tag}_done": np.array(DN), f"{tag}_t": np.array(TT)})
    np.savez_compressed(os.path.join(outdir, "cfg1_lorenz3.npz"), **out)
    print("wrote cfg1_lorenz3: final t", out["small_t"][-1], "any done", out["small_done"].any(),
          "wide nonfinite rows", int(np.sum(~np.isfinite(out["wide_state1"]).all(axis=1))))


def read_xlsx(path):
    z = zipfile.ZipFile(path)
    sheets = []
    for k in (1, 2, 3):
        xml = z.read(f"xl/worksheets/sheet{k}.xml").decode()
        rows = re.findall(r"<row r=\"(\d+)\">(.*?)</row>", xml, flags=re.S)
        data = np.full((2000, 8), np.nan)
        for rnum, body in rows:
            r = int(rnum)
            if r < 2:
                continue
            for col, val in re.findall(r"<c r=\"([A-Z]+)\d+\" t=\"n\"><v>([^<]+)</v>", body):
                ci = ord(col) - ord("B")
                if 0 <= ci < 8:
                    data[r - 2, ci] = float(val)
        sheets.append(data)
    return np.stack(sheets, axis=-1)  # [2000 rows][8 alphas][3 error components]


def gen_xlsx_kat(outdir):
    xl = read_xlsx(os.path.join(R.REF_ROOT, "PMSM_Origin_Data.xlsx"))
    alphas = [1 / 2, 1 / 3, 1 / 4, 1 / 6, 1 / 7, 1 / 8, 1 / 9, 1 / 10]
    combos = [np.array(c, np.float32) for c in ((-1, -1), (-1, 1), (1, -1), (1, 1))]
    out = {}
    for ci, alpha in enumerate(alphas):
        env = R.pmsm_sync(alpha=alpha)
        env.reset(seed=0)
        env.state1 = np.array([10.0, -10.0, 15.0], dtype=np.float32)  # test_evaluate.py:75-76
        env.state2 = np.array([0.0, 0.0, 0.0], dtype=np.float32)
        acts, rows = [], []
        for t in range(2000):
            target = xl[t, ci].astype(np.float32)
            snap = (env.state1.copy(), env.state2.copy(), env.lambda_coef, env.m_t, env.v_t,
                    env.adam_step, env.current_step)
            hit = None
            for a in combos:
                env.state1, env.state2 = snap[0].copy(), snap[1].copy()
                env.lambda_coef, env.m_t, env.v_t, env.adam_step, env.current_step = snap[2:]
                env.step(a)
                e = env.state1 - env.state2
                if np.array_equal(e, target):
                    hit = a
                    break
            if hit is None:
                break
            acts.append(hit); rows.append(target)
        n = len(acts)
        print(f"alpha=1/{round(1 / alpha)}: bang-bang replay reproduces {n} xlsx rows bit-exactly")
        if n >= 40:
            out[f"a{ci}_alpha"] = np.float64(alpha)
            out[f"a{ci}_actions"] = np.array(acts, np.float32)
            out[f"a{ci}_err"] = np.array(rows, np.float32)
    # action-independent KAT quoted in SURVEY 8c: e3 after step 1 is the same in every column
    assert np.all(xl[0, :, 2].astype(np.float32) == np.float32(14.863499641418457))
    np.savez_compressed(os.path.join(outdir, "pmsm_xlsx_kat.npz"), **out)


def eval_inputs(rng, T, K):
    """Synthetic sync-error / control trajectories shaped like the evaluation script's (decaying
    oscillation + noise), with the three special cases of the settling-time logic."""
    t = np.arange(T)[:, None, None]
    tau = rng.uniform(20, 400, size=(1, 3, K))
    e = rng.uniform(0.5, 30, size=(1, 3, K)) * np.exp(-t / tau) * np.cos(t / 7.0) + 0.01 * rng.normal(size=(T, 3, K))
    e[-1, 0, 0] = 1.0          # trajectory 0: component 0 never settles
    e[-1, :, 1] = 1.0          # trajectory 1: nothing settles -> NaN
    e[:, :, 2] = 0.001         # trajectory 2: never leaves the band -> 0
    u = rng.normal(size=(T, 2, K)) * 50
    return e.astype(np.float32).astype(np.float64), u.astype(np.float32).astype(np.float64)   # compact fixture


def gen_eval_metrics(outdir):
    """calculate_advanced_metrics + the steady-state block of code/lorenz_pmsm/test_evaluate.py
    (:25-59, :239-250), executed from the reference file itself (oracle/ref_loader.py)."""
    block = R.eval_steady_block()
    rng = np.random.default_rng(77)
    out = {}
    for tag, T, K, dt in (("long", 2200, 10, 0.001), ("short", 1200, 10, 0.01)):
        e, u = eval_inputs(rng, T, K)
        res = np.array([block(e[:, 0, k], e[:, 1, k], e[:, 2, k], u[:, 0, k], u[:, 1, k], dt) for k in range(K)])
        out.update({f"{tag}_err": e.astype(np.float32), f"{tag}_ctrl": u.astype(np.float32), f"{tag}_dt": np.float64(dt),
                    f"{tag}_metrics": res})          # columns: mae, rmse, max settling time, energy
    np.savez_compressed(os.path.join(outdir, "eval_metrics.npz"), **out)
    print("wrote eval_metrics:", {k: v.shape for k, v in out.items() if hasattr(v, "shape") and v.ndim})


DERIV_KINDS = [("lorenz3", 3, (-30, 30)), ("lorenz3_pair", 3, (-20, 20)), ("lorenz4_pair", 4, (0, 5)),
               ("pmsm_classic", 3, (-10, 10)), ("pmsm_single", 3, (-20, 20))]


def gen_derivatives(outdir):
    """Right-hand sides as the reference evaluates them.  Classic envs: after step(), env.state0 =
    [state1_new, f(state1_new)] (e.g. dynamic.py:77-80, lorenz_env_transient.py:332-339,
    lorenz_env_transient_pmsm.py:107-112) -- pairs (state, derivative) harvested from stepping the
    unmodified env.  HR: the module-level hr_derivatives (lorenz_env_try.py:7-12) called directly with
    the env's constants and controls (a1, a2) = clip(a)*100 as step() forms them (:92-93)."""
    rng = np.random.default_rng(4242)
    out = {}
    for kind, dim, (lo, hi) in DERIV_KINDS:
        S, D = [], []
        ns = {"lorenz3": 4, "lorenz3_pair": 10, "lorenz4_pair": 9, "pmsm_classic": 7, "pmsm_single": 4}[kind]
        for k in range(48):
            env = RC.make_reference(kind)
            st = make_ic(rng, kind, ns, lo, hi, {})
            RC.inject(kind, env, st)
            na = 2 if kind.startswith("pmsm") else 3
            for t in range(6):
                with np.errstate(all="ignore"):
                    env.step(rng.uniform(-0.05, 0.05, na).astype(np.float32))
                s0 = np.asarray(env.state0, np.float64)
                S.append(s0[:dim]); D.append(s0[dim:2 * dim])
        out[f"{kind}_state"], out[f"{kind}_deriv"] = np.array(S), np.array(D)
    mod = R.load("lorenz_env_try.py")
    env = R.hr_sync()
    x = rng.uniform(-3, 3, (256, 3))
    act = rng.uniform(-1.3, 1.3, (256, 2)).astype(np.float32)
    a12 = np.clip(act, -1.0, 1.0) * 100.0                 # float32, as lorenz_env_try.py:92-93
    assert a12.dtype == np.float32
    d = np.array([mod.hr_derivatives(x[k], a12[k, 0], a12[k, 1], env.a, env.b, env.c, env.d, env.r, env.s,
                                     env.I_bias, env.x_rest) for k in range(256)], np.float64)
    d0 = np.array([mod.hr_derivatives(x[k], 0, 0, env.a, env.b, env.c, env.d, env.r, env.s, env.I_bias, env.x_rest)
                   for k in range(256)], np.float64)
    out.update({"hr_sync_state": x, "hr_sync_action": act, "hr_sync_control": a12.astype(np.float32),
                "hr_sync_deriv": d, "hr_sync_deriv_free": d0})
    np.savez_compressed(os.path.join(outdir, "derivatives.npz"), **out)
    print("wrote derivatives:", {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    if not R.available():
        sys.exit("reference tree not found; golden vectors can only be regenerated where it exists")
    gen_cfg1(HERE)
    gen_parity(HERE)
    gen_xlsx_kat(HERE)
    gen_eval_metrics(HERE)
    gen_derivatives(HERE)
