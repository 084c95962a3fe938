"""The SB3 kernels of csrc/tu_rl_ops.cu and the MLP of csrc/tu_policy.cu at the shapes where their
shape-dependent branches switch, against float64 references written here.

Branches reached: k_moments<8> / <32> with its grid-stride loop and f64 input; both k_normalize kernels
and the shared-memory gate between them; k_frame_stack_warp (vector and scalar stores) and the
one-thread-per-row fallback; the 8-step and remainder loops of k_gae; k_eval_partial with several
segments, a single segment, segment remainders and every n_err / n_ctrl; policy_block's three block
sizes with a partial last block, observation and action clipping and T = 1 in k_policy_rollout.

The C-ABI is called directly where the Python wrappers cannot produce an input: padded strides,
stride > n, unaligned output pointers, n_ctrl = 0.  Padding that a kernel must not touch holds a
sentinel and is checked afterwards."""
import ctypes as C
import math
import types
import warnings

import numpy as np
import pytest

from oracle import sb3_ref as S

HIDDEN = 64          # CL_POLICY_HIDDEN
SENTINEL = -1234.5   # written into padding a kernel must leave alone


# ---- float64 references ------------------------------------------------------------------------

def moments_ref(x, shift):
    """Per feature: sum(x - shift) and sum((x - shift)^2), x [n, dim].  The difference is rounded to
    f64 once, as the kernel does; the sums are taken in extended precision (64-bit mantissa), which is
    exact to far below the 1e-12 the kernel is held to."""
    d = np.asarray(x, np.float64) - np.asarray(shift, np.float64)
    dl = d.astype(np.longdouble)
    return dl.sum(axis=0), (dl * dl).sum(axis=0), np.abs(dl).sum(axis=0)


def merge_ref(mean, var, count, x):
    """RunningMeanStd.update_from_moments (Chan et al.) from the exact batch mean and variance of
    x [n, dim], in extended precision.  Returns (mean, var, count, batch_mean)."""
    xl = np.asarray(x, np.float64).astype(np.longdouble)
    n = xl.shape[0]
    bm = xl.sum(axis=0) / n
    bv = ((xl - bm) ** 2).sum(axis=0) / n
    m, v, c = (np.asarray(a, np.float64).astype(np.longdouble) for a in (mean, var, count))
    delta = bm - m
    tot = c + n
    new_mean = m + delta * n / tot
    m2 = v * c + bv * n + delta * delta * c * n / tot
    return new_mean, m2 / tot, tot, bm


def metrics_ref(err, ctrl, dt, band=0.05, steady_start=None):
    """err [T, n_err], ctrl [T, n_ctrl] -> (mae, rmse, settling time, energy): the steady-state block of
    the reference's evaluation script (sb3_ref.steady_state_metrics) with every constant an argument.
    The statements are the same, so at n_err = 3, n_ctrl = 2 the results are the same bits."""
    err, ctrl = np.asarray(err, np.float64), np.asarray(ctrl, np.float64)
    T, n_err = err.shape
    if steady_start is None:
        steady_start = min(1000, T // 2)
    s = err[steady_start:]
    mae = np.mean([np.mean(np.abs(s[:, c])) for c in range(n_err)])
    rmse = np.mean([np.sqrt(np.mean(s[:, c] ** 2)) for c in range(n_err)])
    ts = []
    for c in range(n_err):
        exceed = np.where(np.abs(err[:, c]) > band)[0]
        if len(exceed) == 0:
            ts.append(0.0)
        else:
            stable_idx = exceed[-1] + 1
            ts.append(stable_idx * dt if stable_idx < T else np.nan)
    q = np.zeros(T)
    if ctrl.shape[1] > 0:
        q = np.square(ctrl[:, 0])
        for c in range(1, ctrl.shape[1]):
            q = q + np.square(ctrl[:, c])
    energy = np.sum(q) * dt
    with np.errstate(all="ignore"), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        max_ts = np.nanmax(ts)
    return mae, rmse, max_ts, energy


def frame_stack_term_ref(prev, term_in):
    """StackedObservations.update's terminal observation: the previous stack rolled by one frame without
    its last frame, followed by the env's terminal observation."""
    dim = term_in.shape[1]
    return np.concatenate([prev[:, dim:], term_in], axis=1)


def mlp_ref(packed, z, obs_dim, act_dim):
    """The MlpPolicy's pre-clip actions in f64, read from the packed parameter block at the offsets
    pack_policy documents: W1[64][obs_dim] b1[64] W2[64][64] b2[64] W3[act_dim][64] b3[act_dim]."""
    p = np.asarray(packed, np.float64)
    h, o = HIDDEN, 0

    def take(k, shape):
        nonlocal o
        a = p[o:o + k].reshape(shape)
        o += k
        return a
    W1, b1 = take(h * obs_dim, (h, obs_dim)), take(h, (h,))
    W2, b2 = take(h * h, (h, h)), take(h, (h,))
    W3, b3 = take(act_dim * h, (act_dim, h)), take(act_dim, (act_dim,))
    assert o == p.size
    h1 = np.tanh(np.asarray(z, np.float64) @ W1.T + b1)
    h2 = np.tanh(h1 @ W2.T + b2)
    return h2 @ W3.T + b3


def policy_block(n, sms):
    """A copy of policy_block() in csrc/tu_policy.cu (change both together): fewest threads on the
    fullest SM, ties to the larger block.  It only chooses the n of the block-size tests below."""
    best, best_cost = 128, None
    for b in (128, 64, 32):
        cost = ((-(-n // b) + sms - 1) // sms) * b
        if best_cost is None or cost < best_cost:
            best, best_cost = b, cost
    return best


def _same_metric(got, want):
    """mae / rmse / energy within 1e-12 relative (NaN where the reference is NaN)."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want)
    assert np.all(np.abs(got[ok] - want[ok]) <= 1e-12 * np.abs(want[ok])), np.max(np.abs(got[ok] - want[ok]))


def _same_settling(got, want):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    assert np.array_equal(got[~np.isnan(want)], want[~np.isnan(want)])


# ---- CPU: the references against the pinned ones -------------------------------------------------

@pytest.mark.parametrize("tag", ["long", "short"])
def test_metrics_ref_equals_the_pinned_restatement_bit_for_bit(tag):
    import helpers as H
    gold = np.load(f"{H.GOLDEN}/eval_metrics.npz")
    e, u, dt = gold[f"{tag}_err"].astype(np.float64), gold[f"{tag}_ctrl"].astype(np.float64), float(gold[f"{tag}_dt"])
    for k in range(e.shape[2]):
        want = S.steady_state_metrics(e[:, :, k], u[:, :, k], dt=dt)
        got = metrics_ref(e[:, :, k], u[:, :, k], dt, 0.05)
        for g, w in zip(got, want):
            g, w = float(g), float(w)
            assert (math.isnan(g) and math.isnan(w)) or g == w, (tag, k, got, want)
        # and the fixture itself (the reference's own numbers)
        for c in range(4):
            g, w = float(got[c]), float(gold[f"{tag}_metrics"][k, c])
            assert (math.isnan(g) and math.isnan(w)) or g == w


def test_metrics_ref_edge_cases():
    T, band, dt = 10, 0.05, 0.01
    e = np.zeros((T, 2))
    e[:, 0] = band                         # |e| == band is not an exceedance
    assert metrics_ref(e, np.zeros((T, 0)), dt, band, 0)[2] == 0.0
    e[0, 1] = 1.0                          # only t = 0 leaves the band: settles at dt
    assert metrics_ref(e, np.zeros((T, 0)), dt, band, 0)[2] == dt
    e[T - 1, 1] = 1.0                      # one component outside at T - 1: NaN for it, nanmax finite
    assert metrics_ref(e, np.zeros((T, 0)), dt, band, 0)[2] == 0.0
    e[T - 1, 0] = -1.0                     # every component: NaN
    assert np.isnan(metrics_ref(e, np.zeros((T, 0)), dt, band, 0)[2])
    e[3, 0] = np.nan                       # NaN: never an exceedance, but the sums are NaN
    mae, rmse, ts, en = metrics_ref(e, np.ones((T, 3)), dt, band, 0)
    assert np.isnan(mae) and np.isnan(rmse) and np.isnan(ts) and en == 3 * T * dt
    assert metrics_ref(e, np.ones((T, 3)), dt, band, 4)[0] == np.mean([np.mean(np.abs(e[4:, c])) for c in range(2)])


def test_moments_and_merge_ref_agree_with_running_mean_std():
    rng = np.random.default_rng(11)
    rms = S.RunningMeanStd(shape=(5,))
    mean, var, count = rms.mean.copy(), rms.var.copy(), rms.count
    for k in range(4):
        x = rng.normal(rng.uniform(-1e3, 1e3, 5), rng.uniform(1e-3, 1e3, 5), size=(777 + k, 5))
        s1, s2, _ = moments_ref(x, mean)
        bm, bv = np.mean(x, axis=0), np.var(x, axis=0)
        d = bm - mean
        assert np.all(np.abs(s1 / len(x) - d) <= 1e-12 * (np.abs(d) + np.sqrt(bv)))
        assert np.all(np.abs(s2 / len(x) - (bv + d * d)) <= 1e-12 * (bv + d * d))
        rms.update(x)
        mean, var, count, _ = merge_ref(mean, var, count, x)
        mean, var, count = mean.astype(np.float64), var.astype(np.float64), float(count)
        assert np.allclose(mean, rms.mean, rtol=1e-12, atol=0)
        assert np.allclose(var, rms.var, rtol=1e-12, atol=0)
        assert count == rms.count


def test_policy_block_choices():
    """The n of the policy tests below give each block size a partial last block on a 148-SM B200."""
    for n, b in ((33, 32), (65530, 64), (18939, 128)):
        assert policy_block(n, 148) == b and n % b != 0


def test_mlp_ref_reads_the_packed_layout(chaos_lib):
    import torch
    from gym_lorenz_b200.rl_ops import pack_policy
    torch.manual_seed(3)
    pnet = torch.nn.Sequential(torch.nn.Linear(6, 64), torch.nn.Tanh(), torch.nn.Linear(64, 64), torch.nn.Tanh())
    anet = torch.nn.Linear(64, 2)
    packed = pack_policy((pnet, anet), "cpu", "hr_sync").numpy()
    z =np.random.default_rng(0).normal(size=(50, 6)).astype(np.float32)
    with torch.no_grad():
        want = anet.double()(pnet.double()(torch.as_tensor(z, dtype=torch.float64))).numpy()
    assert np.allclose(mlp_ref(packed, z, 6, 2), want, rtol=1e-13, atol=1e-13)


# ---- GPU plumbing ---------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def gpu(chaos_lib):
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from gym_lorenz_b200 import _lib as L
    return types.SimpleNamespace(torch=torch, L=L, lib=chaos_lib, dev=torch.device("cuda:0"))


def _ptr(t, offset_elems=0):
    return C.c_void_p(t.data_ptr() + offset_elems * t.element_size())


def _call(g, fn, *args):
    rc = fn(C.c_void_p(g.torch.cuda.current_stream(g.dev).cuda_stream), *args)
    g.torch.cuda.synchronize(g.dev)
    return rc


def _ok(g, name, *args):
    rc = _call(g, getattr(g.lib, name), *args)
    assert rc == 0, f"{name} returned {rc}: {g.lib.cl_last_error(None)}"


# ---- moments --------------------------------------------------------------------------------------

def _moment_data(rng, n, dim, f64):
    off, spread = rng.uniform(-1e3, 1e3, dim), 10.0 ** rng.uniform(-3, 3, dim)
    x = off + spread * rng.standard_normal((n, dim))
    shift = off + spread * rng.uniform(-2, 2, dim)          # the running mean: near, not at, the data
    return (x if f64 else x.astype(np.float32)), shift


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 31, 257, 1_000_003])
@pytest.mark.parametrize("dim", [1, 6, 8, 9, 24, 32])
def test_moments_vs_extended_precision_sums(gpu, dim, n):
    torch = gpu.torch
    rng = np.random.default_rng(dim * 7919 + n)
    for f64, name in ((False, "cl_obs_moments"), (True, "cl_moments_f64")):
        x, shift = _moment_data(rng, n, dim, f64)
        s1, s2, sabs = moments_ref(x, shift)
        xd = torch.as_tensor(x, device=gpu.dev)
        padded = torch.full((n, dim + 3), float("nan"), dtype=xd.dtype, device=gpu.dev)
        padded[:, :dim] = xd
        planes = xd.t().contiguous()
        sh = torch.as_tensor(shift, device=gpu.dev)
        for layout, buf, es, cs in (("rows", xd, dim, 1), ("planes", planes, 1, n), ("padded", padded, dim + 3, 1)):
            out = torch.full((2, dim), SENTINEL, dtype=torch.float64, device=gpu.dev)
            _ok(gpu, name, _ptr(buf), es, cs, n, dim, _ptr(sh), _ptr(out))
            got = out.cpu().numpy()
            tag = (name, layout)
            assert np.all(np.abs(got[0] - s1.astype(np.float64)) <= 1e-12 * sabs.astype(np.float64)), tag
            assert np.all(np.abs(got[1] - s2.astype(np.float64)) <= 1e-12 * s2.astype(np.float64)), tag
    # more features than k_moments<32> keeps in registers: refused
    out = torch.zeros((2, 33), dtype=torch.float64, device=gpu.dev)
    big32 = torch.zeros((4, 33), dtype=torch.float32, device=gpu.dev)
    big64 = big32.double()
    sh = torch.zeros(33, dtype=torch.float64, device=gpu.dev)
    assert _call(gpu, gpu.lib.cl_obs_moments, _ptr(big32), 33, 1, 4, 33, _ptr(sh), _ptr(out)) != 0
    assert _call(gpu, gpu.lib.cl_moments_f64, _ptr(big64), 33, 1, 4, 33, _ptr(sh), _ptr(out)) != 0


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [1, 6, 8, 9, 24, 32])
@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_running_mean_std_update_vs_chan_merge(gpu, dtype, dim):
    """Each device update is compared with merge_ref started from the device's own previous state, so
    every merge is checked on its own.  The device forms the batch variance as E[d^2] - E[d]^2 with
    d = x - old_mean: that loses about eps * (batch_mean - old_mean)^2, so the variance is held to
    1e-12 * (var + (batch_mean - old_mean)^2), and the mean to 1e-12 of the larger of |mean| and the
    step it took."""
    torch = gpu.torch
    from gym_lorenz_b200.rl_ops import RunningMeanStd
    rng = np.random.default_rng(dim + (100 if dtype == "float64" else 0))
    rms = RunningMeanStd((dim,), gpu.dev)
    centre = rng.uniform(300, 1e3, dim) * rng.choice([-1, 1], dim)    # first batch far from the initial 0
    for k, n in enumerate((4099, 257, 1, 70_001)):
        x = centre * (1 + 0.1 * k) + 10.0 ** rng.uniform(-2, 2, dim) * rng.standard_normal((n, dim))
        x = x.astype(dtype)
        m0, v0, c0 = rms.mean.cpu().numpy(), rms.var.cpu().numpy(), rms.count
        rms.update(torch.as_tensor(x, device=gpu.dev))
        mean, var, count, bm = merge_ref(m0, v0, c0, x)
        mean, var, bm = mean.astype(np.float64), var.astype(np.float64), bm.astype(np.float64)
        gm, gv = rms.mean.cpu().numpy(), rms.var.cpu().numpy()
        step = np.abs(bm - m0)
        assert np.all(np.abs(gm - mean) <= 1e-12 * np.maximum(np.abs(mean), step)), (k, gm - mean)
        assert np.all(np.abs(gv - var) <= 1e-12 * (var + step ** 2)), (k, gv - var)
        assert rms.count == c0 + n


# ---- normalise + clip -----------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 31, 32, 33, 255, 257, 4099])
@pytest.mark.parametrize("dim", [1, 3, 5, 6, 8, 24, 47, 48, 49, 64])
def test_normalize_bit_exact_for_every_output_layout(gpu, dim, n):
    """Contiguous rows take the shared-memory transpose (k_normalize<true>) while its dynamic shared
    memory fits next to the static one (dim <= 47); the other outputs take the strided kernel.  The
    results are the same bits either way: which kernel ran is checked in the next test."""
    torch = gpu.torch
    rng = np.random.default_rng(dim * 131 + n)
    eps = 1e-8
    rms = S.RunningMeanStd(shape=(dim,))
    rms.mean = rng.uniform(-5, 5, dim)
    rms.var = 10.0 ** rng.uniform(-3, 2, dim)
    rms.var[dim // 2] = 0.0                                  # zero-variance column: divides by sqrt(eps)
    x = (rms.mean + np.sqrt(rms.var + eps) * rng.normal(0, 6, (n, dim))).astype(np.float32)
    specials = np.array([np.inf, -np.inf, np.nan, 1e30, -1e30, 0.0], np.float32)
    mask = rng.random((n, dim)) < 0.05
    x[mask] = rng.choice(specials, int(mask.sum()))
    xd = torch.as_tensor(x, device=gpu.dev)
    xp = xd.t().contiguous()                                 # SoA planes [dim][n]
    md, vd = torch.as_tensor(rms.mean, device=gpu.dev), torch.as_tensor(rms.var, device=gpu.dev)
    for clip in (0.5, 10.0):
        want = S.normalize_obs(x, rms, clip_obs=clip, epsilon=eps)
        assert want.dtype == np.float32
        rows = torch.full((n, dim), SENTINEL, dtype=torch.float32, device=gpu.dev)
        wide = torch.full((n, dim + 5), SENTINEL, dtype=torch.float32, device=gpu.dev)
        shifted = torch.full((n * dim + 1,), SENTINEL, dtype=torch.float32, device=gpu.dev)
        planes = torch.full((dim, n), SENTINEL, dtype=torch.float32, device=gpu.dev)
        cases = (("rows", xd, dim, 1, rows, 0, dim, 1),
                 ("slice", xd, dim, 1, wide, 0, dim + 5, 1),
                 ("unaligned", xd, dim, 1, shifted, 1, dim, 1),
                 ("planes", xp, 1, n, planes, 0, 1, n))
        for tag, src, ies, ics, out, off, oes, ocs in cases:
            _ok(gpu, "cl_obs_normalize", _ptr(src), ies, ics, _ptr(out, off), oes, ocs, n, dim, _ptr(md), _ptr(vd),
                eps, clip)
        got = {"rows": rows.cpu().numpy(), "slice": wide[:, :dim].cpu().numpy(),
               "unaligned": shifted[1:].view(n, dim).cpu().numpy(), "planes": planes.t().cpu().numpy()}
        for tag, g in got.items():
            assert np.array_equal(g, want, equal_nan=True), (tag, clip)
        assert bool((wide[:, dim:] == SENTINEL).all()) and float(shifted[0]) == SENTINEL


@pytest.mark.gpu
def test_normalize_rows_kernel_runs_while_its_shared_memory_fits(gpu):
    """Which kernel cl_obs_normalize launches, read from the profiler's kernel names: contiguous, aligned
    rows take k_normalize<true> up to dim 47 (8 warps x 32 rows x dim floats of dynamic shared memory
    next to 768 B of static: 48,128 + 768 B <= 48 KiB); dim 48 would need 49,152 + 768 B and takes
    k_normalize<false>, as do sliced, unaligned and SoA outputs at every dim."""
    torch = gpu.torch
    from torch.profiler import ProfilerActivity, profile
    n = 300

    def kernels(launch):
        """The k_normalize variants the profiler recorded over three launches.  A session can drop
        records (it does after an earlier profiler session in the same process), never rename one."""
        torch.cuda.synchronize(gpu.dev)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                launch()
        keys = [e.key for e in prof.key_averages() if "k_normalize" in e.key]
        return {"rows" if ("k_normalize<true>" in k or "k_normalizeILb1E" in k) else
                "strided" if ("k_normalize<false>" in k or "k_normalizeILb0E" in k) else k for k in keys}

    kernels(lambda: torch.ones(8, device=gpu.dev).add_(1))   # a first session that may drop records
    for dim in (1, 6, 24, 47, 48, 49, 64):
        x = torch.randn((n, dim), dtype=torch.float32, device=gpu.dev)
        m = torch.zeros(dim, dtype=torch.float64, device=gpu.dev)
        v = torch.ones(dim, dtype=torch.float64, device=gpu.dev)
        rows = torch.empty((n, dim), dtype=torch.float32, device=gpu.dev)
        wide = torch.empty((n, dim + 5), dtype=torch.float32, device=gpu.dev)
        flat = torch.empty((n * dim + 1,), dtype=torch.float32, device=gpu.dev)
        planes = torch.empty((dim, n), dtype=torch.float32, device=gpu.dev)
        for tag, out, off, oes, ocs in (("rows", rows, 0, dim, 1), ("slice", wide, 0, dim + 5, 1),
                                        ("unaligned", flat, 1, dim, 1), ("planes", planes, 0, 1, n)):
            got = kernels(lambda: _ok(gpu, "cl_obs_normalize", _ptr(x), dim, 1, _ptr(out, off), oes, ocs, n, dim,
                                      _ptr(m), _ptr(v), 1e-8, 10.0))
            want = "rows" if tag == "rows" and dim <= 47 else "strided"
            assert got == {want}, (dim, tag, got)


# ---- frame stack ----------------------------------------------------------------------------------

FS_SHAPES = [(d, k) for d in (1, 2, 3, 5, 6, 8) for k in (1, 2, 3, 4)] + [(6, 6), (6, 7), (6, 32)]


def _done_pattern(rng, t, n):
    """None (a null pointer), none, all, 20 %, alternating lanes -- in turn."""
    mode = t % 5
    if mode == 0:
        return None
    if mode == 1:
        return np.zeros(n, np.uint8)
    if mode == 2:
        return np.ones(n, np.uint8)
    if mode == 3:
        return (rng.random(n) < 0.2).astype(np.uint8)
    return (np.arange(n) % 2 == t % 2).astype(np.uint8)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 31, 33, 1000, 4099])
@pytest.mark.parametrize("dim,n_stack", FS_SHAPES)
def test_frame_stack_and_terminal_stack_bit_exact(gpu, dim, n_stack, n):
    """(6, 6) needs exactly 48 KiB of shared memory in k_frame_stack_warp; (6, 7) and (6, 32) take the
    one-thread-per-row kernel.  Two stacks are kept side by side: a 16-byte aligned one (vector loads
    and stores) and one offset by a float (scalar path)."""
    torch = gpu.torch
    rng = np.random.default_rng(dim * 1000 + n_stack * 10 + n)
    rowlen = dim * n_stack
    ref = rng.normal(size=(n, rowlen)).astype(np.float32)
    aligned = torch.as_tensor(ref, device=gpu.dev).contiguous()
    shifted = torch.full((n * rowlen + 1,), SENTINEL, dtype=torch.float32, device=gpu.dev)
    shifted[1:] = aligned.view(-1)
    term = torch.empty((n, rowlen), dtype=torch.float32, device=gpu.dev)
    for t in range(max(n_stack + 2, 10)):
        obs = rng.normal(size=(n, dim)).astype(np.float32)
        term_in = rng.normal(size=(n, dim)).astype(np.float32)
        done = _done_pattern(rng, t, n)
        soa = t % 2 == 1                                     # observations as SoA planes every other push
        od = torch.as_tensor(np.ascontiguousarray(obs.T) if soa else obs, device=gpu.dev)
        es, cs = (1, n) if soa else (dim, 1)
        td = torch.as_tensor(np.ascontiguousarray(term_in.T) if not soa else term_in, device=gpu.dev)
        tes, tcs = (dim, 1) if soa else (1, n)
        dd = None if done is None else torch.as_tensor(done, device=gpu.dev)
        with_term = dd is not None and t % 3 != 0
        want_term = frame_stack_term_ref(ref, term_in)
        ref = S.frame_stack_update(ref, obs, np.zeros(n, np.uint8) if done is None else done)
        for stacked, off in ((aligned, 0), (shifted, 1)):
            term.fill_(SENTINEL)
            if with_term:
                _ok(gpu, "cl_frame_stack_term", _ptr(stacked, off), _ptr(od), es, cs, _ptr(dd), _ptr(td), tes, tcs,
                    _ptr(term), n, dim, n_stack)
                d = done != 0
                assert np.array_equal(term.cpu().numpy()[d], want_term[d]), (t, off)
            else:
                _ok(gpu, "cl_frame_stack", _ptr(stacked, off), _ptr(od), es, cs, None if dd is None else _ptr(dd),
                    n, dim, n_stack)
        assert np.array_equal(aligned.cpu().numpy(), ref), t
        assert np.array_equal(shifted[1:].view(n, rowlen).cpu().numpy(), ref), t
        assert float(shifted[0]) == SENTINEL


# ---- GAE ------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 33, 4099])
@pytest.mark.parametrize("T", [1, 2, 7, 8, 9, 15, 17, 33])
def test_gae_bit_exact_with_padded_stride(gpu, T, n):
    torch = gpu.torch
    rng = np.random.default_rng(T * 10007 + n)
    stride = n + 29
    for starts_mode in ("zeros", "ones", "random"):
        r = rng.normal(size=(T, n)).astype(np.float32)
        v = rng.normal(size=(T, n)).astype(np.float32)
        starts = {"zeros": np.zeros((T, n)), "ones": np.ones((T, n)),
                  "random": rng.random((T, n)) < 0.3}[starts_mode].astype(np.float32)
        lv = rng.normal(size=n).astype(np.float32)
        ld = (rng.random(n) < 0.5).astype(np.float32)
        adv_ref, ret_ref = S.gae(r, v, starts, lv, ld, 0.99, 0.95)

        def padded(a):
            buf = torch.full((T, stride), float("nan"), dtype=torch.float32, device=gpu.dev)
            buf[:, :n] = torch.as_tensor(a, device=gpu.dev)
            return buf
        rd, vd, sd = padded(r), padded(v), padded(starts)
        lvd, ldd = torch.as_tensor(lv, device=gpu.dev), torch.as_tensor(ld, device=gpu.dev)
        adv = torch.full((T, stride), SENTINEL, dtype=torch.float32, device=gpu.dev)
        ret = torch.full((T, stride), SENTINEL, dtype=torch.float32, device=gpu.dev)
        _ok(gpu, "cl_gae", _ptr(rd), _ptr(vd), _ptr(sd), _ptr(lvd), _ptr(ldd), 0.99, 0.95, T, n, stride, _ptr(adv),
            _ptr(ret))
        a, rt = adv.cpu().numpy(), ret.cpu().numpy()
        assert np.array_equal(a[:, :n], adv_ref), starts_mode
        assert np.array_equal(rt[:, :n], ret_ref), starts_mode
        assert np.all(a[:, n:] == SENTINEL) and np.all(rt[:, n:] == SENTINEL)


# ---- evaluation metrics ---------------------------------------------------------------------------

def _metric_inputs(rng, T, n_err, n_ctrl, n, band):
    """Trajectories that cross the band, plus the edge cases by construction in the first five."""
    t = np.arange(T)[:, None, None]
    tau = rng.uniform(1, max(2, T / 2), size=(1, n_err, n))
    e = rng.uniform(0.5, 5, size=(1, n_err, n)) * band * np.exp(-t / tau) * np.cos(t / 3.0)
    e = e + 0.3 * band * rng.normal(size=(T, n_err, n))
    special = min(n, 5)
    e[:, :, :special] = 0.5 * band
    if n > 0:
        e[::2, :, 0] = band                                  # |e| == band: not an exceedance
        e[1::2, :, 0] = -band
    if n > 1:
        e[0, :, 1] = 2 * band                                # leaves the band at t = 0 only: settles at dt
    if n > 2:
        e[T - 1, 0, 2] = -2 * band                           # component 0 outside at T - 1: NaN for it only
    if n > 3:
        e[T - 1, :, 3] = 2 * band                            # every component: NaN
    if n > 4:
        e[rng.integers(T), rng.integers(n_err), 4] = np.nan  # NaN in err: no exceedance, NaN sums
    u = 50 * rng.normal(size=(T, n_ctrl, n))
    return e, u


def _eval(gpu, e, u, T, n_err, n_ctrl, n, stride, steady, dt, band):
    """cl_eval_metrics on [T][n_err][stride] / [T][n_ctrl][stride] planes; padding columns hold NaN."""
    torch = gpu.torch
    ed = torch.full((T, n_err, stride), float("nan"), dtype=torch.float64, device=gpu.dev)
    ed[:, :, :n] = torch.as_tensor(e, device=gpu.dev)
    ud = torch.full((T, max(n_ctrl, 1), stride), float("nan"), dtype=torch.float64, device=gpu.dev)
    ud[:, :n_ctrl, :n] = torch.as_tensor(u, device=gpu.dev)
    out = torch.full((n, 4), SENTINEL, dtype=torch.float64, device=gpu.dev)
    _ok(gpu, "cl_eval_metrics", _ptr(ed), _ptr(ud), T, n_err, n_ctrl, n, stride, steady, dt, band, _ptr(out))
    return out.cpu().numpy()


def _check_metrics(got, e, u, idx, dt, band, steady):
    want = np.array([metrics_ref(e[:, :, i], u[:, :, i], dt, band, steady) for i in idx]).reshape(len(idx), 4)
    g = got[idx]
    for c in (0, 1, 3):
        _same_metric(g[:, c], want[:, c])
    _same_settling(g[:, 2], want[:, 2])


@pytest.mark.gpu
@pytest.mark.parametrize("n_ctrl", [0, 1, 2, 4])
@pytest.mark.parametrize("n_err", [1, 2, 3, 4])
@pytest.mark.parametrize("T", [1, 2, 3, 5, 63, 64, 65, 257, 2401])
def test_eval_metrics_every_component_count(gpu, T, n_err, n_ctrl):
    """33 trajectories: many segments of the time axis (k_eval_partial's segment remainders)."""
    rng = np.random.default_rng(T * 100 + n_err * 10 + n_ctrl)
    n = 33
    for steady, dt, band in ((0, 0.001, 0.05), (min(1000, T // 2), 0.01, 0.3), (T - 1, 0.004, 0.05)):
        e, u = _metric_inputs(rng, T, n_err, n_ctrl, n, band)
        got = _eval(gpu, e, u, T, n_err, n_ctrl, n, n, steady, dt, band)
        _check_metrics(got, e, u, np.arange(n), dt, band, steady)


@pytest.mark.gpu
@pytest.mark.parametrize("n,stride", [(1, 1), (1000, 1000), (1000, 1037)])
@pytest.mark.parametrize("T", [1, 5, 65, 2401])
def test_eval_metrics_sizes_and_strides(gpu, T, n, stride):
    rng = np.random.default_rng(T + n + stride)
    for n_err, n_ctrl, steady in ((3, 2, min(1000, T // 2)), (4, 0, 0), (1, 4, T - 1)):
        e, u = _metric_inputs(rng, T, n_err, n_ctrl, n, 0.05)
        got = _eval(gpu, e, u, T, n_err, n_ctrl, n, stride, steady, 0.001, 0.05)
        _check_metrics(got, e, u, np.arange(n), 0.001, 0.05, steady)


@pytest.mark.gpu
def test_eval_metrics_single_segment_at_600k(gpu):
    """n >= 512 Ki: the time axis is one segment.  Data generated on the device; the edge cases sit in
    the first trajectories and in the last (partial) block, and a seeded sample of 2,000 is checked."""
    torch = gpu.torch
    T, n_err, n_ctrl, n, dt, band = 65, 4, 4, 600_000, 0.001, 0.05
    g = torch.Generator(device=gpu.dev).manual_seed(5)
    ed = band * 1.5 * torch.randn((T, n_err, n), generator=g, dtype=torch.float64, device=gpu.dev)
    ed *= torch.exp(-torch.arange(T, device=gpu.dev, dtype=torch.float64) / 20.0)[:, None, None]
    ud = 50 * torch.randn((T, n_ctrl, n), generator=g, dtype=torch.float64, device=gpu.dev)
    rng = np.random.default_rng(6)
    e5, _ = _metric_inputs(rng, T, n_err, n_ctrl, 5, band)
    ed[:, :, :5] = torch.as_tensor(e5, device=gpu.dev)
    ed[:, :, n - 5:] = torch.as_tensor(e5, device=gpu.dev)
    for steady in (0, min(1000, T // 2), T - 1):
        out = torch.full((n, 4), SENTINEL, dtype=torch.float64, device=gpu.dev)
        _ok(gpu, "cl_eval_metrics", _ptr(ed), _ptr(ud), T, n_err, n_ctrl, n, n, steady, dt, band, _ptr(out))
        idx = np.unique(np.concatenate([np.arange(5), np.arange(n - 5, n), rng.choice(n, 2000, replace=False)]))
        it = torch.as_tensor(idx, device=gpu.dev)
        e = ed[:, :, it].cpu().numpy()
        u = ud[:, :, it].cpu().numpy()
        got = out[it].cpu().numpy()
        _check_metrics(got, e, u, np.arange(len(idx)), dt, band, steady)


@pytest.mark.gpu
def test_eval_metrics_refusals(gpu):
    torch = gpu.torch
    e = torch.zeros((4, 5, 8), dtype=torch.float64, device=gpu.dev)
    out = torch.zeros((8, 4), dtype=torch.float64, device=gpu.dev)
    for T, ne, nc, ss in ((4, 0, 2, 0), (4, 5, 2, 0), (4, 3, 5, 0), (4, 3, -1, 0), (4, 3, 2, 4), (4, 3, 2, -1)):
        assert _call(gpu, gpu.lib.cl_eval_metrics, _ptr(e), _ptr(e), T, ne, nc, 8, 8, ss, 0.001, 0.05, _ptr(out)) != 0


# ---- the fused policy kernel ---------------------------------------------------------------------

def _modules(seed, scale=1.0):
    import torch
    torch.manual_seed(seed)
    pnet = torch.nn.Sequential(torch.nn.Linear(6, 64), torch.nn.Tanh(), torch.nn.Linear(64, 64), torch.nn.Tanh())
    anet = torch.nn.Linear(64, 2)
    with torch.no_grad():
        for p in list(pnet.parameters()) + list(anet.parameters()):
            p.mul_(scale)
    return pnet, anet


def _policy_batch(kind, n, seed=5):
    import torch
    from gym_lorenz_b200.core import ChaosBatch
    kw = {"eval_mode": True} if kind == "hr_sync" else {}
    b = ChaosBatch(kind, n, seed=seed, autoreset=False, max_episode_steps=None, add_noise=True, **kw)
    b.reset()
    b.step(torch.zeros((n, b.act_dim), device=b.device))
    return b


def _frozen_normalizer(b, clip_obs):
    """A VecNormalize frozen on the statistics of the batch's current observations."""
    from gym_lorenz_b200.rl_ops import DeviceVecNormalize
    vn = DeviceVecNormalize(types.SimpleNamespace(batch=b, num_envs=b.num_envs), training=False, clip_obs=clip_obs)
    obs = b._view(b.obs_planes).double()
    vn.obs_rms.mean.copy_(obs.mean(0))
    vn.obs_rms.var.copy_(obs.var(0))
    return vn


def _run_policy(gpu, kind, n, T, steady, scale, clip_obs, seed=7):
    """evaluate_policy, then every action against mlp_ref on the observations it acted on (normalised
    with the kernel's expression) and every metric against metrics_ref on the recorded streams (all
    trajectories up to 2,000, otherwise a seeded sample plus the last block)."""
    from gym_lorenz_b200.rl_ops import evaluate_policy, pack_policy
    b = _policy_batch(kind, n)
    vn = _frozen_normalizer(b, clip_obs) if clip_obs is not None else None
    packed = pack_policy(_modules(seed, scale), b.device, kind)
    obs0 = b._view(b.obs_planes).clone()
    res = evaluate_policy(b, packed, T, normalize=vn, steady_start=steady, record=("obs", "action"))
    gpu.torch.cuda.synchronize(b.device)
    obs = res["obs"][:, :, :n].permute(0, 2, 1).cpu().numpy()            # [T, n, 6]: after each interval
    seen = np.concatenate([obs0.cpu().numpy()[None], obs[:-1]])            # what each interval acted on
    act = res["action"].cpu().numpy()
    lay = gpu.L.layout(gpu.L.KIND_NAMES[kind])
    z = seen.reshape(T * n, 6)
    clipped = 0.0
    if vn is not None:
        mean, var = vn.obs_rms.mean.cpu().numpy(), vn.obs_rms.var.cpu().numpy()
        zz = (z.astype(np.float64) - mean) / np.sqrt(var + vn.epsilon)
        clipped = float(np.mean(np.abs(zz) > clip_obs))
        z = np.clip(zz, -clip_obs, clip_obs).astype(np.float32)
    pre = mlp_ref(packed.cpu().numpy(), z, 6, 2).reshape(T, n, 2)
    want = np.clip(pre, lay.act_low, lay.act_high)
    assert np.max(np.abs(act - want)) <= 1e-5, float(np.max(np.abs(act - want)))
    sat = (pre > lay.act_high + 1e-5) | (pre < lay.act_low - 1e-5)
    assert np.array_equal(act[sat], want[sat])                           # exactly on the box
    # metrics
    err = obs[:, :, :3]
    if n <= 2000:
        idx = np.arange(n)
    else:
        rng = np.random.default_rng(n)
        idx = np.unique(np.concatenate([rng.choice(n, 2000, replace=False), np.arange(n - (n % 128 or 128), n)]))
    m = {k: res[k].cpu().numpy() for k in ("mae", "rmse", "settling_time", "energy")}
    s = min(1000, T // 2) if steady is None else steady
    want_m = np.array([metrics_ref(err[:, i], act[:, i], 0.001, 0.05, s) for i in idx]).reshape(len(idx), 4)
    for c, k in ((0, "mae"), (1, "rmse"), (3, "energy")):
        _same_metric(m[k][idx], want_m[:, c])
    _same_settling(m["settling_time"][idx], want_m[:, 2])
    b.close()
    return clipped, float(np.mean(sat))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["hr_sync", "pmsm_sync"])
def test_policy_clips_observations_and_actions(gpu, kind):
    """A VecNormalize with clip_obs = 0.5 and weights scaled by 5: both clips are active."""
    clipped, saturated = _run_policy(gpu, kind, 1000, 24, None, 5.0, 0.5)
    assert clipped > 0.05, clipped
    assert saturated >= 0.10, saturated


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["hr_sync", "pmsm_sync"])
@pytest.mark.parametrize("T,steady", [(1, 0), (5, 0), (5, 4), (64, 63)])
def test_policy_short_windows(gpu, kind, T, steady):
    _run_policy(gpu, kind, 1000, T, steady, 1.0, 10.0)


@pytest.mark.gpu
@pytest.mark.parametrize("n,block", [(33, 32), (65530, 64), (18939, 128)])
def test_policy_block_sizes_with_partial_blocks(gpu, n, block):
    sms = gpu.torch.cuda.get_device_properties(gpu.dev).multi_processor_count
    if sms == 148:
        assert policy_block(n, sms) == block
    _run_policy(gpu, "hr_sync", n, 8, None, 1.0, 10.0)
    _run_policy(gpu, "pmsm_sync", n, 8, 0, 5.0, 0.5)
