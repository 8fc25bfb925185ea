"""The batch I/O kernels of io_kernels.cu -- K4 polyfit (templated and generic), polyeval, K5 rollout and the roadmap
front end -- against high-precision references, through both entry layouts: the host entries (per-problem rows) and
the device entries (field-major device buffers, the layout bench_io.py feeds them).

References (CPU):
  least squares   the exact solution c* of min ||V c - y||_2 for the Vandermonde matrix V of the double xs (mpmath
                  QR at 60 digits).  A backward-stable QR solve satisfies, per fit,
                      ||c - c*||_2 <= C u kappa(V) (||c*||_2 + kappa(V) ||r*||_2 / ||V||_2),   r* = y - V c*,
                  with u = 2^-53; C = 16 here, asserted where kappa(V) <= 1e12 (past that the bound says nothing).
  polyeval        the exact sum c_i x^i (mpmath.fsum at 60 digits), within (2 ncoef + 2) u sum |c_i x^i|.
  rollout step    one exact Euler step (long double) from the kernel's OWN previous state, so errors do not pile up
                  over H; per component x, y: 8u (|x'| + |v dt|), psi: 4u (|psi'| + |v delta dt / Lf|), v: 2u (|v'| + |a dt|).
                  These rest on the 2-ulp maximum error of double-precision sin / cos / sincos in the accuracy table of
                  the CUDA C++ Programming Guide (the math headers refer to it), and on one rounding per + - * /.
The CPU tests hold the C port (oracle/mpc_oracle.c, Eigen's operation order) to the same bounds and show that the
bounds reject a single-precision computation.  The GPU tests cover every accepted polyfit shape, ragged blocks, the
argument limits of every entry, and the isolation of the problems of a batch."""
import contextlib
import ctypes
import functools

import mpmath
import numpy as np
import pytest
import torch

import oracle_bindings as ob

U = 2.0 ** -53
C_LS = 16.0
KAPPA_MAX = 1e12
ERR_ARG = -1                     # B200MPC_ERR_ARG
SHAPES = [(m, order) for m in range(2, 17) for order in range(1, min(7, m - 1) + 1)]   # every (m, order) accepted
SQUARE = [(m, m - 1) for m in range(2, 9)]
X_RANGES = ((-1.0, 1.0), (0.0, 12.0), (-100.0, 100.0), (50.0, 60.0))   # U(-1,1), sorted road-like, wide, offset
SENTINEL = -7.25e300             # the tail of every output buffer
TAIL = 37

assert len(SHAPES) == 84


# ------------------------------------------------------------------------------------------------ references
def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def assert_bitwise(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape
    bad = bits(a) != bits(b)
    assert not bad.any(), f"{bad.sum()} elements differ, first at {np.argwhere(bad)[0]}: {a[bad][0]!r} vs {b[bad][0]!r}"


def fit_inputs(B, m, seed):
    """Row b draws its xs from X_RANGES[b % 4] (the road-like kind sorted) and ys = 2 sin(3t) + noise, t the xs mapped
    to [-1, 1]."""
    rng = np.random.default_rng(seed)
    xs, ys = np.empty((B, m)), np.empty((B, m))
    kind = np.arange(B) % 4
    for k, (lo, hi) in enumerate(X_RANGES):
        sel = kind == k
        x = rng.uniform(lo, hi, (sel.sum(), m))
        if k == 1:
            x = np.sort(x, axis=1)
        xs[sel] = x
        ys[sel] = 2.0 * np.sin(3.0 * ((x - lo) / (hi - lo) * 2.0 - 1.0)) + 0.05 * rng.standard_normal(x.shape)
    return xs, ys


def exact_fit(xs, ys, order):
    """(c*, ||r*||_2) of the least-squares problem of the exact Vandermonde matrix of the double xs, 60 digits."""
    with mpmath.workdps(60):
        V = mpmath.matrix([[mpmath.mpf(float(x)) ** i for i in range(order + 1)] for x in xs])
        c, r = mpmath.qr_solve(V, mpmath.matrix([mpmath.mpf(float(y)) for y in ys]))
        return np.array([float(ci) for ci in c]), float(r)


class FitRef:
    """Exact answer c* and tolerance C u kappa (||c*|| + kappa ||r*|| / ||V||) of one fit; only computed (and the fit
    only asserted) where kappa <= KAPPA_MAX.  c_star / r_norm: the exact answer when the caller knows it."""

    def __init__(self, xs, ys, order, c_star=None, r_norm=None):
        V = np.vander(np.asarray(xs, dtype=np.float64), order + 1, increasing=True)
        self.kappa = float(np.linalg.cond(V))
        self.asserted = self.kappa <= KAPPA_MAX
        if not self.asserted:
            return
        if c_star is None:
            c_star, r_norm = exact_fit(xs, ys, order)
        self.c_star = c_star
        self.tol = C_LS * U * self.kappa * (np.linalg.norm(c_star) + self.kappa * r_norm / np.linalg.norm(V, 2))

    def error(self, c):
        return float(np.linalg.norm(np.asarray(c, dtype=np.float64) - self.c_star))


@functools.lru_cache(maxsize=None)
def fit_refs(B, m, order, seed, rows):
    xs, ys = fit_inputs(B, m, seed)
    return {b: FitRef(xs[b], ys[b], order) for b in rows}


def check_fits(refs, fits, what="fit"):
    """Asserts every fit whose kappa is within the limit against its exact answer; returns how many were asserted."""
    n = 0
    for b, ref in refs.items():
        if not ref.asserted:
            continue
        err = ref.error(fits[b])
        assert err <= ref.tol, f"{what} row {b}: ||c - c*|| = {err:.3e} > {ref.tol:.3e} (kappa {ref.kappa:.2e})"
        n += 1
    return n


def exact_polyeval(c, x):
    """(sum c_i x^i, sum |c_i x^i|) at 60 digits."""
    with mpmath.workdps(60):
        X, p, terms = mpmath.mpf(float(x)), mpmath.mpf(1), []
        for ci in c:
            terms.append(mpmath.mpf(float(ci)) * p)
            p *= X
        return mpmath.fsum(terms), mpmath.fsum([abs(t) for t in terms])


def polyeval_ratios(coeffs, x, y):
    """|y - exact| / ((2 ncoef + 2) u sum |c_i x^i|) per problem (0 where exact, inf where the bound is 0 and missed)."""
    n = coeffs.shape[1]
    out = np.empty(len(x))
    for b in range(len(x)):
        s, mag = exact_polyeval(coeffs[b], x[b])
        with mpmath.workdps(60):
            err = abs(mpmath.mpf(float(y[b])) - s)
        tol = (2 * n + 2) * U * float(mag)
        out[b] = 0.0 if err == 0 else (float(err) / tol if tol > 0 else np.inf)
    return out


if np.finfo(np.longdouble).nmant >= 63:
    def _hp_context():
        return contextlib.nullcontext()
    _hp = functools.partial(np.asarray, dtype=np.longdouble)
    _cos, _sin = np.cos, np.sin
else:                                       # long double is double here: the same arithmetic on mpmath objects
    def _hp_context():
        return mpmath.workdps(40)
    _hp = np.frompyfunc(mpmath.mpf, 1, 1)
    _cos, _sin = np.frompyfunc(mpmath.cos, 1, 1), np.frompyfunc(mpmath.sin, 1, 1)


def rollout_step_ratios(state4, act, traj, dt, Lf):
    """Per step and component, |kernel step - exact Euler step from the kernel's own previous state| / tolerance.
    state4 (B, 4), act (B, H, 2), traj (B, H, 4) -> (B, H, 4); 0 where exact, inf where the tolerance is 0 and missed."""
    prev = np.concatenate([state4[:, None, :], traj[:, :-1, :]], axis=1)
    with _hp_context():
        x, y, psi, v = (_hp(prev[..., k]) for k in range(4))
        delta, a = _hp(act[..., 0]), _hp(act[..., 1])
        dt_, Lf_ = _hp(np.float64(dt)), _hp(np.float64(Lf))
        vdt, turn, adt = v * dt_, v * delta * dt_ / Lf_, a * dt_
        exact = (x + vdt * _cos(psi), y + vdt * _sin(psi), psi + turn, v + adt)
        tol = (8 * U * (abs(exact[0]) + abs(vdt)), 8 * U * (abs(exact[1]) + abs(vdt)),
               4 * U * (abs(exact[2]) + abs(turn)), 2 * U * (abs(exact[3]) + abs(adt)))
        out = np.empty(traj.shape)
        for k in range(4):
            err = np.asarray(abs(_hp(traj[..., k]) - exact[k]), dtype=np.float64)
            t = np.asarray(tol[k], dtype=np.float64)
            with np.errstate(divide="ignore", invalid="ignore"):
                out[..., k] = np.where(err == 0, 0.0, err / t)
    return out


def rollout_inputs(B, H, seed):
    rng = np.random.default_rng(seed)
    st = np.column_stack([rng.uniform(-50, 50, B), rng.uniform(-50, 50, B), rng.uniform(-4, 4, B), rng.uniform(-5, 40, B)])
    act = np.stack([rng.uniform(-0.44, 0.44, (B, H)), rng.uniform(-1, 1, (B, H))], axis=2)
    return st, act


def dyadic_centerline(n_wp, seed=5):
    """x = k / 2 and y on a 2^-10 grid: differences to a dyadic pose and their squares are exact."""
    rng = np.random.default_rng(seed)
    k = np.arange(n_wp)
    y = 3.0 * np.sin(0.05 * k) + 0.1 * rng.standard_normal(n_wp)
    return np.column_stack([0.5 * k, np.round(y * 1024) / 1024])


def window_refs(poses, cl):
    """Index of the first 6-point window (first nearest point, clamped to n_wp - 6) and its vehicle-frame points at psi 0."""
    d = (poses[:, None, 0] - cl[None, :, 0]) ** 2 + (poses[:, None, 1] - cl[None, :, 1]) ** 2
    best = np.minimum(np.argmin(d, axis=1), len(cl) - 6)   # np.argmin returns the first minimum
    w = best[:, None] + np.arange(6)
    return best, cl[w, 0] - poses[:, None, 0], cl[w, 1] - poses[:, None, 1]


# ------------------------------------------------------------------------------------------------ CPU: the references
@pytest.mark.parametrize("kind", range(4), ids=["unit", "road", "wide", "offset"])
def test_c_port_polyfit_meets_the_least_squares_bound(kind):
    """Eigen's operation order (the C port) satisfies the bound on every accepted shape; the bound is not vacuous: the
    port's answer moved by twice the tolerance fails it, and so does a fit in single precision where kappa <= 1e6 (past
    that, the kappa^2 ||r*|| term of the bound admits even single precision on noisy data)."""
    asserted = single = 0
    for m, order in SHAPES:
        xs, ys = fit_inputs(24, m, 1000 + 17 * m + order)
        rows = tuple(range(kind, 24, 4))
        refs = fit_refs(24, m, order, 1000 + 17 * m + order, rows)
        port = {b: ob.port_polyfit(xs[b], ys[b], order) for b in rows}
        asserted += check_fits(refs, port, what=f"port ({m},{order})")
        rng = np.random.default_rng(m * 8 + order)
        for b, ref in refs.items():
            if not ref.asserted:
                continue
            e = rng.standard_normal(order + 1)
            assert ref.error(port[b] + 2 * ref.tol * e / np.linalg.norm(e)) > ref.tol
            if ref.kappa <= 1e6:
                V32 = np.vander(xs[b].astype(np.float32), order + 1, increasing=True)
                c32 = np.linalg.lstsq(V32, ys[b].astype(np.float32), rcond=None)[0].astype(np.float64)
                assert ref.error(c32) > ref.tol, f"single-precision fit passes ({m},{order}) row {b}"
                single += 1
    assert asserted >= 200 and single >= 50, (asserted, single)   # of 504 fits


def test_c_port_polyeval_meets_the_bound():
    rng = np.random.default_rng(3)
    for n in (1, 2, 3, 4, 7, 8, 16, 64):
        coeffs = rng.standard_normal((64, n))
        x = rng.uniform(-1.5, 1.5, 64) * (40.0 if n <= 4 else 1.0)
        y = np.array([ob.port_polyeval(coeffs[b], x[b]) for b in range(64)])
        r = polyeval_ratios(coeffs, x, y)
        assert r.max() <= 1.0, (n, r.max())
        # moved by twice the tolerance, the same values fail
        s = np.array([float(exact_polyeval(coeffs[b], x[b])[1]) for b in range(64)])
        assert (polyeval_ratios(coeffs, x, y + 2 * (2 * n + 2) * U * s) > 1.0).all()


def test_c_port_global_kinematic_meets_the_step_bound():
    st, act = rollout_inputs(2000, 1, 4)
    st[::7, 2] *= 100.0            # large headings: the full range of sin / cos
    for dt, Lf in ((0.3, 2.0), (0.05, 2.67)):
        nxt = np.array([ob.port_kinematic(st[b], act[b, 0], dt, Lf) for b in range(len(st))])
        r = rollout_step_ratios(st, act, nxt[:, None, :], dt, Lf)
        assert r.max() <= 1.0, r.max()
        # the same step with single-precision sin / cos fails the x / y bounds
        psi32 = st[:, 2].astype(np.float32)
        c32, s32 = np.cos(psi32).astype(np.float64), np.sin(psi32).astype(np.float64)
        bad = nxt.copy()
        bad[:, 0] = st[:, 0] + st[:, 3] * c32 * dt
        bad[:, 1] = st[:, 1] + st[:, 3] * s32 * dt
        rb = rollout_step_ratios(st, act, bad[:, None, :], dt, Lf)[:, 0, :2].max(axis=1)
        assert (rb > 1.0).mean() > 0.9, (rb > 1.0).mean()


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def dev():
    import udacitympc_b200 as mp
    m = mp.MPC(device=0)
    yield Device(m)
    m.close()


def fm(a):
    """(B, K) rows -> a field-major (K, B) device tensor; 1-D arrays as they are."""
    a = np.asarray(a, dtype=np.float64)
    return torch.from_numpy(np.ascontiguousarray(a.T if a.ndim == 2 else a)).cuda()


def out_buffer(n):
    return torch.full((n + TAIL,), SENTINEL, dtype=torch.float64, device="cuda")


class Device:
    """The four device entries on field-major torch buffers.  Every call must launch exactly one kernel and leave the
    sentinel tail of its output buffers untouched."""

    def __init__(self, mpc):
        from udacitympc_b200 import api
        import udacitympc_b200 as mp
        self.mp, self.mpc, self.lib = mp, mpc, api.load_library()

    def call(self, name, *args, outs=()):
        torch.cuda.synchronize()
        n0 = self.mpc.launch_count()
        rc = getattr(self.lib, name)(self.mpc.handle, *args, None)
        assert rc == 0, self.lib.b200mpc_last_error().decode()
        torch.cuda.synchronize()
        assert self.mpc.launch_count() == n0 + 1
        res = []
        for buf, n in outs:
            tail = buf[n:].cpu().numpy()
            assert (tail == SENTINEL).all(), f"{name} wrote past its output"
            res.append(buf[:n].cpu().numpy())
        return res

    def polyfit(self, xs, ys, order):
        B, m = xs.shape
        n = order + 1
        dx, dy, out = fm(xs), fm(ys), out_buffer(n * B)
        (c,) = self.call("b200mpc_polyfit_batch_device", B, dx.data_ptr(), dy.data_ptr(), m, order, out.data_ptr(), outs=[(out, n * B)])
        return c.reshape(n, B).T

    def polyeval(self, coeffs, x):
        B, n = coeffs.shape
        dc, dx, out = fm(coeffs), fm(x), out_buffer(B)
        return self.call("b200mpc_polyeval_batch_device", B, dc.data_ptr(), n, dx.data_ptr(), out.data_ptr(), outs=[(out, B)])[0]

    def rollout(self, st, act, dt, Lf):
        B, H = act.shape[:2]
        ds, da, out = fm(st), fm(act.reshape(B, 2 * H)), out_buffer(4 * H * B)
        (r,) = self.call("b200mpc_rollout_batch_device", B, H, ds.data_ptr(), da.data_ptr(), ctypes.c_double(dt), ctypes.c_double(Lf),
                         out.data_ptr(), outs=[(out, 4 * H * B)])
        return r.reshape(4 * H, B).T.reshape(B, H, 4)

    def roadmap(self, poses, cl):
        B = len(poses)
        dp, dc = fm(poses), torch.from_numpy(np.ascontiguousarray(cl, dtype=np.float64)).cuda()
        st, cf = out_buffer(6 * B), out_buffer(4 * B)
        s, c = self.call("b200mpc_roadmap_reference_batch_device", B, dp.data_ptr(), dc.data_ptr(), len(cl), st.data_ptr(), cf.data_ptr(),
                         outs=[(st, 6 * B), (cf, 4 * B)])
        return s.reshape(6, B).T, c.reshape(4, B).T

    # the host entries (per-problem rows), through the package's wrappers
    def polyfit_host(self, xs, ys, order):
        return self.mp.polyfit_batch(xs, ys, order, mpc=self.mpc)

    def polyeval_host(self, coeffs, x):
        return self.mp.polyeval_batch(coeffs, x, mpc=self.mpc)

    def rollout_host(self, st, act, dt, Lf):
        return self.mp.rollout_batch(st, act, dt, Lf, mpc=self.mpc)

    def roadmap_host(self, poses, cl):
        return self.mp.roadmap_reference_batch(poses, cl, mpc=self.mpc)


FIT_ROWS = tuple(range(12)) + (125, 126, 127, 128)   # both block ends of B = 129


@pytest.mark.gpu
@pytest.mark.parametrize("m,order", SHAPES)
def test_polyfit_every_shape(dev, m, order):
    """B = 129 (a ragged 128-thread block) and B = 1: host and device entries agree bitwise, every checked fit meets the
    least-squares bound against the exact answer and agrees with the C port within the sum of the two tolerances."""
    seed = 2000 + 17 * m + order
    xs, ys = fit_inputs(129, m, seed)
    host = dev.polyfit_host(xs, ys, order)
    assert_bitwise(dev.polyfit(xs, ys, order), host)
    refs = fit_refs(129, m, order, seed, FIT_ROWS)
    check_fits(refs, host, what=f"({m},{order})")
    port = {b: ob.port_polyfit(xs[b], ys[b], order) for b in FIT_ROWS}
    for b, ref in refs.items():
        if ref.asserted:
            assert np.linalg.norm(host[b] - port[b]) <= 2 * ref.tol, (b, host[b], port[b])
    for b in (0, 128):     # a batch of one computes what the same row does in a batch
        assert_bitwise(dev.polyfit(xs[b:b + 1], ys[b:b + 1], order)[0], host[b])
        assert_bitwise(dev.polyfit_host(xs[b:b + 1], ys[b:b + 1], order)[0], host[b])


@pytest.mark.gpu
@pytest.mark.parametrize("m,order", [(6, 3), (16, 7)])
def test_polyfit_large_batch(dev, m, order):
    xs, ys = fit_inputs(4097, m, 31 + m)
    host = dev.polyfit_host(xs, ys, order)
    assert_bitwise(dev.polyfit(xs, ys, order), host)
    rows = tuple(range(0, 4097, 257)) + (4095, 4096)
    assert check_fits(fit_refs(4097, m, order, 31 + m, rows), host) > 0


@pytest.mark.gpu
def test_polyfit_edges(dev):
    """ys = 0 gives exactly zero coefficients; ys sampled from a polynomial of degree <= order with dyadic coefficients
    at small integer xs is recovered within the bound with r* = 0; xs scaled to ~1e-3 and ~1e3."""
    rng = np.random.default_rng(8)
    exact_n = scaled_n = 0
    for m, order in SHAPES:
        xs = np.stack([rng.choice(np.arange(-8.0, 9.0), m, replace=False) for _ in range(5)])
        zero = np.zeros_like(xs)
        for fit in (dev.polyfit(xs, zero, order), dev.polyfit_host(xs, zero, order)):
            assert (fit == 0).all(), (m, order, fit)
        deg = rng.integers(0, order + 1, 5)
        k = rng.integers(-8, 9, (5, order + 1)) * (np.arange(order + 1)[None, :] <= deg[:, None])
        ys = np.array([[sum(int(k[b, i]) * int(x) ** i for i in range(order + 1)) / 4 for x in xs[b]] for b in range(5)])
        fits = dev.polyfit(xs, ys, order)
        assert_bitwise(fits, dev.polyfit_host(xs, ys, order))
        refs = {b: FitRef(xs[b], ys[b], order, c_star=k[b] / 4.0, r_norm=0.0) for b in range(5)}
        exact_n += check_fits(refs, fits, what=f"polynomial data ({m},{order})")
        for scale in (1e-3, 1e3):
            sx, sy = fit_inputs(4, m, 5000 + m * 8 + order)
            sx = sx / np.abs(sx).max(axis=1, keepdims=True) * scale
            fits = dev.polyfit(sx, sy, order)
            assert_bitwise(fits, dev.polyfit_host(sx, sy, order))
            scaled_n += check_fits({b: FitRef(sx[b], sy[b], order) for b in range(4)}, fits, what=f"scale {scale} ({m},{order})")
    assert exact_n >= 5 * 70 and scaled_n >= 40, (exact_n, scaled_n)


@pytest.mark.gpu
@pytest.mark.parametrize("m,order", SQUARE)
def test_polyfit_square_systems_interpolate(dev, m, order):
    """m = order + 1: the last reflector is the identity (rr == 1, the tail <= DBL_MIN branch) and r* = 0."""
    xs, ys = fit_inputs(129, m, 77 + m)
    fits = dev.polyfit(xs, ys, order)
    assert_bitwise(fits, dev.polyfit_host(xs, ys, order))
    assert check_fits(fit_refs(129, m, order, 77 + m, tuple(range(129))), fits) >= 48


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 3, 4, 7, 8, 16, 64])
def test_polyeval(dev, n):
    """Host rows and device field-major (d_coeffs[i*B+b]) agree bitwise and meet the bound; x = 0 returns c_0, and so
    does ncoef = 1; at x = +-2 with ncoef = 64 every power is exact and so, with coefficients k_i 2^-i, is the sum."""
    rng = np.random.default_rng(40 + n)
    for B in (1, 255, 256, 257, 4097):
        coeffs = rng.standard_normal((B, n))
        x = rng.uniform(-1.5, 1.5, B) * (40.0 if n <= 4 else 1.0)
        y = dev.polyeval(coeffs, x)
        assert_bitwise(y, dev.polyeval_host(coeffs, x))
        r = polyeval_ratios(coeffs, x, y)
        assert r.max() <= 1.0, (B, r.max(), int(r.argmax()))
    coeffs = rng.standard_normal((300, n))
    x = np.zeros(300)
    x[::2] = rng.uniform(-3, 3, 150)
    y = dev.polyeval(coeffs, x)
    assert_bitwise(y[1::2], coeffs[1::2, 0])
    if n == 1:
        assert_bitwise(y, coeffs[:, 0])
    if n == 64:
        k = rng.integers(-3, 4, (300, 64))
        c = k * 2.0 ** -np.arange(64)
        x = np.where(np.arange(300) % 2 == 0, 2.0, -2.0)
        expect = np.array([sum(int(k[b, i]) * (1 if x[b] > 0 or i % 2 == 0 else -1) for i in range(64)) for b in range(300)], dtype=np.float64)
        assert_bitwise(dev.polyeval(c, x), expect)
        assert_bitwise(dev.polyeval_host(c, x), expect)


@pytest.mark.gpu
@pytest.mark.parametrize("H", [1, 2, 25, 1024, 4096])
def test_rollout(dev, H):
    """Every step within the local bound of an exact Euler step; host and device bitwise (H <= 1024, the host entry's
    limit); for H <= 25 the whole trajectory within 1e-12 (relative to magnitude) of the C port's loop; dt = 0 returns
    the input state at every step, bitwise."""
    B = 257 if H <= 1024 else 300
    st, act = rollout_inputs(B, H, 50 + H)
    st[::5, 2] *= 50.0
    for dt in (0.3, 0.05, 0.0):
        for Lf in (2.0, 2.67):
            traj = dev.rollout(st, act, dt, Lf)
            if H <= 1024:
                assert_bitwise(traj, dev.rollout_host(st, act, dt, Lf))
            r = rollout_step_ratios(st, act, traj, dt, Lf)
            assert r.max() <= 1.0, (dt, Lf, r.max(), np.unravel_index(r.argmax(), r.shape))
            if dt == 0.0:
                assert_bitwise(traj, np.broadcast_to(st[:, None, :], traj.shape))
            if H <= 25 and dt > 0:
                for b in range(0, B, 8):
                    s = st[b]
                    for t in range(H):
                        s = ob.port_kinematic(s, act[b, t], dt, Lf)
                        assert (np.abs(traj[b, t] - s) <= 1e-12 * np.maximum(1.0, np.abs(s))).all(), (b, t, traj[b, t], s)


ROADMAP_SIZES = [6, 7, 246, 3072, 3073, 12000]   # 3073: the first centre line over 48 KB of shared memory


@pytest.mark.gpu
@pytest.mark.parametrize("n_wp", ROADMAP_SIZES)
def test_roadmap_front_end(dev, n_wp):
    from test_gpu_parity import roadmap_reference_oracle
    cl = dyadic_centerline(n_wp)
    rng = np.random.default_rng(n_wp)
    B = 300
    k = rng.integers(0, n_wp, B)
    pos = np.round((cl[k] + rng.normal(scale=0.7, size=(B, 2))) * 1024) / 1024
    poses = np.column_stack([pos, rng.uniform(-3, 3, B), rng.uniform(0, 40, B)])
    # poses exactly at the first and the last points: the window clamps to n_wp - 6
    ends = np.r_[0:min(6, n_wp), n_wp - 6:n_wp]
    poses[:len(ends), :2] = cl[ends]
    # exact ties in squared distance between points k and k+1 whose windows differ; the first must win
    ties = rng.integers(0, n_wp - 6, 40) if n_wp >= 7 else np.zeros(0, dtype=int)
    t0 = len(ends)
    poses[t0:t0 + len(ties), :2] = (cl[ties] + cl[ties + 1]) / 2
    st, cf = dev.roadmap(poses, cl)
    sh, ch = dev.roadmap_host(poses, cl)
    assert_bitwise(st, sh)
    assert_bitwise(cf, ch)
    # general psi: the numpy restatement, within its tolerance relative to the coefficients (cte = c0 and
    # epsi = -atan(c1) move no more than the coefficients do)
    for b in range(0, B, 3):
        so, co = roadmap_reference_oracle(poses[b], cl)
        tol = 1e-9 * max(1.0, np.abs(co).max())
        np.testing.assert_allclose(cf[b], co, rtol=0, atol=tol)
        np.testing.assert_allclose(st[b], so, rtol=0, atol=tol)
    # state: (0, 0, 0, v, c0, -atan(c1))
    assert (st[:, :3] == 0).all()
    assert_bitwise(st[:, 3], poses[:, 3])
    assert_bitwise(st[:, 4], cf[:, 0])
    for b in range(B):
        with mpmath.workdps(60):
            e = -mpmath.atan(mpmath.mpf(float(cf[b, 1])))
            assert abs(mpmath.mpf(float(st[b, 5])) - e) <= 2 * np.spacing(abs(float(e))), b
    # psi = 0 with dyadic coordinates: the vehicle-frame points are exact, so the fit meets the least-squares bound
    poses[:, 2] = 0.0
    st0, cf0 = dev.roadmap(poses, cl)
    assert_bitwise(cf0, dev.roadmap_host(poses, cl)[1])
    best, lx, ly = window_refs(poses, cl)
    assert (best[:len(ends)] == np.minimum(ends, n_wp - 6)).all()
    refs = {b: FitRef(lx[b], ly[b], 3) for b in range(0, B, 5)}
    refs.update({b: FitRef(lx[b], ly[b], 3) for b in range(t0 + len(ties))})
    assert check_fits(refs, cf0) == len(refs)
    for j, i in enumerate(ties):
        b = t0 + j
        assert best[b] == i
        second = FitRef(cl[i + 1:i + 7, 0] - poses[b, 0], cl[i + 1:i + 7, 1] - poses[b, 1], 3)
        assert second.error(cf0[b]) > 100 * refs[b].tol, "the tie does not tell the two windows apart"


# ------------------------------------------------------------------------------------------------ GPU: isolation
def _poison(a, rows, value):
    a = a.copy()
    a[rows] = value
    return a


@pytest.mark.gpu
def test_problems_are_isolated(dev):
    """For each kernel: the reversed batch gives the reversed results bitwise, and problems holding NaN or inf leave
    every other problem bitwise equal to a clean batch."""
    B = 257
    bad = np.array([0, 3, 128, 200, 256])
    good = np.setdiff1d(np.arange(B), bad)
    rev = slice(None, None, -1)

    for m, order in ((6, 3), (9, 5)):
        xs, ys = fit_inputs(B, m, 90 + m)
        c = dev.polyfit(xs, ys, order)
        assert_bitwise(dev.polyfit(xs[rev], ys[rev], order), c[rev])
        xb = _poison(xs, bad[:3], np.nan)
        yb = _poison(ys, bad[3:], np.inf)
        assert_bitwise(dev.polyfit(xb, yb, order)[good], c[good])

    coeffs, x = np.random.default_rng(1).standard_normal((B, 7)), np.random.default_rng(2).uniform(-1, 1, B)
    y = dev.polyeval(coeffs, x)
    assert_bitwise(dev.polyeval(coeffs[rev], x[rev]), y[rev])
    assert_bitwise(dev.polyeval(_poison(coeffs, bad[:3], np.nan), _poison(x, bad[3:], np.inf))[good], y[good])

    st, act = rollout_inputs(B, 9, 3)
    tr = dev.rollout(st, act, 0.1, 2.67)
    assert_bitwise(dev.rollout(st[rev], act[rev], 0.1, 2.67), tr[rev])
    assert_bitwise(dev.rollout(_poison(st, bad[:3], np.nan), _poison(act, bad[3:], np.inf), 0.1, 2.67)[good], tr[good])

    cl = dyadic_centerline(246)
    rng = np.random.default_rng(4)
    poses = np.column_stack([cl[rng.integers(0, 246, B)] + rng.normal(size=(B, 2)), rng.uniform(-3, 3, B), rng.uniform(0, 40, B)])
    s, c = dev.roadmap(poses, cl)
    s2, c2 = dev.roadmap(poses[rev], cl)
    assert_bitwise(s2, s[rev])
    assert_bitwise(c2, c[rev])
    pb = _poison(_poison(poses, bad[:3], np.nan), bad[3:], np.inf)
    s3, c3 = dev.roadmap(pb, cl)
    assert_bitwise(s3[good], s[good])
    assert_bitwise(c3[good], c[good])


# ------------------------------------------------------------------------------------------------ GPU: entry semantics
@pytest.mark.gpu
def test_device_entries_run_on_the_callers_stream(dev):
    """Each entry queues its kernel on the stream it is given: behind a delay and the copy of its inputs on that stream,
    it reads the inputs and its outputs are complete once that stream synchronises."""
    lib, h = dev.lib, dev.mpc.handle
    B = 333
    xs, ys = fit_inputs(B, 6, 9)
    coeffs, x = np.random.default_rng(5).standard_normal((B, 5)), np.random.default_rng(6).uniform(-1, 1, B)
    st, act = rollout_inputs(B, 3, 7)
    cl = dyadic_centerline(246)
    poses = np.column_stack([cl[np.arange(B) % 240], np.zeros(B), np.full(B, 10.0)])
    src = [fm(a) for a in (xs, ys, coeffs, x, st, act.reshape(B, 6), poses)]
    dst = [torch.zeros_like(t) for t in src]
    dcl = torch.from_numpy(cl).cuda()
    cf, y, tr, s6, c4 = (torch.zeros(n, B, dtype=torch.float64, device="cuda") for n in (4, 1, 12, 6, 4))
    stream = torch.cuda.Stream()
    torch.cuda.synchronize()
    n0 = dev.mpc.launch_count()
    with torch.cuda.stream(stream):
        torch.cuda._sleep(20_000_000)
        for d, s in zip(dst, src):
            d.copy_(s)
    sp = ctypes.c_void_p(stream.cuda_stream)
    dx, dy, dc, dxv, ds, da, dpo = (t.data_ptr() for t in dst)
    assert lib.b200mpc_polyfit_batch_device(h, B, dx, dy, 6, 3, cf.data_ptr(), sp) == 0
    assert lib.b200mpc_polyeval_batch_device(h, B, dc, 5, dxv, y.data_ptr(), sp) == 0
    assert lib.b200mpc_rollout_batch_device(h, B, 3, ds, da, 0.3, 2.0, tr.data_ptr(), sp) == 0
    assert lib.b200mpc_roadmap_reference_batch_device(h, B, dpo, dcl.data_ptr(), 246, s6.data_ptr(), c4.data_ptr(), sp) == 0
    assert dev.mpc.launch_count() == n0 + 4
    stream.synchronize()
    assert_bitwise(cf.cpu().numpy().T, dev.polyfit_host(xs, ys, 3))
    assert_bitwise(y.cpu().numpy()[0], dev.polyeval_host(coeffs, x))
    assert_bitwise(tr.cpu().numpy().T.reshape(B, 3, 4), dev.rollout_host(st, act, 0.3, 2.0))
    sh, ch = dev.roadmap_host(poses, cl)
    assert_bitwise(s6.cpu().numpy().T, sh)
    assert_bitwise(c4.cpu().numpy().T, ch)


def _host_ptrs(*arrays):
    return [a.ctypes.data_as(ctypes.POINTER(ctypes.c_double)) for a in arrays]


@pytest.mark.gpu
def test_empty_batches_launch_nothing(dev):
    lib, h = dev.lib, dev.mpc.handle
    n0 = dev.mpc.launch_count()
    assert lib.b200mpc_polyfit_batch_device(h, 0, None, None, 6, 3, None, None) == 0
    assert lib.b200mpc_polyeval_batch_device(h, 0, None, 4, None, None, None) == 0
    assert lib.b200mpc_rollout_batch_device(h, 0, 5, None, None, 0.3, 2.0, None, None) == 0
    assert lib.b200mpc_roadmap_reference_batch_device(h, 0, None, None, 246, None, None, None) == 0
    assert lib.b200mpc_polyfit_batch(h, 0, None, None, 6, 3, None) == 0
    assert lib.b200mpc_polyeval_batch(h, 0, None, 4, None, None) == 0
    assert lib.b200mpc_rollout_batch(h, 0, 5, None, None, 0.3, 2.0, None) == 0
    assert lib.b200mpc_roadmap_reference_batch(h, 0, None, None, 246, None, None) == 0
    assert dev.mpc.launch_count() == n0


@pytest.mark.gpu
def test_argument_limits(dev):
    """Each rejected argument returns B200MPC_ERR_ARG and launches nothing; the accepted maxima run."""
    lib, h = dev.lib, dev.mpc.handle
    B = 3
    size = 4 * 4097 * B + 2 * 12001   # in bounds for every call below
    src, dst = torch.zeros(size, dtype=torch.float64, device="cuda"), torch.empty(size, dtype=torch.float64, device="cuda")
    p, q = src.data_ptr(), dst.data_ptr()
    hb = [np.zeros(4 * 1025 * B + 2 * 12001) for _ in range(3)]
    h0, h1, h2 = _host_ptrs(*hb)
    nan = float("nan")
    rejected = [
        ("b200mpc_polyfit_batch_device", (B, p, p, 1, 1, q, None)),
        ("b200mpc_polyfit_batch_device", (B, p, p, 17, 7, q, None)),
        ("b200mpc_polyfit_batch_device", (B, p, p, 6, 0, q, None)),
        ("b200mpc_polyfit_batch_device", (B, p, p, 12, 8, q, None)),
        ("b200mpc_polyfit_batch_device", (B, p, p, 5, 5, q, None)),
        ("b200mpc_polyfit_batch", (B, h0, h1, 1, 1, h2)),
        ("b200mpc_polyfit_batch", (B, h0, h1, 17, 7, h2)),
        ("b200mpc_polyfit_batch", (B, h0, h1, 6, 0, h2)),
        ("b200mpc_polyfit_batch", (B, h0, h1, 12, 8, h2)),
        ("b200mpc_polyfit_batch", (B, h0, h1, 5, 5, h2)),
        ("b200mpc_polyeval_batch_device", (B, p, 0, p, q, None)),
        ("b200mpc_polyeval_batch_device", (B, p, 65, p, q, None)),
        ("b200mpc_polyeval_batch", (B, h0, 0, h1, h2)),
        ("b200mpc_polyeval_batch", (B, h0, 65, h1, h2)),
        ("b200mpc_rollout_batch_device", (B, 0, p, p, 0.3, 2.0, q, None)),
        ("b200mpc_rollout_batch_device", (B, 4097, p, p, 0.3, 2.0, q, None)),
        ("b200mpc_rollout_batch_device", (B, 5, p, p, 0.3, 0.0, q, None)),
        ("b200mpc_rollout_batch_device", (B, 5, p, p, 0.3, nan, q, None)),
        ("b200mpc_rollout_batch", (B, 0, h0, h1, 0.3, 2.0, h2)),
        ("b200mpc_rollout_batch", (B, 1025, h0, h1, 0.3, 2.0, h2)),
        ("b200mpc_rollout_batch", (B, 5, h0, h1, 0.3, 0.0, h2)),
        ("b200mpc_rollout_batch", (B, 5, h0, h1, 0.3, nan, h2)),
        ("b200mpc_roadmap_reference_batch_device", (B, p, p, 5, q, q, None)),
        ("b200mpc_roadmap_reference_batch_device", (B, p, p, 12001, q, q, None)),
        ("b200mpc_roadmap_reference_batch", (B, h0, h1, 5, h2, h2)),
        ("b200mpc_roadmap_reference_batch", (B, h0, h1, 12001, h2, h2)),
    ]
    torch.cuda.synchronize()
    n0 = dev.mpc.launch_count()
    for name, args in rejected:
        assert getattr(lib, name)(h, *args) == ERR_ARG, (name, args)
    assert dev.mpc.launch_count() == n0
    accepted = [
        ("b200mpc_polyfit_batch_device", (B, p, p, 16, 7, q, None)),
        ("b200mpc_polyfit_batch", (B, h0, h1, 16, 7, h2)),
        ("b200mpc_polyeval_batch_device", (B, p, 64, p, q, None)),
        ("b200mpc_polyeval_batch", (B, h0, 64, h1, h2)),
        ("b200mpc_rollout_batch_device", (B, 4096, p, p, 0.3, 2.0, q, None)),
        ("b200mpc_rollout_batch", (B, 1024, h0, h1, 0.3, 2.0, h2)),
        ("b200mpc_roadmap_reference_batch_device", (B, p, p, 12000, q, q, None)),
        ("b200mpc_roadmap_reference_batch", (B, h0, h1, 12000, h2, h2)),
    ]
    for name, args in accepted:
        assert getattr(lib, name)(h, *args) == 0, (name, lib.b200mpc_last_error().decode())
    torch.cuda.synchronize()
    assert dev.mpc.launch_count() == n0 + len(accepted)


@pytest.mark.gpu
def test_polyeval_beyond_two_to_the_31_elements(dev):
    """ncoef * B > 2^31: the element offsets of the field-major coefficient array need 64 bits (about 18 GB)."""
    n, B = 64, 2 ** 25 + 1
    free, _ = torch.cuda.mem_get_info()
    if free < 40 * 2 ** 30:
        pytest.skip(f"needs 40 GB of free device memory, {free / 2 ** 30:.0f} GB free")
    g = torch.Generator(device="cuda").manual_seed(12)
    coeffs = torch.empty((n, B), dtype=torch.float64, device="cuda").uniform_(-1.0, 1.0, generator=g)
    x = torch.empty(B, dtype=torch.float64, device="cuda").uniform_(-1.2, 1.2, generator=g)
    y = out_buffer(B)
    try:
        (yv,) = dev.call("b200mpc_polyeval_batch_device", B, coeffs.data_ptr(), n, x.data_ptr(), y.data_ptr(), outs=[(y, B)])
        rows = np.r_[0:8, B - 64:B]
        c = coeffs[:, torch.from_numpy(rows).cuda()].cpu().numpy().T
        r = polyeval_ratios(c, x.cpu().numpy()[rows], yv[rows])
        assert r.max() <= 1.0, r.max()
    finally:
        del coeffs, x, y
        torch.cuda.empty_cache()
