"""-m "not gpu": pins of the oracle TNLP (oracle/ref_build/mpc_tnlp.cpp, driven by the reference's own Ipopt 3.12.7 +
MUMPS binaries in oracle/_ref) to the problem FG_eval defines (mpc_to_line/solution/MPC.cpp:45-140).

The reference gets its derivatives from CppAD (MPC.cpp:241-243), which is absent here, so the TNLP supplies closed-form
derivatives.  Ipopt's own derivative checker (IpTNLPAdapter.cpp, option `derivative_test second-order`) compares them
with finite differences of eval_f / eval_g -- the two functions that restate MPC.cpp:57-76 and :88-138 line by line --
at a randomly perturbed point: no mismatch line may appear."""
import os

import numpy as np
import pytest

import oracle_bindings as ob
from conftest import golden

needs_ref = pytest.mark.skipif(not ob.ref_available(), reason="oracle/_ref (reference binaries) not built here")


def _derivative_check(state, coeffs, tmp_path, tag, **kw):
    out = os.path.join(str(tmp_path), f"ipopt_{tag}.txt")
    # forward differences of an objective of size ~4e4 (25 x (v - 40)^2): with Ipopt's default step 1e-8 the cancellation
    # noise alone is ~4e-4 of a gradient entry, so the step is 1e-6 and the tolerance 1e-3 (a wrong or missing term shows
    # up as an O(1) relative error, see test_derivative_checker_is_not_vacuous)
    opts = "\n".join(["derivative_test second-order", "derivative_test_perturbation 1e-6", "derivative_test_tol 1e-3",
                      "point_perturbation_radius 0.5", f"output_file {out}", "file_print_level 4", "max_iter 2"])
    ob.ref_solve(state, coeffs, opts=opts, **kw)
    text = open(out).read()
    assert "Starting derivative checker for first derivatives" in text, text[:400]
    assert "Starting derivative checker for second derivatives" in text
    assert "No errors detected by derivative checker" in text, [l for l in text.splitlines() if "error" in l.lower() or "*" in l][:20]
    assert "Derivative checker detected" not in text
    return text


@needs_ref
def test_ipopt_derivative_checker_finds_no_mismatch_degree1(tmp_path):
    g = golden("line_256.npz")
    for b in (0, 7, 100):
        _derivative_check(g["states"][b], g["coeffs"][b], tmp_path, f"line{b}")


@needs_ref
def test_ipopt_derivative_checker_finds_no_mismatch_degree3_and_weights(tmp_path):
    g = golden("roadmap_256.npz")
    for b in (0, 31):
        _derivative_check(g["states"][b], g["fit"][b], tmp_path, f"road{b}")
    _derivative_check(g["states"][5], g["fit"][5], tmp_path, "roadw", weights=[3.0, 0.5, 0.2, 10.0, 2.0, 50.0, 4.0])
    _derivative_check(g["states"][9], g["fit"][9], tmp_path, "roadN10", N=10, dt=0.08, Lf=2.0, ref_v=25.0)


@needs_ref
def test_derivative_checker_is_not_vacuous(tmp_path):
    """The same check flags a wrong derivative: with finite differences compared at an absurd tolerance the checker
    reports errors, so 'No errors detected' above means something."""
    g = golden("roadmap_256.npz")
    out = os.path.join(str(tmp_path), "ipopt_bad.txt")
    opts = "\n".join(["derivative_test second-order", "derivative_test_tol 1e-14", "point_perturbation_radius 0.5",
                      f"output_file {out}", "file_print_level 4", "max_iter 1"])
    ob.ref_solve(g["states"][0], g["fit"][0], opts=opts)
    assert "Derivative checker detected" in open(out).read()


@needs_ref
def test_unit_weights_entry_is_the_unweighted_problem():
    g = golden("line_256.npz")
    for b in range(3):
        a = ob.ref_solve(g["states"][b], g["coeffs"][b])
        w = ob.ref_solve(g["states"][b], g["coeffs"][b], weights=[1.0] * 7)
        assert a["iters"] == w["iters"] == g["iters"][b] and np.array_equal(a["x"], w["x"]) and np.array_equal(a["x"], g["x"][b])


def test_weighted_goldens_are_reproduced_by_the_binaries_and_by_the_port():
    """The stored results of the reference's binaries with non-unit weights: the port reproduces them, and so do the
    binaries themselves where they are built."""
    g = golden("weights_64.npz")
    for name in ("a", "b"):
        w = g[f"w_{name}"]
        p = ob.default_params(w_cte=w[0], w_epsi=w[1], w_v=w[2], w_delta=w[3], w_a=w[4], w_ddelta=w[5], w_da=w[6])
        for kind in ("line", "road"):
            st, cf = g[f"{kind}_states"], g[f"{kind}_coeffs"]
            for b in (0, 13, 31):
                if ob.ref_available():
                    r = ob.ref_solve(st[b], cf[b], weights=w)
                    assert np.array_equal(r["x"], g[f"{kind}_{name}_x"][b])
                o = ob.port_solve(st[b], cf[b], params=p)
                assert o["status"] == 0 and o["iters"] == g[f"{kind}_{name}_iters"][b]
                np.testing.assert_allclose(o["x"], g[f"{kind}_{name}_x"][b], rtol=0, atol=1e-9)
                assert abs(o["obj"] - g[f"{kind}_{name}_obj"][b]) <= 1e-9 * abs(o["obj"])
