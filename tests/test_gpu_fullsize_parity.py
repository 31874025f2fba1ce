"""Parity against the CPU oracle AT THE SIZES BASELINE.json QUOTES (VERDICT r1 "missing #2"): not properties of the GPU
against itself, but the oracle's numbers -- computed live where that takes seconds, and from committed oracle runs
(tests/golden/*_oracle.json, generator scripts beside them) where the serial CPU path needs minutes to an hour.

  config #2  cg! laplace_matrix(Float64, 256, 3): first 20 iterations vs a live oracle.c run; the whole solve to
             reltol = sqrt(eps) (638 iterations) vs tests/golden/cg_laplace3d_256_oracle.json            src/cg.jl:43-66
  config #4  cg! laplace_matrix(Float64, 512, 3) on one GPU: the whole solve (about 1000 iterations) vs
             tests/golden/cg_laplace3d_512_oracle.json: iteration count, every residual, x at 4096 positions, ||x||
  config #3  gmres!(restart = 30) CGS and DGKS, one cycle on advection_dominated(256) vs a live oracle.gmres_
                                                                                                       src/gmres.jl:57-106
  config #5  lobpcg block 16 fp32 laplace 256^3, 4 steps vs tests/golden/lobpcg_laplace3d_256_f32_oracle.json
                                                                                                       src/lobpcg.jl:692-749
Tolerances are written at each assert; fp64 paths: 1e-10 relative (BASELINE.json north_star)."""
import json
import os

import numpy as np
import pytest

from bench import rhs_slab

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TOL = 1e-10


@pytest.fixture(scope="module")
def isb():
    import iterativesolvers_jl_b200 as m
    m.default_context()
    return m


def _golden(name):
    path = os.path.join(GOLDEN, name)
    if not os.path.exists(path):
        pytest.skip(f"{name} not generated (see the make_*_golden.py script beside it)")
    with open(path) as f:
        return json.load(f)


def _bench_rhs(n):
    b = rhs_slab(0, n)
    b /= np.sqrt(float(np.sum(b * b)))      # fixed summation order: np.dot's depends on the host's BLAS thread count
    return b


def _cg_vs_golden(isb, N):
    g = _golden(f"cg_laplace3d_{N}_oracle.json")
    ctx = isb.default_context()
    n = N ** 3
    assert g["n"] == n
    A = isb.B200CSR.laplacian(N, 3)
    b = isb.DeviceArray.from_numpy(ctx, _bench_rhs(n))
    x = isb.DeviceArray.zeros(ctx, n)
    x, h = isb.cg_(x, A, b, initially_zero=True, log=True, maxiter=20000)       # reltol = sqrt(eps): the reference default
    res, ref = h["resnorm"], np.array(g["resnorm"])
    assert h.isconverged and g["isconverged"]
    assert h.niters == g["iters"] and h.mvps == g["mvps"], (h.niters, g["iters"])
    hist_err = float(np.max(np.abs(res - ref) / ref))
    xs = x.numpy()
    idx, xref = np.array(g["x_sample_index0"]), np.array(g["x_samples"])
    x_err = float(np.linalg.norm(xs[idx] - xref) / np.linalg.norm(xref))
    nrm_err = abs(float(np.sqrt(np.dot(xs, xs))) - g["x_norm2"]) / g["x_norm2"]
    print(f"cg! {N}^3 vs oracle: {h.niters} iterations, history max rel diff {hist_err:.2e}, x rel err (sampled) "
          f"{x_err:.2e}, ||x|| rel diff {nrm_err:.2e}")
    assert hist_err <= TOL and x_err <= TOL and nrm_err <= TOL, (hist_err, x_err, nrm_err)
    for v in (b, x):
        v.free()
    A.close()


def test_cg_256cubed_first_iterations_vs_live_oracle(isb, oracle):
    """20 iterations of cg! at config #2's size against oracle.c run now (pins the committed golden files' generator too)."""
    N, its = 256, 20
    ctx = isb.default_context()
    O = oracle.laplace_matrix(np.float64, N, 3, base=1)
    bh = _bench_rhs(O.n)
    xo, ho = oracle.cg_csc_c(np.zeros(O.n), O, bh, initially_zero=True, maxiter=its, reltol=0.0)
    A = isb.B200CSR.laplacian(N, 3)
    x = isb.DeviceArray.zeros(ctx, O.n)
    x, h = isb.cg_(x, A, isb.DeviceArray.from_numpy(ctx, bh), initially_zero=True, log=True, maxiter=its, reltol=0.0)
    assert h.niters == ho.niters == its
    hist_err = float(np.max(np.abs(h["resnorm"] - ho["resnorm"]) / ho["resnorm"]))
    x_err = float(np.linalg.norm(x.numpy() - xo) / np.linalg.norm(xo))
    g = _golden("cg_laplace3d_256_oracle.json")
    assert np.array_equal(np.array(g["resnorm"][:its]), ho["resnorm"])      # the committed run is this oracle's output
    print(f"cg! 256^3, {its} iterations vs live oracle: history {hist_err:.2e}, x {x_err:.2e}")
    assert hist_err <= TOL and x_err <= TOL
    A.close()


def test_cg_256cubed_full_solve_vs_oracle_golden(isb):
    _cg_vs_golden(isb, 256)


def test_cg_512cubed_full_solve_vs_oracle_golden(isb):
    """the headline problem: the drift SURVEY section 7 'hard part 3' said to watch, measured."""
    _cg_vs_golden(isb, 512)


@pytest.mark.parametrize("orth", ["cgs", "dgks"])
def test_gmres_256cubed_one_cycle_vs_live_oracle(isb, oracle, orth):
    """config #3: one restart cycle of 30 inner iterations.  Tolerance 1e-9 on the residual history (each of the 30
    Gram-Schmidt steps sums 16.7 M products in a different order than the CPU; measured 2.6e-10 .. 4.9e-10) and 1e-6 on x
    (x = V y with y from the 30 x 30 triangular solve of the rotated Hessenberg matrix, which amplifies the perturbation of
    H by its condition number on this advection-dominated operator; measured 5.2e-8 with the three-kernel
    orthogonalisation, 3.1e-7 with the fused one -- same algorithm, another summation order)."""
    ctx = isb.default_context()
    N = 256
    cp, rv, nz, shape, b = isb.advection_dominated(N, 1000.0, base=1)
    n = shape[0]
    O = oracle.CSC(n, n, cp, rv, nz, 1)
    xo, ho = oracle.gmres_(np.zeros(n), O, b, restart=30, maxiter=30, orth_meth=orth, initially_zero=True, log=True,
                           reltol=0.0)
    A = isb.B200CSR.from_csc_arrays(cp, rv, nz, shape, base=1)
    xd = isb.DeviceArray.zeros(ctx, n)
    xd, h = isb.gmres_(xd, A, isb.DeviceArray.from_numpy(ctx, b), restart=30, maxiter=30, orth_meth=orth,
                       initially_zero=True, log=True, reltol=0.0)
    assert h.niters == ho.niters == 30 and h.mvps == ho.mvps
    hist_err = float(np.max(np.abs(h["resnorm"] - ho["resnorm"]) / ho["resnorm"]))
    x_err = float(np.linalg.norm(xd.numpy() - xo) / np.linalg.norm(xo))
    print(f"gmres!(30, {orth}) advection 256^3 one cycle vs live oracle: history {hist_err:.2e}, x {x_err:.2e}")
    assert hist_err <= 1e-9 and x_err <= 1e-6
    xd.free()
    A.close()


def test_lobpcg_256cubed_fp32_four_steps_vs_oracle_golden(isb):
    """config #5: the per-iteration Ritz values of the fp32 engine (3xTF32 tensor-pipe products, fp32 accumulation) against
    the oracle's fp32 numpy run.  Tolerance: 1e-4 relative on every Ritz value of every step (fp32 Gram matrices over
    16.7 M rows; VERDICT r1 next-step 2), 5e-2 relative on the residual norms (differences of nearly equal fp32 numbers)."""
    g = _golden("lobpcg_laplace3d_256_f32_oracle.json")
    ctx = isb.default_context()
    N, bs = g["grid"], g["blocksize"]
    A = isb.B200CSR.laplacian(N, 3, np.float32)
    X0 = np.random.default_rng(g["seed"]).random((N ** 3, bs), dtype=np.float32)
    r = isb.lobpcg(A, False, isb.DeviceArray.from_numpy(ctx, X0), maxiter=g["steps"], tol=0.0, log=True)
    assert r.iterations == g["iterations_reported"] and len(r.trace) == len(g["trace"])
    worst_l, worst_r = 0.0, 0.0
    for (it, rn, lam), t in zip(r.trace, g["trace"]):
        assert it == t["iteration"]
        lo, ro = np.array(t["ritz_values"]), np.array(t["residual_norms"])
        worst_l = max(worst_l, float(np.max(np.abs(np.asarray(lam, dtype=np.float64) - lo) / np.abs(lo))))
        worst_r = max(worst_r, float(np.max(np.abs(np.asarray(rn, dtype=np.float64) - ro) / np.abs(ro))))
    print(f"lobpcg 256^3 fp32 bs=16, {g['steps']} steps vs oracle: Ritz values {worst_l:.2e}, residual norms {worst_r:.2e}")
    assert worst_l <= 1e-4 and worst_r <= 5e-2
    A.close()
