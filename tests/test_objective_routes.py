"""The per-expert hyper-parameter objectives (`sgp_bcm_nll`: regression BCM NLL + gradient, `sgp_laplace_nll`: Laplace
classification objective) against the fp64 oracle on every dispatch route, at both sides of each route boundary.

How a BCM evaluation is routed (csrc/bcm_nll.cu `launch_bcm_nll`, csrc/api.cu `sgp_bcm_nll`), n_max = largest expert:
  register kernel <2,4>   one non-Eye term, n_max <= 64                  (rb = (n_max+15)/16 sixteen-column blocks)
  register kernel <3,6>   one non-Eye term, 65 <= n_max <= 96
  register kernel <4,7>   one non-Eye term, 97 <= n_max <= 112
  register kernel <4,8>   one non-Eye term, 113 <= n_max <= 128, if its shared memory fits (not: RBF at d >= 94)
  smem kernel, staged     >= 2 non-Eye terms, or one term the register kernel does not take, while
                          bcm_nll_smem_bytes(n_max) + 8 n_max (d|1) <= 113 KB (rows copied to shared memory)
  smem kernel, global     the same kernel with the rows read from global memory (always for n_max >= 128)
  general path            bcm_nll_smem_bytes(n_max) > 227 KB, i.e. n_max >= 169 (last_bcm_path() == 1)
The gradient sweeps ARD dimensions 16 at a time (DCH), once per non-Eye term when any term carries ARD betas.
Laplace (csrc/laplace.cu) has one kernel, for n_max <= 117; the rows come from global memory when they do not fit.

Data: X ~ U[0,1)^d with a different scale per column and ARD betas distinct per dimension (so that a dimension mix-up
changes the numbers), an Eye term of 1e-2 .. 3e-2.  Every case asserts max cond(K_e) <= 1e6 before comparing.

Gates (the ones of tests/test_gpu_parity.py, with scales that cannot be near zero):
  NLL       |nll - nll0| <= 1e-9 * sum_e (1/2 |y_e' alpha_e| + 1/2 |log det K_e|)
  gradient  per group (all trainable scales; each term's betas; each sigma): max|g - g0| <= 1e-8 * max|g0| of the group
  Laplace   |v - v0| <= 1e-9 * sum_e |v0_e| (-log Z_e > 0); gradient groups as above; modes f to 1e-9
On a B200 (1000 W limit) every case measured <= 6e-14 on every gate.
"""
import numpy as np
import pytest

import oracle
import spark_gp_b200 as sg
from oracle.classification import classification_likelihood_and_gradient
from spark_gp_b200 import _native as N

TOL_NLL, TOL_GRAD, TOL_F, MAX_COND = 1e-9, 1e-8, 1e-9, 1e6


@pytest.fixture(scope="module")
def eng():
    e = sg.ProjectedProcessEngine(0)
    yield e
    e.close()


# ---------------- data, kernels, oracle -------------------------------------------------------------------------------
def _betas(d, reverse=False):
    b = np.linspace(0.3, 1.2, d) * np.sqrt(6.0 / d)
    return b[::-1] * 0.8 if reverse else b


def _sigma(d):
    return 0.9 * np.sqrt(d / 6.0)


def _experts(sizes, d, seed, labels=False):
    """Experts as contiguous blocks of the given sizes: (X, y, offsets)."""
    rng = np.random.default_rng(seed)
    n = int(np.sum(sizes))
    X = rng.random((n, d)) * np.linspace(1.6, 0.4, d)
    w = rng.standard_normal(d) / np.sqrt(d)
    f = np.sin(4.0 * X @ w) + 0.3 * np.cos(3.0 * X[:, 0])
    if labels:
        y = (f + 0.3 * rng.standard_normal(n) > np.median(f)).astype(np.float64)
    else:
        y = f + 0.1 * rng.standard_normal(n)
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    return X, y, off


# A kernel spec builds the same kernel from the product DSL (M = spark_gp_b200) or the oracle (M = oracle).
def ard(M, d):
    return 1.3 * M.ARDRBFKernel(_betas(d)) + M.WhiteNoiseKernel(0.02, 0, 1)


def ard_const_eye(M, d):
    return 1.2 * M.ARDRBFKernel(_betas(d)) + M.const(1e-2) * M.EyeKernel()


def rbf_noise(M, d):
    return M.Scalar(1.4).between(0).and_(30) * M.RBFKernel(_sigma(d), 1e-6, 100) + M.WhiteNoiseKernel(0.02, 0, 1)


def rbf_const(M, d):
    return M.RBFKernel(_sigma(d)) + M.const(3e-2) * M.EyeKernel()


def ard_72_hypers(M, d):            # d = 71: one trainable scale + 71 betas = MAX_HYPERS
    return 1.1 * M.ARDRBFKernel(_betas(d)) + M.const(2e-2) * M.EyeKernel()


def two_ard_eye_between(M, d):      # flattened terms: ARD, Eye, ARD -> the second ARD is non-Eye term 1 (flat_of)
    return 0.7 * M.ARDRBFKernel(_betas(d)) + M.WhiteNoiseKernel(0.02, 0, 1) + 1.9 * M.ARDRBFKernel(_betas(d, True))


def ard_plus_rbf(M, d):
    return 0.9 * M.ARDRBFKernel(_betas(d)) + 0.5 * M.RBFKernel(_sigma(d)) + M.const(2e-2) * M.EyeKernel()


def four_terms_nested(M, d):        # kMaxTerms non-Eye terms under two levels of trainable scalars
    return (1.2 * (0.8 * M.ARDRBFKernel(_betas(d)) + 0.5 * M.RBFKernel(_sigma(d)))
            + 0.9 * (1.1 * M.ARDRBFKernel(_betas(d, True)) + 0.6 * M.RBFKernel(0.7 * _sigma(d)))
            + M.const(2e-2) * M.EyeKernel())


def _oracle_experts(spec, X, y, off):
    d = X.shape[1]
    return [(y[off[e]:off[e + 1]], spec(oracle, d).set_training_vectors(X[off[e]:off[e + 1]]))
            for e in range(len(off) - 1)]


def _conditioning(experts, theta):
    """(max_e cond(K_e), sum_e 1/2 |y_e' K_e^-1 y_e| + 1/2 |log det K_e|): the NLL gate's scale."""
    cond, scale = 0.0, 0.0
    for ye, k in experts:
        K = k.set_hyperparameters(theta).training_kernel()
        cond = max(cond, float(np.linalg.cond(K)))
        scale += 0.5 * abs(float(ye @ np.linalg.solve(K, ye))) + 0.5 * abs(np.linalg.slogdet(K)[1])
    return cond, scale


def _groups(kernel):
    """Hyper-parameter indices per gradient group: all trainable scales, each term's ARD betas, each RBF sigma."""
    groups = {}
    for i, h in enumerate(kernel.hyper_descriptors()):
        if h["kind"] == N.SGP_HYPER_SCALE:
            key = "scales"
        elif h["kind"] == N.SGP_HYPER_ARD_BETA:
            key = "betas[term %d]" % h["term"]
        else:
            key = "sigma[%d]" % i
        groups.setdefault(key, []).append(i)
    return groups


def _compare(label, v, g, v0, g0, scale, groups):
    """Asserts the NLL and gradient gates; prints the measured errors."""
    e_v = abs(v - v0) / scale
    errs = {}
    for key, idx in groups.items():
        ref = np.abs(g0[idx]).max()
        diff = np.abs(g[idx] - g0[idx]).max()
        errs[key] = diff / ref if ref > 0 else diff
    print("%-44s value %.2e  " % (label, e_v) + "  ".join("%s %.2e" % kv for kv in errs.items()))
    assert len(g) == len(g0)
    assert e_v <= TOL_NLL, (label, e_v)
    for key, e in errs.items():
        assert e <= TOL_GRAD, (label, key, e)


# ---------------- BCM: one case per route and boundary ----------------------------------------------------------------
# (sizes, d, kernel spec, last_bcm_path).  Each comment names the route and the mistake in the CUDA source it would catch.
BCM_CASES = [
    # reg <2,4>: 1x1 matrices, all padding; a pivot or padding slip in the sweep, a non-zero beta gradient without pairs
    pytest.param([1] * 6, 3, ard, 0, id="reg24-n1"),
    # reg <2,4> at its top (64) with ragged padding; d = 17: the second ARD chunk (k0 = 16, kn = 1)
    pytest.param([63, 64, 61, 64, 63], 17, ard, 0, id="reg24-n63_64-d17-2chunks"),
    # reg <3,6> at its bottom (65): the rb threshold 64/65; d = 16: exactly one chunk (Q taken from D)
    pytest.param([64, 65, 65, 60], 16, ard, 0, id="reg36-n64_65-d16-1chunk"),
    # reg <3,6> at its top (96): RBF sigma (Q summed over all d) with a trainable Eye scale
    pytest.param([96, 95, 96], 40, rbf_noise, 0, id="reg36-n96-rbf-d40"),
    # reg <4,7> at its bottom (97): the rb threshold 96/97; d = 33: three chunks, the last one of one dimension
    pytest.param([97, 90, 97], 33, ard, 0, id="reg47-n97-d33-3chunks"),
    # reg <4,7> at its top (112); d = 64: four full chunks (k0 = 0, 16, 32, 48)
    pytest.param([112, 110, 112], 64, ard, 0, id="reg47-n112-d64-4chunks"),
    # reg <4,8> at its bottom (113): the rb threshold 112/113
    pytest.param([113, 100, 113], 5, ard, 0, id="reg48-n113-d5"),
    # reg <4,8> at its top (128) with MAX_HYPERS = 72 hyper-parameters (5 chunks, the last of 7 dimensions)
    pytest.param([128, 127, 128], 71, ard_72_hypers, 0, id="reg48-n128-d71-72hypers"),
    # reg <4,8> smem exceeds 227 KB at d = 100 -> smem kernel, rows from global memory (xld = d, not d|1)
    pytest.param([128, 120, 128], 100, rbf_const, 0, id="smem_global-n128-rbf-d100-reg_too_big"),
    # one term at 129: past the register kernel (the 128/129 threshold) -> smem kernel, rows from global
    pytest.param([129, 129, 120], 7, ard, 0, id="smem_global-n129-d7"),
    # one term at 168: the largest on-chip expert (ex_ltl_inplace column blocks, 8 (n(n+1)+3n+33) <= 227 KB)
    pytest.param([168] * 7 + [150], 64, ard, 0, id="smem_global-n168-d64"),
    # one term at 169: the general path (global-memory LU), identity padding of the smaller expert
    pytest.param([169, 160, 169], 20, ard, 1, id="general-n169-d20"),
    # two ARD terms with an Eye term between them: flat_of, the n_terms x chunks sweeps (term 1's betas at ts = 1)
    pytest.param([100, 98, 100], 20, two_ard_eye_between, 0, id="smem_staged-two_ard_eye_between-d20"),
    # four non-Eye terms (kMaxTerms) under nested trainable scalars: the SCALE coefficients of each term
    pytest.param([80, 77, 80], 6, four_terms_nested, 0, id="smem_staged-four_terms_nested-d6"),
    pytest.param([169, 150, 169], 6, four_terms_nested, 1, id="general-four_terms_nested-n169-d6"),
    # two terms at 104, d = 40: staged rows would exceed 113 KB -> rows from global, three chunks per term
    pytest.param([104, 103, 104], 40, ard_plus_rbf, 0, id="smem_global-two_terms-n104-d40"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("sizes,d,spec,path", BCM_CASES)
def test_bcm_route_vs_oracle(eng, sizes, d, spec, path):
    """sgp_bcm_nll on the route named in the id vs the oracle's BCM objective over the same blocks; a second evaluation
    must be bit-identical (the per-expert rows are reduced in a fixed order)."""
    X, y, off = _experts(sizes, d, seed=1000 + int(np.sum(sizes)) + d)
    k = spec(sg, d)
    theta = k.getHyperparameters()
    experts = _oracle_experts(spec, X, y, off)
    nll0, g0 = oracle.regression.bcm_objective(experts, theta)
    cond, scale = _conditioning(experts, theta)
    assert cond <= MAX_COND, cond
    eng.experts_upload(X, y, off)
    nll, g = eng.bcm_nll(k)
    assert eng.last_bcm_path() == path
    _compare("bcm %s (cond %.1e)" % (eng.last_bcm_path(), cond), nll, g, nll0, g0, scale, _groups(k))
    nll2, g2 = eng.bcm_nll(k)
    assert nll2 == nll and np.array_equal(g2, g)


@pytest.mark.gpu
def test_bcm_mixed_sizes_one_launch(eng):
    """Experts of 1 .. 128 points in one launch (n_max = 128: reg <4,8>, every expert padded differently): the total
    matches the oracle; each expert evaluated alone (on the route its own size selects) matches the oracle's value for
    that expert; the singles add up to the batched total within the same gates.  Catches identity padding leaking
    between experts of different sizes and a per-expert offset mix-up."""
    sizes, d = [1, 2, 16, 17, 63, 64, 65, 100, 128], 17
    X, y, off = _experts(sizes, d, seed=2024)
    k = ard(sg, d)
    theta = k.getHyperparameters()
    groups = _groups(k)
    experts = _oracle_experts(ard, X, y, off)
    nll0, g0 = oracle.regression.bcm_objective(experts, theta)
    cond, scale = _conditioning(experts, theta)
    assert cond <= MAX_COND, cond
    eng.experts_upload(X, y, off)
    nll, g = eng.bcm_nll(k)
    assert eng.last_bcm_path() == 0
    _compare("mixed batch", nll, g, nll0, g0, scale, groups)
    v_sum, g_sum = 0.0, np.zeros_like(g)
    for e, n_e in enumerate(sizes):
        s = slice(off[e], off[e + 1])
        eng.experts_upload(X[s], y[s], [0, n_e])
        v1, g1 = eng.bcm_nll(k)
        v0e, g0e = oracle.regression.bcm_objective([experts[e]], theta)
        _compare("mixed single n=%d" % n_e, v1, g1, v0e, g0e, _conditioning([experts[e]], theta)[1], groups)
        v_sum += v1
        g_sum += g1
    _compare("mixed sum of singles vs batch", v_sum, g_sum, nll, g, scale, groups)


@pytest.mark.gpu
def test_objective_limits_rejected(eng):
    """5 non-Eye terms (kMaxTerms = 4), 73 hyper-parameters (MAX_HYPERS = 72) and a Laplace expert of 118 points (the
    kernel holds n_max <= 117) are refused with SGP_E_BADARG; the accepted side of each limit is pinned above/below."""
    X, y, off = _experts([10, 12], 72, seed=5)
    eng.experts_upload(X, y, off)
    five = (sg.RBFKernel(1.0) + sg.RBFKernel(1.1) + sg.RBFKernel(1.2) + sg.RBFKernel(1.3) + sg.RBFKernel(1.4)
            + sg.const(1e-2) * sg.EyeKernel())
    assert len([t for t in five.flatten() if t["type"] != N.SGP_TERM_EYE]) == 5
    with pytest.raises(ValueError, match="non-Eye"):
        eng.bcm_nll(five)
    k73 = 1.0 * sg.ARDRBFKernel(_betas(72)) + sg.const(1e-2) * sg.EyeKernel()
    assert k73.numberOfHyperparameters() == 73
    with pytest.raises(ValueError, match="hyper-parameters"):
        eng.bcm_nll(k73)
    X, y, off = _experts([118, 40], 3, seed=6, labels=True)
    eng.experts_upload(X, y, off)
    with pytest.raises(ValueError, match="117"):
        eng.laplace_nll(ard_const_eye(sg, 3), 1e-6)


# ---------------- Laplace ---------------------------------------------------------------------------------------------
LAPLACE_CASES = [
    # 1-point experts: no pairs, the beta gradient is exactly zero
    pytest.param([1] * 5, 3, ard_const_eye, id="n1-d3"),
    # 64/65 ragged: uneven padding; d = 17: the second ARD chunk of the sweep
    pytest.param([64, 65, 65, 64], 17, ard_const_eye, id="n64_65-d17-2chunks"),
    # the largest expert the kernel takes (117): rows from global memory; d = 33: three chunks
    pytest.param([117, 116, 117], 33, ard_const_eye, id="n117-rows_from_global-d33"),
    # two ARD terms with an Eye term between them (flat_of, one sweep per term and chunk)
    pytest.param([90, 88], 20, two_ard_eye_between, id="two_ard_eye_between-d20"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("sizes,d,spec", LAPLACE_CASES)
def test_laplace_route_vs_oracle(eng, sizes, d, spec):
    """Two consecutive evaluations at two thetas (the second warm-starts from the modes of the first, as the
    reference's cached experts do): -log Z, its gradient and every expert's mode f vs the oracle."""
    tol = 1e-6
    X, y, off = _experts(sizes, d, seed=3000 + int(np.sum(sizes)) + d, labels=True)
    experts = _oracle_experts(spec, X, y, off)
    fs = [np.zeros(len(ye)) for ye, _ in experts]
    k = spec(sg, d)
    groups = _groups(k)
    theta0 = k.getHyperparameters()
    eng.experts_upload(X, y, off)
    for theta in (theta0, theta0 * np.where(np.arange(len(theta0)) % 2 == 0, 1.3, 0.8)):
        cond, _ = _conditioning(experts, theta)
        assert cond <= MAX_COND, cond
        v0, g0, scale = 0.0, 0.0, 0.0
        for (ye, ke), f in zip(experts, fs):
            ve, ge = classification_likelihood_and_gradient(ye, f, ke, theta, tol)
            v0 += ve
            g0 = g0 + ge
            scale += abs(ve)
        v, g = eng.laplace_nll(spec(sg, d).setHyperparameters(theta), tol)
        _compare("laplace (cond %.1e)" % cond, v, g, v0, g0, scale, groups)
        f_ref = np.concatenate(fs)
        e_f = np.abs(eng.experts_f(len(X)) - f_ref).max() / max(1.0, np.abs(f_ref).max())
        print("%-44s modes %.2e" % ("laplace", e_f))
        assert e_f <= TOL_F


# ---------------- the oracle itself, on the new kernel structures (CPU) ----------------------------------------------
@pytest.mark.parametrize("spec,d", [(two_ard_eye_between, 5), (four_terms_nested, 4), (ard, 17)],
                         ids=["two_ard_eye_between", "four_terms_nested", "ard-d17"])
def test_oracle_bcm_gradient_vs_finite_differences(spec, d):
    """The GPU gates above are only as good as the oracle: its analytic BCM gradient must match central finite
    differences of its own objective for the kernel structures the route tests use."""
    X, y, off = _experts([23, 30], d, seed=77)
    experts = _oracle_experts(spec, X, y, off)
    theta = spec(oracle, d).get_hyperparameters()
    _, g0 = oracle.regression.bcm_objective(experts, theta)
    fd = np.zeros_like(theta)
    for i in range(len(theta)):
        h = 1e-5 * max(abs(theta[i]), 1e-2)
        tp, tm = theta.copy(), theta.copy()
        tp[i] += h
        tm[i] -= h
        fd[i] = (oracle.regression.bcm_objective(experts, tp)[0] - oracle.regression.bcm_objective(experts, tm)[0]) / (2 * h)
    err = np.abs(fd - g0) / np.maximum(np.abs(g0), 1e-3 * np.abs(g0).max())
    print("oracle vs finite differences: max rel %.2e" % err.max())
    assert err.max() < 1e-6
