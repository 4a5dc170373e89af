"""GPU parity tests (run on a B200: `pytest -m gpu`).  Everything goes through the C-ABI (ctypes) and is
compared with the fp64 oracle on identical seeded inputs, or with the committed golden fixtures.

Arithmetic modes (include/sgp.h): AUTO (default) = the tcgen05 int8 exact-accumulation Gram on accumulate calls of
>= 32768 points whose scaled squared norms are inside the magnitude budget (tensor-core distances for one non-Eye term and
d <= 32, direct fp32 distances for sums of up to 4 terms / d <= 72), else the fp64 DMMA kernel (F64); I8 / I8_DIRECT force
the two int8 modes; F64_STRICT = all-fp64 verification mode.

Tolerances (written here once):
  TOL_STRICT = 1e-11  G, b in SGP_PREC_F64_STRICT (all-fp64) mode, relative to max|G| / max|b|
  TOL_STATS  = 1e-6   G, b in SGP_PREC_F64 (fp32-accurate elements, fp64 accumulation); SURVEY 8(d) gate
  TOL_I8     = 3e-6   G, b in SGP_PREC_I8 on SMALL shards: the kernel elements carry the fp32 rounding of the
                      tensor-core distance contraction (|dT| <= 1.7e-6 measured => 1.2e-6 relative per element);
                      the Gram accumulation itself is exact.  Element errors are independent, so on real shard
                      sizes they average out: the 1M-point test below holds TOL_STATS (measured 1.5e-7).
  TOL_PRED   = 1e-5   posterior mean / variance (BASELINE.json north_star tolerance), every mode; magicVector /
                      magicMatrix to 1e-5 in strict mode
  TOL_MAGIC  = 1e-3   magicVector / magicMatrix in the default mode: they are cond(A)-amplified images of the
                      1e-7 element rounding and are not themselves part of the parity contract (the mean and
                      variance they produce are, and those hold TOL_PRED)
"""
import os

import numpy as np
import pytest

import oracle
import spark_gp_b200 as sg
from spark_gp_b200 import _native as N

pytestmark = pytest.mark.gpu

TOL_STRICT, TOL_STATS, TOL_PRED, TOL_MAGIC, TOL_I8 = 1e-11, 1e-6, 1e-5, 1e-3, 3e-6
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def eng():
    e = sg.ProjectedProcessEngine(0)
    yield e
    e.close()


def rel(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max() / max(np.abs(np.asarray(b)).max(), 1e-300))


def oracle_stats(okernel_factory, X, y, Z, n_e=100):
    experts = oracle.get_expert_labels_and_kernels(X, y, okernel_factory, n_e)
    theta = okernel_factory().get_hyperparameters()
    return oracle.projected_process(experts, Z, okernel_factory, theta)


MODES = {"strict": (N.SGP_PREC_F64_STRICT, TOL_STRICT), "f64": (N.SGP_PREC_F64, TOL_STATS), "i8": (N.SGP_PREC_I8, TOL_I8),
         "i8d": (N.SGP_PREC_I8_DIRECT, TOL_STATS)}


def run_stats(eng, kernel, X, y, Z, precision=N.SGP_PREC_AUTO, splits=None):
    eng.set_precision(precision)
    eng.begin(kernel, Z)
    if splits is None:
        eng.accumulate(X, y)
    else:
        lo = 0
        for hi in list(splits) + [len(X)]:
            eng.accumulate(X[lo:hi], y[lo:hi])
            lo = hi
    return eng.finish()


# ---------------- the reference's own golden vectors, through the CUDA path ---------------------------
DATASET = np.array([[1.0, 2.0], [2.0, 3.0], [5.0, 7.0]])


def test_rbf_cross_kernel_golden(eng):                      # RBFKernelTest.scala:62-76
    eng.begin(sg.RBFKernel(np.sqrt(0.2)), DATASET[1:])      # "training vectors" = dataset.drop(1)
    ck = eng.cross_kernel(DATASET[:1])
    assert ck.shape == (1, 2)                               # test.length x train.length
    correct = np.array([[6.737947e-03, 3.053624e-45]])
    assert np.all(np.abs(ck - correct) < 1e-4)
    assert np.allclose(ck, correct, rtol=1e-6, atol=0)


def test_rbf_training_kernel_golden(eng):                   # RBFKernelTest.scala:29-39 (cross(X,X) == training kernel)
    eng.begin(sg.RBFKernel(np.sqrt(0.2)), DATASET)
    K = eng.cross_kernel(DATASET)
    correct = np.array([[1.000000e+00, 6.737947e-03, 3.053624e-45],
                        [6.737947e-03, 1.000000e+00, 7.187782e-28],
                        [3.053624e-45, 7.187782e-28, 1.000000e+00]])
    assert np.allclose(K, correct, rtol=1e-6, atol=0)


def test_survey_smoke_values(eng):                          # SURVEY.md 8(c) derived values
    k = 1 * sg.ARDRBFKernel(np.array([0.2, 0.3])) + sg.const(1) * sg.EyeKernel() + sg.const(1e-4) * sg.EyeKernel()
    y = np.array([0.5, -1.0, 2.0])
    Z = DATASET[[0, 2]]
    for prec, tol in ((N.SGP_PREC_F64_STRICT, 1e-11), (N.SGP_PREC_F64, 1e-6), (N.SGP_PREC_I8, 3e-6)):
        G, b = run_stats(eng, k, DATASET, y, Z, prec)
        assert np.allclose(G, [[1.774140301212, 0.256300623707], [0.256300623707, 1.030412437856]], rtol=tol)
        assert np.allclose(b, [-0.266943005698, 1.862489218084], rtol=tol)
        mv, mm = eng.magic()
        assert np.allclose(mv, [-0.122545269186, 0.627149214156], rtol=max(tol, 1e-10) * 10)
        assert np.allclose(mm, [[-0.233122498440, -0.013597424403], [-0.013597424403, -0.167542879982]],
                           rtol=max(tol, 1e-10) * 10)
        mean, var = eng.predict(np.array([[3.0, 4.0]]))
        assert np.isclose(mean[0], 0.164885948858, rtol=max(tol, 1e-10) * 10)
        assert np.isclose(var[0], 1.887496212554, rtol=max(tol, 1e-10) * 10)


# ---------------- committed golden fixtures ------------------------------------------------------------
def _small_case(name):
    z = np.load(os.path.join(GOLD, "small_cases.npz"))
    return {k.split("/", 1)[1]: z[k] for k in z.files if k.startswith(name + "/")}


SMALL_KERNELS = {
    "ard_ragged": lambda d: 2.5 * sg.ARDRBFKernel(np.linspace(0.5, 1.5, d)) + sg.const(0.3) * sg.EyeKernel(),
    "rbf_wide": lambda d: sg.RBFKernel(3.0),
    "sum_two": lambda d: 1.5 * sg.ARDRBFKernel(np.full(d, 0.7)) + 0.5 * sg.RBFKernel(2.0) + sg.const(1) * sg.EyeKernel(),
}


@pytest.mark.parametrize("name", list(SMALL_KERNELS))
@pytest.mark.parametrize("mode", ["strict", "f64", "auto"])
def test_small_golden_cases(eng, name, mode):
    c = _small_case(name)
    d = c["X"].shape[1]
    kernel = SMALL_KERNELS[name](d) + sg.const(1e-3) * sg.EyeKernel()       # GPC:18 sigma2 term
    strict = mode == "strict"
    prec = {"strict": N.SGP_PREC_F64_STRICT, "f64": N.SGP_PREC_F64, "auto": N.SGP_PREC_AUTO}[mode]
    G, b = run_stats(eng, kernel, c["X"], c["y"], c["Z"], prec)
    tol = TOL_STRICT if strict else TOL_STATS          # AUTO keeps calls of < 32768 points on the fp64 kernel
    assert rel(G, c["G"]) < tol and rel(b, c["b"]) < tol
    assert np.array_equal(G, G.T)
    mv, mm = eng.magic()
    assert rel(mv, c["magic_vector"]) < (TOL_PRED if strict else TOL_MAGIC)
    assert rel(mm, c["magic_matrix"]) < (TOL_PRED if strict else TOL_MAGIC)
    mean, var = eng.predict(c["Xtest"])
    assert rel(mean, c["mean"]) < TOL_PRED
    assert np.abs(var / c["var"] - 1).max() < TOL_PRED


@pytest.mark.parametrize("mode", ["strict", "f64", "i8", "i8d"])
def test_airfoil_golden(eng, mode):
    """BASELINE config 1 (airfoil, expert=100, active=1000, ARD(5)); fixture made by tests/golden/make_golden.py.
    "i8" / "i8d" = the int8 Gram FORCED on this shard (tensor-core / direct fp32 distances): the statistics are fine (direct:
    1e-6), the posterior mean is not -- the kernel values of this data are tiny (scaled squared norms up to ~40) and the
    fixed-point elements carry an absolute error of 2^-24, which cond(A) = 6e7 amplifies to 1.5e-4.  AUTO never runs the
    int8 Gram on such data (magnitude budget, test_auto_magnitude_gate)."""
    c = np.load(os.path.join(GOLD, "airfoil_case.npz"))
    kernel = (1 * sg.ARDRBFKernel(5) + sg.const(1) * sg.EyeKernel() + sg.const(float(c["sigma2"])) * sg.EyeKernel())
    kernel.setHyperparameters(c["theta"])
    strict = mode == "strict"
    G, b = run_stats(eng, kernel, c["X"], c["y"], c["Z"], MODES[mode][0])
    tol = MODES[mode][1]
    if mode == "i8":
        # explicit SGP_PREC_I8 on this 1353-point shard (AUTO would pick the fp64 kernel): standardised features with
        # beta up to 1.4 give scaled squared norms up to ~30, so the fp32 accumulator of the tensor-core distance
        # contraction rounds at ~2e-6 and the statistics are only good to ~1e-5 -- documented, not parity-grade
        tol = 2e-5
    gmax = np.abs(c["G_diag"]).max()
    assert np.abs(np.diag(G) - c["G_diag"]).max() / gmax < tol
    assert np.abs(G[0] - c["G_row0"]).max() / gmax < tol
    assert abs(G.sum() - c["G_sum"]) / abs(c["G_sum"]) < tol
    assert rel(b, c["b"]) < tol
    mv, mm = eng.magic()
    mean, var = eng.predict(c["Xtest"])
    print("airfoil[%s]: dmean=%.2e dvar=%.2e" % (mode, rel(mean, c["mean"]), np.abs(var / c["var"] - 1).max()))
    if mode not in ("i8", "i8d"):   # forced int8 on this shard is NOT parity-grade (measured 1.5e-4 on the mean); AUTO never picks it
        assert rel(mv, c["magic_vector"]) < (TOL_PRED if strict else TOL_MAGIC)
        assert rel(np.diag(mm), c["magic_matrix_diag"]) < (TOL_PRED if strict else TOL_MAGIC)
        assert rel(mean, c["mean"]) < TOL_PRED
        assert np.abs(var / c["var"] - 1).max() < TOL_PRED


def test_auto_magnitude_gate(eng):
    """AUTO runs the int8 Gram only on shards whose scaled squared norms are small: large norms mean tiny kernel values,
    where the 2^-24 ABSOLUTE error of the fixed-point elements -- with either distance form -- loses the posterior mean on
    ill-conditioned systems (profiles/r02o_i8_conditioning.txt: airfoil-like data 1.5e-4 .. 1.5e-2 against 7e-7 .. 7e-6 of
    the fp64 kernel).  Airfoil (mean scaled squared norm ~6 for points and active set, maxima ~40) stays on the fp64
    kernel even when the shard is large -- and keeps the posterior mean / variance inside 1e-5 of the all-fp64 mode; the
    benchmark's unit cube (mean ~2.2) runs the int8 kernel; small shards stay on the fp64 kernel."""
    c = np.load(os.path.join(GOLD, "airfoil_case.npz"))
    kernel = (1 * sg.ARDRBFKernel(5) + sg.const(1) * sg.EyeKernel() + sg.const(float(c["sigma2"])) * sg.EyeKernel())
    kernel.setHyperparameters(c["theta"])
    reps = 200                                              # 270k points
    X, y = np.tile(c["X"], (reps, 1)), np.tile(c["y"], reps)
    rng0 = np.random.default_rng(8)
    X = X + 0.05 * rng0.standard_normal(X.shape); y = y + 0.05 * rng0.standard_normal(len(y))    # distinct points
    G, b = run_stats(eng, kernel, X, y, c["Z"], N.SGP_PREC_AUTO)
    assert eng.last_path() == N.SGP_PREC_F64
    eng.magic(); mean, var = eng.predict(c["Xtest"])
    Gs, bs = run_stats(eng, kernel, X, y, c["Z"], N.SGP_PREC_F64_STRICT)
    eng.magic(); mean0, var0 = eng.predict(c["Xtest"])
    print("airfoil x200 (jittered), AUTO -> fp64 kernel: dG=%.2e db=%.2e dmean=%.2e dvar=%.2e" % (
        rel(G, Gs), rel(b, bs), rel(mean, mean0), np.abs(var / var0 - 1).max()))
    assert rel(G, Gs) < TOL_STATS and rel(b, bs) < TOL_STATS
    assert rel(mean, mean0) < TOL_PRED and np.abs(var / var0 - 1).max() < TOL_PRED
    rng = np.random.default_rng(2)
    Xu = rng.random((300000, 16), dtype=np.float32)
    ku = 1 * sg.ARDRBFKernel(np.full(16, np.sqrt(18.0 / 16))) + sg.const(1) * sg.EyeKernel()
    run_stats(eng, ku, Xu, rng.random(300000), Xu[:256].astype(np.float64), N.SGP_PREC_AUTO)
    assert eng.last_path() == N.SGP_PREC_I8
    run_stats(eng, ku, Xu[:5000], rng.random(5000), Xu[:256].astype(np.float64), N.SGP_PREC_AUTO)
    assert eng.last_path() == N.SGP_PREC_F64                # small shard


# ---------------- seeded inputs vs the oracle, edge cases ---------------------------------------------
@pytest.mark.parametrize("n,d,m", [(1, 1, 1), (15, 2, 3), (16, 4, 128), (17, 5, 129), (257, 7, 256), (1000, 33, 200),
                                   (2048, 16, 384), (333, 70, 50), (200, 80, 40)])
def test_ragged_shapes_vs_oracle(eng, n, d, m):
    rng = np.random.default_rng(n * 1000 + d * 10 + m)
    X = rng.standard_normal((n, d))
    y = rng.standard_normal(n)
    Z = rng.standard_normal((m, d))
    beta = rng.uniform(0.2, 0.9, d) / np.sqrt(d)
    k = 1.7 * sg.ARDRBFKernel(beta) + sg.const(1e-2) * sg.EyeKernel()
    ok = lambda: 1.7 * oracle.ARDRBFKernel(beta) + oracle.const(1e-2) * oracle.EyeKernel()
    _, G0, b0 = oracle_stats(ok, X, y, Z, n_e=max(2, min(100, n)))
    G, b = run_stats(eng, k, X, y, Z, N.SGP_PREC_F64_STRICT)
    assert rel(G, G0) < TOL_STRICT and rel(b, b0) < TOL_STRICT
    G, b = run_stats(eng, k, X, y, Z, N.SGP_PREC_F64)
    assert rel(G, G0) < TOL_STATS and rel(b, b0) < TOL_STATS
    if d <= 72:                              # int8 Gram: tensor-core distances for d <= 32, direct fp32 distances up to 72
        G, b = run_stats(eng, k, X, y, Z, N.SGP_PREC_I8)
        assert eng.last_path() == (N.SGP_PREC_I8 if d <= 32 else N.SGP_PREC_I8_DIRECT)
        assert rel(G, G0) < TOL_I8 and rel(b, b0) < TOL_I8
        assert np.array_equal(G, G.T)
        G, b = run_stats(eng, k, X, y, Z, N.SGP_PREC_I8_DIRECT)
        assert eng.last_path() == N.SGP_PREC_I8_DIRECT
        assert rel(G, G0) < TOL_I8 and rel(b, b0) < TOL_I8
    else:
        with pytest.raises(ValueError):                     # explicit I8 request on a non-qualifying shape
            run_stats(eng, k, X, y, Z, N.SGP_PREC_I8)
    G, b = run_stats(eng, k, X, y, Z, N.SGP_PREC_AUTO)      # AUTO always works (small shard -> fp64 kernel)
    assert rel(G, G0) < TOL_STATS and rel(b, b0) < TOL_STATS


def test_i8_operand_range_falls_back(eng):
    """Coordinates far outside the fp16 operand range: SGP_PREC_I8 reports SGP_E_RANGE at finish (no silent garbage);
    the Estimator mirror then reruns on the fp64 DMMA kernel -- still on the GPU."""
    rng = np.random.default_rng(5)
    X = rng.standard_normal((500, 4)) * 1e4
    y = rng.standard_normal(500)
    Z = X[:64].copy()
    k = 1 * sg.ARDRBFKernel(np.full(4, 1.0)) + sg.const(1e-2) * sg.EyeKernel()
    eng.set_precision(N.SGP_PREC_I8)
    eng.begin(k, Z)
    eng.accumulate(X, y)
    with pytest.raises(sg.OperandRangeError):
        eng.finish()
    G, b = run_stats(eng, k, X, y, Z, N.SGP_PREC_F64_STRICT)
    ok = lambda: 1 * oracle.ARDRBFKernel(np.full(4, 1.0)) + oracle.const(1e-2) * oracle.EyeKernel()
    _, G0, b0 = oracle_stats(ok, X, y, Z)
    assert rel(G, G0) < TOL_STRICT
    from spark_gp_b200.regression import ExplicitActiveSetProvider
    gp = (sg.GaussianProcessRegression().setKernel(lambda: 1 * sg.ARDRBFKernel(4)).setSigma2(1e-2)
          .setActiveSetProvider(ExplicitActiveSetProvider(Z)).setMaxIter(0))
    Xbig, ybig = np.tile(X, (600, 1)), np.tile(y, 600)     # 300k points: AUTO considers the int8 kernel, falls back
    gp.fit(Xbig, ybig)
    assert rel(gp.last_stats[0], 600.0 * G0) < TOL_STATS


def test_empty_shard_and_only_eye_kernel(eng):
    rng = np.random.default_rng(3)
    X, y, Z = rng.standard_normal((40, 3)), rng.standard_normal(40), rng.standard_normal((5, 3))
    k = 1 * sg.ARDRBFKernel(3) + sg.const(0.1) * sg.EyeKernel()
    eng.set_precision(N.SGP_PREC_AUTO)                      # (the engine fixture is shared: pin the mode)
    eng.begin(k, Z)
    eng.accumulate(X[:0], y[:0])                            # empty shard is a no-op
    eng.accumulate(X, y)
    G1, b1 = eng.finish()
    G2, b2 = run_stats(eng, k, X, y, Z)
    assert np.array_equal(G1, G2) and np.array_equal(b1, b2)
    G, b = run_stats(eng, sg.const(2.0) * sg.EyeKernel(), X, y, Z)    # Eye only: crossKernel == 0 (Kernel.scala:157)
    assert not G.any() and not b.any()


def test_shard_linearity_and_fp32_inputs(eng):
    """G, b are sums over points: any split of the shard gives the same statistics (to fp64 rounding);
    fp32 inputs are consumed exactly (identical to their fp64 up-cast)."""
    rng = np.random.default_rng(11)
    X = rng.random((5000, 8), dtype=np.float32)
    y = np.sin(X.astype(np.float64).sum(1))
    Z = X[:300].astype(np.float64)
    k = 1 * sg.ARDRBFKernel(np.full(8, 1.5)) + sg.const(1) * sg.EyeKernel()
    G1, b1 = run_stats(eng, k, X, y, Z)
    G2, b2 = run_stats(eng, k, X, y, Z, splits=[17, 1000, 1001, 4096])
    assert rel(G2, G1) < 1e-13 and rel(b2, b1) < 1e-13
    G3, b3 = run_stats(eng, k, X.astype(np.float64), y, Z)
    assert rel(G3, G1) < 1e-13 and rel(b3, b1) < 1e-13
    G4, b4 = run_stats(eng, k, X, 2.0 * y, Z)               # b is linear in y, G independent of y
    assert np.array_equal(G4, G1) and rel(b4, 2.0 * b1) < 1e-15
    assert np.array_equal(G1, G1.T)


def test_determinism(eng):
    rng = np.random.default_rng(12)
    X, y, Z = rng.random((3000, 6)), rng.random(3000), rng.random((260, 6))
    k = 1 * sg.ARDRBFKernel(6)+ sg.const(1) * sg.EyeKernel()
    G1, b1 = run_stats(eng, k, X, y, Z)
    G2, b2 = run_stats(eng, k, X, y, Z)
    assert np.array_equal(G1, G2) and np.array_equal(b1, b2)   # no atomics: bit-reproducible


# ---------------- error behaviour ------------------------------------------------------------------------
def test_not_positive_definite(eng):
    k = 1 * sg.ARDRBFKernel(2) + sg.const(1e-12) * sg.EyeKernel()
    eng.begin(k, DATASET)
    with pytest.raises(sg.NotPositiveDefiniteException):
        eng.magic(G=-10.0 * np.eye(3), b=np.ones(3))


def test_call_order_errors():
    e = sg.ProjectedProcessEngine(0)
    with pytest.raises(sg.TrainingVectorsNotInitializedException):
        e._check(e._lib.sgp_stats_accumulate(e._h, None, 0, None, 0))
    with pytest.raises(sg.TrainingVectorsNotInitializedException):
        e._check(e._lib.sgp_predict(e._h, None, 0, None, None))
    with pytest.raises(ValueError):
        e.begin(sg.Scalar(1.0) * sg.ARDRBFKernel(3), np.zeros((4, 2)))     # beta length != d
    e.close()


# ---------------- Estimator surface ------------------------------------------------------------------------
def test_estimator_fit_predict_matches_oracle():
    from spark_gp_b200.regression import ExplicitActiveSetProvider
    rng = np.random.default_rng(21)
    X = rng.random((3000, 4))
    y = np.sin(3 * X.sum(1)) + 0.05 * rng.standard_normal(3000)
    Z = X[rng.permutation(3000)[:200]]
    theta = np.array([1.3, 1.1, 0.9, 1.2, 0.8])
    gp = (sg.GaussianProcessRegression().setKernel(lambda: 1 * sg.ARDRBFKernel(4) + sg.const(1) * sg.EyeKernel())
          .setSigma2(1e-4).setActiveSetSize(200).setDatasetSizeForExpert(100)
          .setActiveSetProvider(ExplicitActiveSetProvider(Z)))
    model = gp.fit(X, y, hyperparameters=theta)
    ofac = oracle.get_kernel(lambda: 1 * oracle.ARDRBFKernel(4) + oracle.const(1) * oracle.EyeKernel(), 1e-4)
    experts = oracle.get_expert_labels_and_kernels(X, y, ofac, 100)
    pred, G0, b0 = oracle.projected_process(experts, Z, ofac, theta)
    Xt = rng.random((500, 4))
    m0, v0 = pred.predict_many(Xt)
    assert rel(model.predict(Xt), m0) < TOL_PRED
    mean, var = model.rawPredictor.predict(Xt)
    assert rel(mean, m0) < TOL_PRED and np.abs(var / v0 - 1).max() < TOL_PRED
    m1, v1 = model.rawPredictor.predict(Xt[0])
    o1 = pred.predict(Xt[0])
    assert abs(m1 - o1[0]) < TOL_PRED * abs(m0).max() and abs(v1 / o1[1] - 1) < TOL_PRED


# ---------------- BASELINE-size run: size-independent properties -----------------------------------------------
def test_full_size_config2_properties(eng):
    """synthetic 1M x 16 fp32, active=1000 (BASELINE configs[1]): the oracle cannot finish this in seconds, so
    check (a) a 20k-point sub-shard against the oracle, (b) shard-additivity of the full run, (c) symmetry,
    (d) trace(G) = sum_n |k_n|^2 >= 0 and G_jj <= N * C^2."""
    rng = np.random.default_rng(13)
    N_, d, m = 1_000_000, 16, 1000
    X = rng.random((N_, d), dtype=np.float32)
    y = np.sin(X.astype(np.float64).sum(1)) + 0.1 * rng.standard_normal(N_)
    Z = X[rng.permutation(N_)[:m]].astype(np.float64)
    beta = np.full(d, np.sqrt(18.0 / d))
    k = 1 * sg.ARDRBFKernel(beta) + sg.const(1) * sg.EyeKernel() + sg.const(1e-4) * sg.EyeKernel()
    ok = lambda: 1 * oracle.ARDRBFKernel(beta) + oracle.const(1) * oracle.EyeKernel() + oracle.const(1e-4) * oracle.EyeKernel()
    Gs, bs = run_stats(eng, k, X[:20000], y[:20000], Z)
    _, G0, b0 = oracle_stats(ok, X[:20000].astype(np.float64), y[:20000], Z, n_e=100)
    assert rel(Gs, G0) < TOL_STATS and rel(bs, b0) < TOL_STATS
    G, b = run_stats(eng, k, X, y, Z)
    Gh, bh = run_stats(eng, k, X[:400_000], y[:400_000], Z)
    Gt, bt = run_stats(eng, k, X[400_000:], y[400_000:], Z)
    assert rel(Gh + Gt, G) < 1e-12 and rel(bh + bt, b) < 1e-12
    assert np.array_equal(G, G.T)
    assert np.all(np.diag(G) > 0) and np.all(np.diag(G) <= N_ * 1.0 + 1e-6)
    assert np.all(np.abs(G) <= np.sqrt(np.outer(np.diag(G), np.diag(G))) * (1 + 1e-12))   # Cauchy-Schwarz
    mv, _ = eng.magic(G, b, copy_out=True)
    assert np.all(np.isfinite(mv))
    # (e) full-size prediction parity of the default (tcgen05 int8) path against the all-fp64 kernel, which the small
    # cases above pin on the oracle:  posterior mean and variance at 1000 held-out points within TOL_PRED
    Xt = rng.random((1000, d))
    mean8, var8 = eng.predict(Xt)
    Gs64, bs64 = run_stats(eng, k, X, y, Z, N.SGP_PREC_F64_STRICT)
    assert rel(G, Gs64) < TOL_STATS and rel(b, bs64) < TOL_STATS
    eng.magic()
    mean64, var64 = eng.predict(Xt)
    print("1M x 16, m=1000: int8 vs all-fp64: dG=%.2e db=%.2e dmean=%.2e dvar=%.2e" % (
        rel(G, Gs64), rel(b, bs64), rel(mean8, mean64), np.abs(var8 / var64 - 1).max()))
    assert rel(mean8, mean64) < TOL_PRED
    assert np.abs(var8 / var64 - 1).max() < TOL_PRED
    # regression guard for the int8 digit layout (8-bit unsigned top digit): measured 2.1e-6 / 4.9e-9 here; the first,
    # byte-aligned layout gave 7.9e-6 / 1.2e-8 -- still inside TOL_PRED but with a 1.3x margin only
    assert rel(mean8, mean64) < 0.5 * TOL_PRED


# ---------------- the hyper-parameter objective (BCM NLL + gradient, SURVEY 8 f1) ------------------------------------
TOL_NLL = 1e-9     # fp64 Cholesky on the GPU vs the oracle's LU (GPR:59): far inside the north star's 1e-5 on the LML


def _bcm_case(kernel_pair, n=1237, d=4, n_e=100, seed=4):
    from spark_gp_b200.hyperopt import pack_experts
    rng = np.random.default_rng(seed)
    X = rng.random((n, d))
    y = np.sin(3 * X.sum(1)) + 0.1 * rng.standard_normal(n)
    mk, mo = kernel_pair
    k = mk()
    ofac = mo
    experts = oracle.get_expert_labels_and_kernels(X, y, ofac, n_e)
    nll0, g0 = oracle.regression.bcm_objective(experts, k.getHyperparameters())
    return X, y, k, nll0, g0, pack_experts(X, y, n_e)


@pytest.mark.parametrize("which", ["ard", "rbf_noise", "sum"])
def test_bcm_nll_and_gradient_vs_oracle(eng, which):
    pairs = {
        "ard": (lambda: 1.3 * sg.ARDRBFKernel(np.array([1.1, 0.7, 1.9, 0.4])) + sg.const(1) * sg.EyeKernel() + sg.const(1e-2) * sg.EyeKernel(),
                lambda: 1.3 * oracle.ARDRBFKernel(np.array([1.1, 0.7, 1.9, 0.4])) + oracle.const(1) * oracle.EyeKernel() + oracle.const(1e-2) * oracle.EyeKernel()),
        "rbf_noise": (lambda: sg.Scalar(2.0).between(0).and_(30) * sg.RBFKernel(0.6, 1e-6, 10) + sg.WhiteNoiseKernel(0.5, 0, 1) + sg.const(1e-3) * sg.EyeKernel(),
                      lambda: oracle.Scalar(2.0).between(0).and_(30) * oracle.RBFKernel(0.6, 1e-6, 10) + oracle.WhiteNoiseKernel(0.5, 0, 1) + oracle.const(1e-3) * oracle.EyeKernel()),
        "sum": (lambda: 0.7 * (1.5 * sg.ARDRBFKernel(np.full(4, 0.9)) + 0.5 * sg.RBFKernel(2.0)) + sg.const(0.2) * sg.EyeKernel(),
                lambda: 0.7 * (1.5 * oracle.ARDRBFKernel(np.full(4, 0.9)) + 0.5 * oracle.RBFKernel(2.0)) + oracle.const(0.2) * oracle.EyeKernel()),
    }
    X, y, k, nll0, g0, (Xp, yp, off) = _bcm_case(pairs[which])
    eng.experts_upload(Xp, yp, off)
    nll, g = eng.bcm_nll(k)
    assert abs(nll - nll0) / abs(nll0) < TOL_NLL
    assert np.abs(g - g0).max() / np.abs(g0).max() < 1e-8
    assert len(g) == k.numberOfHyperparameters()


def test_airfoil_bcm_nll_golden(eng):
    """BCM objective on the airfoil fixture (15 experts of ~90 points): log-marginal-likelihood parity, 1e-5 gate."""
    from spark_gp_b200.hyperopt import pack_experts
    c = np.load(os.path.join(GOLD, "airfoil_case.npz"))
    kernel = (1 * sg.ARDRBFKernel(5) + sg.const(1) * sg.EyeKernel() + sg.const(float(c["sigma2"])) * sg.EyeKernel())
    kernel.setHyperparameters(c["theta"])
    eng.experts_upload(*pack_experts(c["X"], c["y"], 100))
    nll, g = eng.bcm_nll(kernel)
    assert abs(nll - float(c["bcm_nll"])) / abs(float(c["bcm_nll"])) < 1e-9
    assert np.abs(g - c["bcm_grad"]).max() / np.abs(c["bcm_grad"]).max() < 1e-8


def test_fit_with_hyperparameter_optimisation():
    """GaussianProcessRegression.fit end to end (optimizeHypers -> produceModel), Synthetics.scala-style data: the
    reference asserts 10-fold CV RMSE < 0.11 on noisy sin(x) (regression/examples/Synthetics.scala:25-33); here a
    hold-out RMSE under the same threshold, and the objective must not increase."""
    rng = np.random.default_rng(13)
    X = np.linspace(0, 1, 2000)[:, None]
    y = np.sin(X[:, 0]) + np.sqrt(0.01) * rng.standard_normal(2000)
    idx = rng.permutation(2000)
    tr, te = idx[:1800], idx[1800:]
    gp = (sg.GaussianProcessRegression()
          .setKernel(lambda: 1 * sg.RBFKernel(0.1, 1e-6, 10) + sg.WhiteNoiseKernel(0.5, 0, 1))
          .setDatasetSizeForExpert(100).setActiveSetSize(100).setSeed(13).setSigma2(1e-3).setMaxIter(30))
    model = gp.fit(X[tr], y[tr])
    rmse = float(np.sqrt(np.mean((model.predict(X[te]) - y[te]) ** 2)))
    assert rmse < 0.11
    assert gp.last_objective["evaluations"] >= 2
    from spark_gp_b200.hyperopt import BcmObjective
    eng = sg.ProjectedProcessEngine(0)
    obj = BcmObjective(eng, gp.getKernel, X[tr], y[tr], 100)
    f0, _ = obj(gp.getKernel().getHyperparameters())
    f1, _ = obj(model.hyperparameters)
    eng.close()
    assert f1 <= f0


# ---------------- BASELINE config 3: mnist68 binary classification path (d = 784, RBFKernel(10), y := Laplace mode f) ----
def test_mnist68_classification_path_golden(eng):
    """classification/GaussianProcessClassifier.scala:62-65: produceModel runs the SAME projected-process statistics
    with the per-expert latent mode f in place of the labels.  f comes from the oracle's Laplace loop (fixture); the
    statistics (d = 784 > 32 -> fp64 DMMA kernel with a chunked feature loop), the tail and the raw prediction f* run
    on the GPU.  predictRaw = (-f*, f*), probability = sigmoid(f*) (GPCls:141-156)."""
    c = np.load(os.path.join(GOLD, "mnist68_case.npz"))
    n = int(c["n_rows"])
    X = (c["pixels"].astype(np.float64) - c["mean"]) / c["std"]
    Xtr, Xte = X[:n], X[n:n + 100]
    Z = Xtr[c["active_idx"]]
    kernel = sg.RBFKernel(float(c["sigma"])) + sg.const(float(c["sigma2"])) * sg.EyeKernel()
    G, b = run_stats(eng, kernel, Xtr, c["f"], Z)
    assert eng.last_path() == N.SGP_PREC_F64
    gmax = np.abs(c["G_diag"]).max()
    assert np.abs(np.diag(G) - c["G_diag"]).max() / gmax < TOL_STATS
    assert np.abs(G[0] - c["G_row0"]).max() / gmax < TOL_STATS
    assert rel(b, c["b"]) < TOL_STATS
    eng.magic()
    fstar, var = eng.predict(Xte)
    assert rel(fstar, c["fstar"]) < TOL_PRED
    assert np.abs(var / c["var"] - 1).max() < TOL_PRED
    prob0 = 1.0 / (1.0 + np.exp(-fstar))                   # raw2probabilityInPlace: values(0) = sigmoid(f)  (GPCls:143-144)
    assert np.all((prob0 > 0.5) == (c["fstar"] > 0))


# ---------------- classification: batched Laplace objective (GPCls:74-129) -------------------------------------------
def test_laplace_nll_gradient_and_modes_vs_oracle(eng):
    """Two consecutive objective evaluations at different theta (the second warm-starts from the first's modes, as the
    reference's cached experts do): -log Z, its gradient and every expert's latent mode f vs the oracle."""
    from oracle.classification import classification_likelihood_and_gradient
    from spark_gp_b200.hyperopt import pack_experts, group_for_experts
    rng = np.random.default_rng(31)
    n, d, n_e, tol = 730, 3, 100, 1e-6
    X = rng.standard_normal((n, d))
    y = (np.sin(2 * X[:, 0]) + X[:, 1] * X[:, 2] + 0.3 * rng.standard_normal(n) > 0).astype(np.float64)
    mk = lambda: 1.2 * sg.ARDRBFKernel(np.array([0.8, 0.5, 1.1])) + sg.const(1e-2) * sg.EyeKernel()
    mo = lambda: 1.2 * oracle.ARDRBFKernel(np.array([0.8, 0.5, 1.1])) + oracle.const(1e-2) * oracle.EyeKernel()
    groups = group_for_experts(n, n_e)
    experts = oracle.get_expert_labels_and_kernels(X, y, mo, n_e)
    fs = [np.zeros(len(g)) for g in groups]
    eng.experts_upload(*pack_experts(X, y, n_e))
    theta0 = mk().getHyperparameters()
    for theta in (theta0, theta0 * np.array([1.4, 0.7, 1.3, 0.9])):
        v0, g0 = 0.0, 0.0
        for (ye, ke), f in zip(experts, fs):
            v, g = classification_likelihood_and_gradient(ye, f, ke, theta, tol)
            v0 += v; g0 = g0 + g
        v, g = eng.laplace_nll(mk().setHyperparameters(theta), tol)
        assert abs(v - v0) / abs(v0) < 1e-9
        assert np.abs(g - g0).max() / np.abs(g0).max() < 1e-7
        f_gpu = eng.experts_f(n)
        assert np.abs(f_gpu - np.concatenate(fs)).max() < 1e-9 * max(1.0, np.abs(np.concatenate(fs)).max())


def test_classifier_fit_mnist68_fixture():
    """GaussianProcessClassifier.fit at fixed theta (MNIST.scala:28-32: RBFKernel(10), tol = 1e-3) on the mnist68
    fixture: the GPU Laplace modes equal the oracle's (fixture `f`), the model's raw predictions equal the oracle's f*."""
    from spark_gp_b200.regression import ExplicitActiveSetProvider
    c = np.load(os.path.join(GOLD, "mnist68_case.npz"))
    n = int(c["n_rows"])
    X = (c["pixels"].astype(np.float64) - c["mean"]) / c["std"]
    Xtr, Xte, ytr = X[:n], X[n:n + 100], c["y01"][:n]
    gp = (sg.GaussianProcessClassifier().setDatasetSizeForExpert(100).setActiveSetSize(500)
          .setKernel(lambda: sg.RBFKernel(float(c["sigma"]))).setTol(1e-3)
          .setActiveSetProvider(ExplicitActiveSetProvider(Xtr[c["active_idx"]])))
    model = gp.fit(Xtr, ytr, hyperparameters=np.array([float(c["sigma"])]))
    assert np.abs(gp.last_latent - c["f"]).max() < 1e-8
    raw = model.predictRaw(Xte)
    assert rel(raw[:, 1], c["fstar"]) < TOL_PRED and np.allclose(raw[:, 0], -raw[:, 1])
    # prediction = argmax of the RAW vector (Spark's raw2prediction without thresholds): class 1 iff f > 0; only the
    # probability column carries the reference's quirk (sigmoid(f) on class 0)
    acc = np.mean(model.predict(Xte) == c["y01"][n:n + 100])
    assert acc > 0.95
    prob = model.predictProbability(Xte)
    assert np.allclose(prob[:, 0], 1.0 / (1.0 + np.exp(-raw[:, 1]))) and np.allclose(prob.sum(1), 1.0)
    with pytest.raises(RuntimeError):
        gp.fit(Xtr, ytr + 1.0)


@pytest.mark.gpu
def test_greedy_active_set_provider_matches_oracle():
    """SURVEY 8(f4): GreedilyOptimizingActiveSetProvider (ActiveSetProvider.scala:58-139).  Statistics and the per-point
    quadratic forms come from the GPU (sgp_stats_*, sgp_set_magic + sgp_predict); the selected points must be the ones
    the CPU restatement selects, round by round (first point given explicitly: Spark's takeSample stream is unpinned)."""
    from oracle.active_set import greedy_active_set
    rng = np.random.default_rng(21)
    n, d, m, n_e = 600, 3, 8, 50
    X = rng.random((n, d)); y = np.sin(3 * X.sum(1)) + 0.05 * rng.standard_normal(n)
    beta = np.full(d, 1.7)
    ofac = oracle.get_kernel(lambda: 1.3 * oracle.ARDRBFKernel(beta) + oracle.const(1) * oracle.EyeKernel(), 1e-2)
    theta = ofac().get_hyperparameters()
    experts = oracle.get_expert_labels_and_kernels(X, y, ofac, n_e)
    for _, k in experts:
        k.set_hyperparameters(theta)
    want = greedy_active_set(m, experts, ofac, theta, X[5])
    gp = (sg.GaussianProcessRegression().setKernel(lambda: 1.3 * sg.ARDRBFKernel(beta) + sg.const(1) * sg.EyeKernel())
          .setSigma2(1e-2).setDatasetSizeForExpert(n_e).setActiveSetSize(m).setMaxIter(0)
          .setActiveSetProvider(sg.GreedilyOptimizingActiveSetProvider(first_index=5, precision=N.SGP_PREC_F64_STRICT)))
    got = gp._activeSetProvider(m, X, y, gp.getKernel, theta, 13, gp=gp)          # rank-1 updates on the device (default)
    assert got.shape == want.shape
    assert np.array_equal(got, want), "greedy selection (rank-1 updates) differs from the restatement"
    slow = sg.GreedilyOptimizingActiveSetProvider(first_index=5, precision=N.SGP_PREC_F64_STRICT, incremental=False)
    got2 = slow(m, X, y, gp.getKernel, theta, 13, gp=gp)                          # a statistics pass per round
    assert np.array_equal(got2, want), "greedy selection (round-by-round form) differs from the restatement"
    # and through fit(): the model is the projected process on that active set
    model = gp.fit(X, y, hyperparameters=theta)
    k0 = ofac().set_hyperparameters(theta)
    pred, _, _ = oracle.projected_process(experts, want, ofac, theta)
    m0, _ = pred.predict_many(X[:50])
    assert np.abs(model.predict(X[:50]) - m0).max() / np.abs(m0).max() <= TOL_PRED


# ---------------- round 2: the headline int8 path pinned DIRECTLY on the oracle ----------------------------------------
def _bench_workload(n, d, m, seed=13):
    """bench.py's synthetic workload (SURVEY 8(d)): X ~ U[0,1)^d in fp32, y = sin(sum x) + 0.1 eps, active set = m rows
    of a seeded permutation, kernel 1*ARD(beta = sqrt(18/d)) + 1.const*Eye + sigma2.const*Eye."""
    rng = np.random.default_rng(seed)
    X = rng.random((n, d), dtype=np.float32)
    y = np.sin(X.astype(np.float64).sum(1)) + 0.1 * rng.standard_normal(n)
    Z = X[rng.permutation(n)[:m]].astype(np.float64)
    beta = np.full(d, np.sqrt(18.0 / d))
    k = 1 * sg.ARDRBFKernel(beta) + sg.const(1) * sg.EyeKernel() + sg.const(1e-4) * sg.EyeKernel()
    ok = lambda: 1 * oracle.ARDRBFKernel(beta) + oracle.const(1) * oracle.EyeKernel() + oracle.const(1e-4) * oracle.EyeKernel()
    return X, y, Z, k, ok


def _oracle_stats_chunked(ok, X, y, Z, chunk=2048):
    """PGPH:20-36 with contiguous 'experts' of `chunk` points: G and b are plain sums over points, so the partition into
    experts is immaterial (test_shard_linearity pins that on the GPU side); big chunks keep the CPU dgemms efficient."""
    theta = ok().get_hyperparameters()
    X = np.asarray(X, dtype=np.float64)
    experts = [(y[i:i + chunk], ok().set_training_vectors(X[i:i + chunk]).set_hyperparameters(theta))
               for i in range(0, len(X), chunk)]
    return oracle.get_matrix_kmn_knm_and_vector_kmny(experts, Z)


def test_i8_headline_path_vs_oracle(eng):
    """BASELINE configs[1] shape on a shard AUTO routes to the tcgen05 int8 kernel (>= 32768 points): G, b <= 1e-6
    (SURVEY 8(d) gate) and posterior mean / variance at 1000 held-out points <= 1e-5 against the ORACLE itself (all
    worker cores, ~3 s) -- not against another kernel of this library."""
    from oracle.cpu_baseline import stats_parallel
    n, d, m = 300_000, 16, 1000
    X, y, Z, k, ok = _bench_workload(n, d, m)
    G, b = run_stats(eng, k, X, y, Z, N.SGP_PREC_AUTO)
    assert eng.last_path() == N.SGP_PREC_I8
    mv, mm = eng.magic()
    assert eng.last_tail_path() == 1                                   # Cholesky PD check + solves
    Xt = np.random.default_rng(99).random((1000, d))
    mean, var = eng.predict(Xt)
    G0, b0, _ = stats_parallel(X.astype(np.float64), y, Z, ok, ok().get_hyperparameters(), 100)
    kernel0 = ok().set_hyperparameters(ok().get_hyperparameters()).set_training_vectors(Z)
    mv0, mm0 = oracle.get_magic_vector(kernel0, G0, b0)                # eigvalsh check + LU, as the reference
    m0, v0 = oracle.GaussianProjectedProcessRawPredictor(mv0, mm0, kernel0).predict_many(Xt)
    eg, eb, em, ev = rel(G, G0), rel(b, b0), rel(mean, m0), float(np.abs(var / v0 - 1).max())
    print("int8 path vs ORACLE, 300k x 16, m=1000: dG=%.2e db=%.2e dmean=%.2e dvar=%.2e" % (eg, eb, em, ev))
    assert eg < TOL_STATS and eb < TOL_STATS
    assert em < TOL_PRED and ev < TOL_PRED
    assert np.array_equal(G, G.T)


@pytest.mark.parametrize("n,d,m", [(20480, 32, 2000), (8192, 8, 4000), (16384, 17, 300), (16384, 31, 300),
                                   (16384, 1, 130), (12345, 16, 1000)])
def test_i8_config_shapes_vs_oracle(eng, n, d, m):
    """Sub-shards of BASELINE configs[3] (d=32, m=2000: two 64-column K chunks of the distance contraction, 136 G tiles)
    and configs[4] (d=8, m=4000: 528 G tiles = more CTAs than SMs), plus d = 17 / 31 / 1 and a ragged point count, on
    the forced int8 kernel against the oracle, at the SURVEY 8(d) gate of 1e-6 (measured 1.3e-7 .. 7.7e-7,
    profiles/r02a_gpu_tests_r1kernel.log)."""
    X, y, Z, k, ok = _bench_workload(n, d, m, seed=100 + d)
    G0, b0 = _oracle_stats_chunked(ok, X, y, Z)
    G, b = run_stats(eng, k, X, y, Z, N.SGP_PREC_I8)
    assert eng.last_path() == N.SGP_PREC_I8
    eg, eb = rel(G, G0), rel(b, b0)
    print("int8 vs oracle n=%d d=%d m=%d: dG=%.2e db=%.2e" % (n, d, m, eg, eb))
    assert eg < TOL_STATS and eb < TOL_STATS
    assert np.array_equal(G, G.T)
    Gs, bs = run_stats(eng, k, X, y, Z, N.SGP_PREC_F64)               # the fp64 DMMA kernel on the same shapes
    assert rel(Gs, G0) < TOL_STATS and rel(bs, b0) < TOL_STATS


def test_tail_paths(eng):
    """sgp_magic: Cholesky fast path on a well-posed model; the reference's literal dsyevd + LU sequence when the
    factorization breaks down -- indefinite A raises NotPositiveDefiniteException like PGPH:62-65; a kernel WITHOUT any Eye
    term on duplicated active points has a singular K_mm: Cholesky of K_mm breaks down and the LU path reports the
    singular matrix like Breeze's MatrixSingularException (or returns LU's answer if rounding keeps the pivots non-zero)."""
    rng = np.random.default_rng(8)
    X, y, Z = rng.random((500, 3)), rng.random(500), rng.random((40, 3))
    k = 1 * sg.ARDRBFKernel(3) + sg.const(0.1) * sg.EyeKernel()
    run_stats(eng, k, X, y, Z, N.SGP_PREC_F64)
    eng.magic()
    assert eng.last_tail_path() == 1
    with pytest.raises(sg.NotPositiveDefiniteException):
        eng.magic(G=-10.0 * np.eye(40), b=np.ones(40))
    assert eng.last_tail_path() == 1 or eng.last_tail_path() == 0
    # slow path that SUCCEEDS: A positive definite but K_mm's Cholesky breaks down is impossible (A = wn K + G with wn>0)
    # -> exercise the eigenvalue branch with a semi-definite A: G = -wn*K_mm + v v' makes A = v v' (rank one, PSD)
    ok = lambda: 1 * oracle.ARDRBFKernel(3) + oracle.const(0.1) * oracle.EyeKernel()
    kmm = ok().set_training_vectors(Z).training_kernel()
    v = rng.random(40)
    try:
        eng.magic(G=-0.1 * kmm + np.outer(v, v), b=np.ones(40))
    except (sg.NotPositiveDefiniteException, sg.MatrixSingularException):
        pass                                                            # either outcome is the reference's (rounding decides)
    assert eng.last_tail_path() == 0


def test_two_contexts_two_devices_two_threads():
    """One process (one JVM in INTEGRATION.md's `create(pid % nGPUs)`), contexts on two different GPUs driven from two
    threads through the C-ABI: both must produce the single-context result.  Needs >= 2 visible GPUs."""
    import threading
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    X, y, Z, k, ok = _bench_workload(300_000, 16, 256, seed=5)
    out = {}

    def work(dev):
        e = sg.ProjectedProcessEngine(dev)
        try:
            for prec in (N.SGP_PREC_AUTO, N.SGP_PREC_F64):
                out[(dev, prec)] = run_stats(e, k, X, y, Z, prec)
                out[(dev, prec, "path")] = e.last_path()
        except Exception as ex:                                        # surfaced in the main thread
            out[(dev, "err")] = ex
        finally:
            e.close()

    ts = [threading.Thread(target=work, args=(dev,)) for dev in (0, 1)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    for dev in (0, 1):
        assert (dev, "err") not in out, out.get((dev, "err"))
    assert out[(0, N.SGP_PREC_AUTO, "path")] == N.SGP_PREC_I8 and out[(1, N.SGP_PREC_AUTO, "path")] == N.SGP_PREC_I8
    for prec in (N.SGP_PREC_AUTO, N.SGP_PREC_F64):
        assert np.array_equal(out[(0, prec)][0], out[(1, prec)][0]) and np.array_equal(out[(0, prec)][1], out[(1, prec)][1])


def test_auto_budget_checked_over_whole_window(eng):
    """AUTO chooses the kernel on the first chunk of a call; the scaled squared norms of EVERY chunk are summed on the
    device and checked at finish, so an unrepresentative first chunk cannot silently degrade the statistics: here the first
    600k points are benign and the rest have large norms -> SGP_E_RANGE at finish, and the Estimator's helper reruns on
    the fp64 kernel."""
    rng = np.random.default_rng(17)
    d, m = 8, 128
    Xa = rng.random((600_000, d), dtype=np.float32)
    Xb = (rng.random((1_000_000, d), dtype=np.float32) * 12.0)
    X = np.vstack([Xa, Xb]); y = rng.random(len(X))
    Z = Xa[:m].astype(np.float64)
    k = 1 * sg.ARDRBFKernel(np.full(d, 1.0)) + sg.const(1) * sg.EyeKernel()
    eng.set_precision(N.SGP_PREC_AUTO)
    eng.begin(k, Z)
    eng.accumulate(X, y)
    assert eng.last_path() == N.SGP_PREC_I8
    with pytest.raises(sg.OperandRangeError):
        eng.finish()
    G, b = eng.statistics(k, Z, X, y)
    assert eng.last_path() == N.SGP_PREC_F64
    eng.set_precision(N.SGP_PREC_AUTO)
    assert np.all(np.isfinite(G))


def test_bcm_large_experts_general_path(eng):
    """datasetSizeForExpert has no upper bound in the reference (GaussianProcessParams.scala:36).  Experts of 400 points
    exceed the on-chip objective kernel: the evaluation takes the global-memory LU path (the reference's own arithmetic,
    logDetAndInv.scala:36-63) and must match the oracle like the fast path does."""
    from spark_gp_b200.hyperopt import pack_experts
    rng = np.random.default_rng(44)
    n, d, n_e = 2030, 5, 400
    X = rng.random((n, d)); y = np.sin(3 * X.sum(1)) + 0.1 * rng.standard_normal(n)
    mk = lambda: 1.3 * sg.ARDRBFKernel(np.linspace(0.6, 1.8, d)) + 0.4 * sg.RBFKernel(1.5) + sg.const(1e-2) * sg.EyeKernel()
    mo = lambda: 1.3 * oracle.ARDRBFKernel(np.linspace(0.6, 1.8, d)) + 0.4 * oracle.RBFKernel(1.5) + oracle.const(1e-2) * oracle.EyeKernel()
    k = mk()
    experts = oracle.get_expert_labels_and_kernels(X, y, mo, n_e)
    nll0, g0 = oracle.regression.bcm_objective(experts, k.getHyperparameters())
    eng.experts_upload(*pack_experts(X, y, n_e))
    nll, g = eng.bcm_nll(k)
    assert eng.last_bcm_path() == 1
    assert abs(nll - nll0) / abs(nll0) < TOL_NLL
    assert np.abs(g - g0).max() / np.abs(g0).max() < 1e-8
    # the same path on small experts (forced by a matrix Cholesky cannot factor: duplicated points, no Eye term):
    # no NotPositiveDefinite error -- the reference's LU carries on; only an exactly singular matrix may fail
    Xd = np.vstack([X[:60], X[:60]]); yd = np.concatenate([y[:60], y[:60]])
    eng.experts_upload(*pack_experts(Xd, yd, 120))
    try:
        v, gg = eng.bcm_nll(1.0 * sg.ARDRBFKernel(np.full(d, 0.7)))
        assert np.isfinite(v) and np.all(np.isfinite(gg))
    except sg.MatrixSingularException:
        pass
    assert eng.last_bcm_path() == 1
    # and the fast path is still the one taken for the default expert size
    eng.experts_upload(*pack_experts(X, y, 100))
    nll1, g1 = eng.bcm_nll(k)
    assert eng.last_bcm_path() == 0
    ex100 = oracle.get_expert_labels_and_kernels(X, y, mo, 100)
    nll2, g2 = oracle.regression.bcm_objective(ex100, k.getHyperparameters())
    assert abs(nll1 - nll2) / abs(nll2) < TOL_NLL


def test_device_side_expert_grouping_matches_host_packing(eng):
    """sgp_experts_upload_grouped (GPC:26-31 as a strided gather on the device) must reproduce the host-side expert-major
    packing exactly: the BCM objective is bit-identical, for fp64 and fp32 inputs, with and without a remainder (N % E)."""
    from spark_gp_b200.hyperopt import pack_experts
    rng = np.random.default_rng(77)
    k = 1.3 * sg.ARDRBFKernel(np.array([1.1, 0.7, 1.9])) + sg.const(1e-2) * sg.EyeKernel()
    for n in (1200, 1237):
        X = rng.random((n, 3)); y = rng.standard_normal(n)
        eng.experts_upload(*pack_experts(X, y, 100))
        v0, g0 = eng.bcm_nll(k)
        E = eng.experts_upload_grouped(X, y, 100)
        assert E == int(np.floor(n / 100 + 0.5))
        v1, g1 = eng.bcm_nll(k)
        assert v0 == v1 and np.array_equal(g0, g1)
        X32 = X.astype(np.float32)
        eng.experts_upload(*pack_experts(X32.astype(np.float64), y, 100))
        v2, g2 = eng.bcm_nll(k)
        eng.experts_upload_grouped(X32, y, 100)
        v3, g3 = eng.bcm_nll(k)
        assert v2 == v3 and np.array_equal(g2, g3)


@pytest.mark.parametrize("n,d,m", [(5000, 8, 4000), (70001, 16, 1000), (3000, 32, 200), (130, 3, 129)])
def test_kmn_sweep_vs_fp64_cross_kernel(eng, n, d, m):
    """K_nm sweep (fp32, tensor-core distances) against the fp64 cross kernel of the same context, which the reference's
    RBF goldens pin (test_rbf_*): element-wise <= 1e-5 relative to the kernel scale (north-star tolerance), measured ~3e-7."""
    rng = np.random.default_rng(n + d)
    X = rng.random((n, d), dtype=np.float32)
    Z = X[rng.permutation(n)[:min(m, n)]].astype(np.float64)
    if len(Z) < m:
        Z = np.vstack([Z, rng.random((m - len(Z), d))])
    k = 2.5 * sg.ARDRBFKernel(np.full(d, np.sqrt(18.0 / d))) + sg.const(1) * sg.EyeKernel()
    eng.set_precision(N.SGP_PREC_AUTO)
    eng.begin(k, Z)
    K32 = eng.kmn_sweep(X)
    K64 = eng.cross_kernel(X.astype(np.float64))
    err = float(np.abs(K32 - K64).max() / 2.5)
    print("sweep n=%d d=%d m=%d: max |dK| / C = %.2e" % (n, d, m, err))
    assert K32.shape == (n, m) and err < 1e-5


# ---------------- int8 Gram with direct fp32 distances (SGP_PREC_I8_DIRECT) -------------------------------------------
def test_i8_direct_headline_shape_vs_oracle(eng):
    """The headline shape on the direct-distance mode against the ORACLE: same 1e-6 / 1e-5 gates as the tensor-distance
    mode."""
    from oracle.cpu_baseline import stats_parallel
    n, d, m = 300_000, 16, 1000
    X, y, Z, k, ok = _bench_workload(n, d, m)
    G, b = run_stats(eng, k, X, y, Z, N.SGP_PREC_I8_DIRECT)
    assert eng.last_path() == N.SGP_PREC_I8_DIRECT
    eng.magic()
    Xt = np.random.default_rng(99).random((1000, d))
    mean, var = eng.predict(Xt)
    G0, b0, _ = stats_parallel(X.astype(np.float64), y, Z, ok, ok().get_hyperparameters(), 100)
    kernel0 = ok().set_hyperparameters(ok().get_hyperparameters()).set_training_vectors(Z)
    mv0, mm0 = oracle.get_magic_vector(kernel0, G0, b0)
    m0, v0 = oracle.GaussianProjectedProcessRawPredictor(mv0, mm0, kernel0).predict_many(Xt)
    eg, eb, em, ev = rel(G, G0), rel(b, b0), rel(mean, m0), float(np.abs(var / v0 - 1).max())
    print("int8 direct vs ORACLE, 300k x 16, m=1000: dG=%.2e db=%.2e dmean=%.2e dvar=%.2e" % (eg, eb, em, ev))
    assert eg < TOL_STATS and eb < TOL_STATS
    assert em < TOL_PRED and ev < TOL_PRED
    assert np.array_equal(G, G.T)


@pytest.mark.parametrize("case", ["two_terms", "d40", "d64", "three_terms_d12", "offset_1e3", "rbf_plus_ard"])
def test_i8_direct_widened_shapes_vs_oracle(eng, case):
    """What the tensor-distance mode cannot take: sums of several non-Eye terms, 32 < d <= 64, data far from the origin
    (the active-set mean is subtracted in fp64 before the fp32 rounding).  Oracle in fp64, gate 1e-6."""
    rng = np.random.default_rng(sum(map(ord, case)))
    n, m = 16384 + 77, 300
    d = {"two_terms": 8, "d40": 40, "d64": 64, "three_terms_d12": 12, "offset_1e3": 6, "rbf_plus_ard": 5}[case]
    X = rng.random((n, d))
    if case == "offset_1e3":
        X += 1000.0
    y = np.sin(X.sum(1)) + 0.1 * rng.standard_normal(n)
    Z = X[rng.permutation(n)[:m]].copy()
    b1 = rng.uniform(0.5, 1.5, d) * np.sqrt(6.0 / d)
    b2 = rng.uniform(0.5, 1.5, d) * np.sqrt(20.0 / d)
    b3 = rng.uniform(0.5, 1.5, d) * np.sqrt(2.0 / d)
    if case in ("two_terms",):
        mk = lambda S: 0.7 * S.ARDRBFKernel(b1) + 1.9 * S.ARDRBFKernel(b2) + S.const(1e-3) * S.EyeKernel()
    elif case == "three_terms_d12":
        mk = lambda S: 0.7 * S.ARDRBFKernel(b1) + 1.9 * S.ARDRBFKernel(b2) + 0.2 * S.ARDRBFKernel(b3) + S.const(1e-3) * S.EyeKernel()
    elif case == "rbf_plus_ard":
        mk = lambda S: 1.1 * S.RBFKernel(0.6) + 0.4 * S.ARDRBFKernel(b2) + S.const(1e-3) * S.EyeKernel()
    else:
        mk = lambda S: 1.3 * S.ARDRBFKernel(b1) + S.const(1e-3) * S.EyeKernel()
    k, ok = mk(sg), (lambda: mk(oracle))
    G0, b0 = _oracle_stats_chunked(ok, X, y, Z)
    G, b = run_stats(eng, k, X, y, Z, N.SGP_PREC_I8_DIRECT)
    assert eng.last_path() == N.SGP_PREC_I8_DIRECT
    eg, eb = rel(G, G0), rel(b, b0)
    print("int8 direct vs oracle [%s] n=%d d=%d m=%d: dG=%.2e db=%.2e" % (case, n, d, m, eg, eb))
    assert eg < TOL_STATS and eb < TOL_STATS
    assert np.array_equal(G, G.T)


def test_auto_routes_multi_term_kernels_to_direct_mode(eng):
    """AUTO on a large shard with a SUM of two ARD terms and d = 40 (tensor-core distances take neither): the int8 Gram with
    direct distances, inside the same magnitude budget -- statistics 1e-6, posterior mean / variance 1e-5 against the
    all-fp64 mode; the same kernels on data with large scaled norms go to the fp64 kernel."""
    rng = np.random.default_rng(41)
    n, m = 120_000, 500
    for d, mk in ((8, lambda b1, b2: 0.7 * sg.ARDRBFKernel(b1) + 0.6 * sg.ARDRBFKernel(b2) + sg.const(1e-2) * sg.EyeKernel()),
                  (40, lambda b1, b2: 1.2 * sg.ARDRBFKernel(b1) + sg.const(1e-2) * sg.EyeKernel())):
        X = rng.random((n, d), dtype=np.float32)
        y = np.sin(X.astype(np.float64).sum(1)) + 0.1 * rng.standard_normal(n)
        Z = X[rng.permutation(n)[:m]].astype(np.float64)
        b1, b2 = np.full(d, np.sqrt(12.0 / d)), np.full(d, np.sqrt(30.0 / d))
        k = mk(b1, b2)
        Xt = rng.random((500, d))
        G, b = run_stats(eng, k, X, y, Z, N.SGP_PREC_AUTO)
        assert eng.last_path() == N.SGP_PREC_I8_DIRECT
        eng.magic(); mean, var = eng.predict(Xt)
        Gs, bs = run_stats(eng, k, X, y, Z, N.SGP_PREC_F64_STRICT)
        eng.magic(); mean0, var0 = eng.predict(Xt)
        print("AUTO -> direct, d=%d: dG=%.2e db=%.2e dmean=%.2e dvar=%.2e" % (
            d, rel(G, Gs), rel(b, bs), rel(mean, mean0), np.abs(var / var0 - 1).max()))
        assert rel(G, Gs) < TOL_STATS and rel(b, bs) < TOL_STATS
        assert rel(mean, mean0) < TOL_PRED and np.abs(var / var0 - 1).max() < TOL_PRED
        run_stats(eng, k, 6.0 * X, y, 6.0 * Z, N.SGP_PREC_AUTO)          # scaled squared norms x 36: above the budget
        assert eng.last_path() == N.SGP_PREC_F64
    eng.set_precision(N.SGP_PREC_AUTO)


def test_i8_direct_norm_limit_and_error_growth(eng):
    """The direct mode rounds centred, scaled coordinates to fp32: the exponent error grows like 2^-24 sqrt(q) (|x|+|z|),
    and the rounding of an active point is common to all its kernel values (it does not average out over the shard).
    Adversarial layout: clusters far apart, unit-scale structure inside each.  Measured dG 1.2e-7 / 6.6e-7 / 2.7e-6 at
    scaled squared norms ~10 / ~1300 / ~7700: norms above 2048 are refused (SGP_E_RANGE at finish), below the limit the
    statistics stay inside 1e-6."""
    rng = np.random.default_rng(23)
    n, d, m = 65536, 8, 256
    base = rng.random((n, d))
    errs = []
    for spread in (1.0, 10.0, 25.0, 400.0):
        # clusters `spread` apart, unit-scale structure inside each: norms grow, neighbour distances do not
        X = base + spread * rng.integers(0, 3, (n, 1)) * np.ones((1, d))
        y = np.sin(base.sum(1))
        Z = X[rng.permutation(n)[:m]].copy()
        beta = np.full(d, 1.0)
        k = 1 * sg.ARDRBFKernel(beta) + sg.const(1e-3) * sg.EyeKernel()
        ok = lambda: 1 * oracle.ARDRBFKernel(beta) + oracle.const(1e-3) * oracle.EyeKernel()
        eng.set_precision(N.SGP_PREC_I8_DIRECT)
        eng.begin(k, Z)
        eng.accumulate(X, y)
        if spread >= 25.0:                   # scaled squared norm ~ 8 * (25 * 1.2)^2 = 7200 > 2048
            with pytest.raises(sg.OperandRangeError):
                eng.finish()
            continue
        G, b = eng.finish()
        G0, b0 = _oracle_stats_chunked(ok, X, y, Z)
        errs.append((spread, rel(G, G0), rel(b, b0)))
    print("int8 direct, error vs cluster spread:", ", ".join("%g: dG=%.1e db=%.1e" % e for e in errs))
    assert all(e[1] < TOL_STATS and e[2] < TOL_STATS for e in errs)


def test_greedy_rank1_larger_cases():
    """The rank-1 form (sgp_greedy_active_set) on a case with 64 rounds and all-distinct selections against the CPU
    restatement AND the round-by-round GPU form; a sum of two ARD terms with repeated selections (the reference does not
    exclude selected points: nearly singular bordered steps -> the Cholesky refresh path) against the round-by-round form;
    and the time per round at 200k points (the reference's form costs a statistics pass + two predictions per round)."""
    import time
    from oracle.active_set import greedy_active_set
    rng = np.random.default_rng(77)
    n, d, m, n_e = 3000, 4, 64, 100
    X = rng.random((n, d)); y = np.sin(4 * X.sum(1)) + 0.1 * rng.standard_normal(n)
    beta = np.full(d, 3.0)
    ofac = oracle.get_kernel(lambda: 1.0 * oracle.ARDRBFKernel(beta) + oracle.const(1) * oracle.EyeKernel(), 1e-1)
    theta = ofac().get_hyperparameters()
    experts = oracle.get_expert_labels_and_kernels(X, y, ofac, n_e)
    for _, k in experts:
        k.set_hyperparameters(theta)
    want = greedy_active_set(m, experts, ofac, theta, X[5])
    gp = (sg.GaussianProcessRegression().setKernel(lambda: 1.0 * sg.ARDRBFKernel(beta) + sg.const(1) * sg.EyeKernel())
          .setSigma2(1e-1).setDatasetSizeForExpert(n_e).setActiveSetSize(m).setMaxIter(0))
    fast = sg.GreedilyOptimizingActiveSetProvider(first_index=5)
    slow = sg.GreedilyOptimizingActiveSetProvider(first_index=5, precision=N.SGP_PREC_F64_STRICT, incremental=False)
    a = fast(m, X, y, gp.getKernel, theta, 1, gp=gp)
    b = slow(m, X, y, gp.getKernel, theta, 1, gp=gp)
    print("greedy 3000 x 4 -> 64 points: %d distinct (oracle %d)" % (len(np.unique(a, axis=0)), len(np.unique(want, axis=0))))
    assert np.array_equal(a, want), "rank-1 selection differs from the restatement"
    assert np.array_equal(b, want), "round-by-round selection differs from the restatement"
    # repeated selections, two terms, ragged last expert
    n, d, m = 20011, 5, 48
    X = rng.random((n, d)); y = np.sin(2 * X.sum(1)) + 0.1 * rng.standard_normal(n)
    b1, b2 = rng.uniform(0.8, 2.5, d), rng.uniform(2.0, 5.0, d)
    gp = (sg.GaussianProcessRegression().setKernel(lambda: 0.8 * sg.ARDRBFKernel(b1) + 0.5 * sg.ARDRBFKernel(b2))
          .setSigma2(1e-2).setDatasetSizeForExpert(n_e).setActiveSetSize(m).setMaxIter(0))
    theta = gp.getKernel().getHyperparameters()
    fast = sg.GreedilyOptimizingActiveSetProvider(first_index=123)
    slow = sg.GreedilyOptimizingActiveSetProvider(first_index=123, precision=N.SGP_PREC_F64_STRICT, incremental=False)
    t0 = time.perf_counter(); a = fast(m, X, y, gp.getKernel, theta, 1, gp=gp); t1 = time.perf_counter()
    b = slow(m, X, y, gp.getKernel, theta, 1, gp=gp); t2 = time.perf_counter()
    print("greedy 20011 x 5 -> 48 points (%d distinct): rank-1 %.3f s, round-by-round %.3f s" % (
        len(np.unique(a, axis=0)), t1 - t0, t2 - t1))
    assert np.array_equal(a, b)
    # scale: 200k points, 256 selected -- O(N m) per round
    n2, d2, m2 = 200_000, 8, 256
    X2 = rng.random((n2, d2)); y2 = np.sin(2 * X2.sum(1)) + 0.1 * rng.standard_normal(n2)
    bb = np.full(d2, 3.0)
    gp2 = (sg.GaussianProcessRegression().setKernel(lambda: 1 * sg.ARDRBFKernel(bb) + sg.const(1) * sg.EyeKernel())
           .setSigma2(1e-1).setActiveSetSize(m2).setMaxIter(0))
    fast = sg.GreedilyOptimizingActiveSetProvider(first_index=7)
    t0 = time.perf_counter()
    a2 = fast(m2, X2, y2, gp2.getKernel, gp2.getKernel().getHyperparameters(), 1, gp=gp2)
    t1 = time.perf_counter()
    print("greedy 200000 x 8 -> 256 points (%d distinct): rank-1 %.3f s = %.2f ms per round" % (
        len(np.unique(a2, axis=0)), t1 - t0, 1e3 * (t1 - t0) / m2))
    assert a2.shape == (m2, d2) and np.all(np.isfinite(a2))
