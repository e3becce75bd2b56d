"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through
the C ABI, against the CPU oracle on the same seeded inputs.

Tolerances (BASELINE.json north_star): 1e-4 relative on responsibilities (with an
absolute floor of 1e-6), means and covariances; integer-exact final cluster count;
log-likelihood 1e-5 relative (FP32 in the reference; the engine reduces it in
double, SURVEY.md H6)."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, random_spd_params, fitted_params, assert_params_close, gpu_count, RUN_RTOL_N, RUN_MEMB

pytestmark = pytest.mark.gpu

PATHS = ["simt", "auto"]


def path_id(pkg, name):
    return {"simt": pkg.PATH_SIMT, "auto": pkg.PATH_AUTO, "tensor": pkg.PATH_TENSOR}[name]


def assert_memb_close(got, ref, rtol=1e-4, atol=1e-6):
    np.testing.assert_allclose(got, ref, rtol=rtol, atol=atol)


def run_level_check(got, ref, K, path, memb=None, rtol=1e-4):
    """Parity after many EM iterations: the calibrated run-level bar of conftest.py (1e-3 relative / 1e-5 absolute on
    responsibilities, 5e-4 on N_k, 1e-4 scaled on means / covariances) for BOTH paths.  Measured deviations from the exact
    oracle (scripts/exp_acc.py, round 2): config 1 x 100 iterations 4.2e-5 on responsibilities for the tensor path (SIMT
    5.8e-6, the reference's own FP32 arithmetic 6.5e-6); config-2 slice x 10: 2.3e-4 (SIMT 2.2e-5, reference FP32 6.5e-5)."""
    assert_params_close(got, ref, K, rtol=rtol, rtol_N=RUN_RTOL_N)
    assert_memb_close(got.memberships, ref.memberships, **(memb or RUN_MEMB))


@pytest.fixture(scope="module")
def loaded(pkg):
    pkg.load_library()
    return pkg


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("N,D,K", [(10_000, 4, 8), (5_003, 16, 32), (4_097, 24, 64), (1_000, 1, 3),
                                   (777, 32, 5), (3_000, 7, 130), (33, 3, 2), (20_000, 24, 16)])
def test_estep_parity(loaded, oracle64, path, N, D, K):
    pkg = loaded
    ev = pkg.synth.make_blobs(N, D, min(K, 8), seed=100 + D)
    ref = fitted_params(pkg, oracle64, ev, K)
    with pkg.Engine(ev, K) as eng:
        eng.set_option("path", path_id(pkg, path))
        eng.set_clusters(K, ref)
        ll = eng.estep(K)
        got = eng.get_clusters(K, with_memberships=True)
    ll_ref = oracle64.estep(oracle64.transpose(ev), ref, K)
    assert_memb_close(got.memberships, ref.memberships)
    np.testing.assert_allclose(got.memberships.sum(0), 1.0, atol=1e-5)
    assert abs(ll - ll_ref) <= 1e-5 * abs(ll_ref)


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("N,D,K", [(5_003, 16, 32), (4_097, 24, 64)])
def test_estep_random_params_stress(loaded, oracle64, path, N, D, K):
    """Unfitted random parameters: Mahalanobis distances of several hundred for every
    cluster of an event; FP32 evaluation noise of the quadratic form is then ~1e-4
    relative (the reference's own FP32 kernels are no better), hence the looser bar."""
    pkg = loaded
    ev = pkg.synth.make_blobs(N, D, 8, seed=100 + D)
    ref = random_spd_params(pkg, K, D, np.random.default_rng(D * 7 + K), spread=6.0)
    ref.memberships = np.zeros((K, N), np.float32)
    oracle64.constants(ref, K)
    with pkg.Engine(ev, K) as eng:
        eng.set_option("path", path_id(pkg, path))
        eng.set_clusters(K, ref)
        ll = eng.estep(K)
        got = eng.get_clusters(K, with_memberships=True)
    ll_ref = oracle64.estep(oracle64.transpose(ev), ref, K)
    assert_memb_close(got.memberships, ref.memberships, rtol=1e-3, atol=1e-5)
    assert abs(ll - ll_ref) <= 1e-5 * abs(ll_ref)


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("N,D,K", [(10_000, 4, 8), (5_003, 16, 32), (4_097, 24, 64), (1_000, 1, 3),
                                   (777, 32, 5), (3_000, 7, 130), (33, 3, 2), (20_000, 24, 16)])
def test_mstep_constants_parity(loaded, oracle64, path, N, D, K):
    """gmm_mstep (N, means, R) then gmm_constants (Rinv, constant, pi) from the
    SAME responsibilities as the oracle."""
    pkg = loaded
    ev = pkg.synth.make_blobs(N, D, min(K, 8), seed=200 + D)
    ref = fitted_params(pkg, oracle64, ev, K)
    soa = oracle64.transpose(ev)
    with pkg.Engine(ev, K) as eng:
        eng.set_option("path", path_id(pkg, path))
        eng.seed(K)                       # establishes the global-mean shift
        eng.set_clusters(K, ref)
        eng.estep(K)
        eng.mstep(K)
        eng.constants(K)
        got = eng.get_clusters(K)
    oracle64.estep(soa, ref, K)
    oracle64.mstep(soa, ref, K)
    oracle64.constants(ref, K)
    assert_params_close(got, ref, K)


@pytest.mark.parametrize("N,D,K", [(300_000, 24, 64), (150_001, 16, 32), (100_003, 24, 17), (65_000, 8, 64), (257, 16, 5),
                                   (60_001, 24, 128), (30_001, 16, 100), (20_000, 8, 200)])
def test_estep_tensor_path_large(loaded, oracle64, N, D, K):
    """The tcgen05 E-step (resident whitening factors) over many tiles per CTA, odd event counts
    (partial last tile), cluster counts that do not fill an MMA group, and more than 64 clusters
    (one pass per 64 clusters + the combine kernel)."""
    pkg = loaded
    ev = pkg.synth.make_blobs(N, D, min(K, 16), seed=400 + D)
    ref = fitted_params(pkg, oracle64, ev, K, iters=1)
    with pkg.Engine(ev, K) as eng:
        eng.set_option("path", pkg.PATH_TENSOR)
        eng.seed(K)
        eng.set_clusters(K, ref)
        ll = eng.estep(K)
        got = eng.get_clusters(K, with_memberships=True)
    ll_ref = oracle64.estep(oracle64.transpose(ev), ref, K)
    assert_memb_close(got.memberships, ref.memberships)
    np.testing.assert_allclose(got.memberships.sum(0), 1.0, atol=1e-5)
    assert abs(ll - ll_ref) <= 1e-5 * abs(ll_ref)


@pytest.mark.parametrize("sigma", [1e-3, 1e-4, 1e-5])
@pytest.mark.parametrize("N,D,K", [(20_000, 24, 64), (9_001, 16, 9), (8_000, 8, 70)])
def test_estep_tensor_tight_and_wide_clusters(loaded, oracle64, N, D, K, sigma):
    """Clusters far narrower than the data (whitening factors 1e3 .. 1e6 in the kernel's standardised coordinates,
    beyond the FP16 range without the per-cluster power-of-two operand scale) next to ordinary and very wide ones:
    GMM_PATH_TENSOR must evaluate them itself (no SIMT fallback) at the per-operator bar."""
    pkg = loaded
    ev = pkg.synth.make_blobs(N, D, min(K, 8), seed=500 + D)
    ref = fitted_params(pkg, oracle64, ev, K)
    rng = np.random.default_rng(K)
    for k, idx in ((0, 123), (K - 1, 4567)):                 # two needle clusters sitting on events
        ref.means[k] = ev[idx] + rng.normal(0, sigma, D).astype(np.float32)
        ref.R[k] = np.eye(D, dtype=np.float32) * np.float32(sigma * sigma)
        ref.N[k] = 3.0
    ref.R[1] = np.eye(D, dtype=np.float32) * np.float32(400.0)   # and one far wider than the data
    oracle64.constants(ref, K)
    with pkg.Engine(ev, K) as eng:
        eng.set_option("path", pkg.PATH_TENSOR)
        eng.set_clusters(K, ref)
        ll = eng.estep(K)
        got = eng.get_clusters(K, with_memberships=True)
    ll_ref = oracle64.estep(oracle64.transpose(ev), ref, K)
    assert_memb_close(got.memberships, ref.memberships)
    assert ref.memberships[0, 123] > 0.5 and ref.memberships[K - 1, 4567] > 0.5      # the needles do capture their events
    assert abs(ll - ll_ref) <= 1e-5 * abs(ll_ref)


@pytest.mark.parametrize("N,D,K", [(200_000, 24, 64), (150_001, 16, 32), (100_000, 4, 8), (70_000, 24, 100)])
def test_mstep_tensor_path_large(loaded, oracle64, N, D, K):
    """The tcgen05 M-step (GMM_PATH_TENSOR) on enough events to exercise several TMEM
    flush chunks per CTA, against the oracle M-step on the same responsibilities."""
    pkg = loaded
    ev = pkg.synth.make_blobs(N, D, min(K, 16), seed=300 + D)
    ref = fitted_params(pkg, oracle64, ev, K, iters=1)
    soa = oracle64.transpose(ev)
    with pkg.Engine(ev, K) as eng:
        eng.set_option("path", pkg.PATH_TENSOR)
        eng.seed(K)
        eng.set_clusters(K, ref)
        eng.estep(K)
        eng.mstep(K)
        eng.constants(K)
        got = eng.get_clusters(K)
    oracle64.estep(soa, ref, K)
    oracle64.mstep(soa, ref, K)
    oracle64.constants(ref, K)
    assert_params_close(got, ref, K)


def test_mstep_tensor_large_clusters_and_outliers(loaded, oracle64):
    """Tensor M-step with clusters of 50k-180k events (long exact accumulation chains: every 128-event chain of a big
    cluster is close to the 2^24-quanta budget) and with a few far outliers in the data (they widen the fixed-point
    quanta of the feature rows: the statistics stay unbiased, inside the per-call 1e-4 bar)."""
    pkg = loaded
    N, D, K = 400_000, 24, 3
    ev = pkg.synth.make_blobs(N, D, K, seed=808)
    for variant in ("plain", "outliers"):
        if variant == "outliers":
            ev = ev.copy()
            sd = ev.std(0)
            ev[1000] += 20.0 * sd              # 20 global standard deviations away in every dimension
            ev[250_000, 3] -= 40.0 * sd[3]
        ref = fitted_params(pkg, oracle64, ev, K, iters=2)
        soa = oracle64.transpose(ev)
        with pkg.Engine(ev, K) as eng:
            eng.set_option("path", pkg.PATH_TENSOR)
            eng.seed(K)
            eng.set_clusters(K, ref)
            eng.estep(K)
            eng.mstep(K)
            eng.constants(K)
            got = eng.get_clusters(K)
            assert eng.profile()["mstep_tensor_launches"] == 1
        oracle64.estep(soa, ref, K)
        oracle64.mstep(soa, ref, K)
        oracle64.constants(ref, K)
        assert_params_close(got, ref, K)


def test_mstep_extreme_outlier_uses_fp64_kernel(loaded, oracle64):
    """An outlier beyond 64 global standard deviations leaves the tensor M-step's fixed-point budget: GMM_PATH_AUTO runs
    the FP64 SIMT M-step for that data set (per-call parity unchanged), GMM_PATH_TENSOR reports the condition."""
    pkg = loaded
    N, D, K = 50_000, 8, 4
    ev = pkg.synth.make_blobs(N, D, K, seed=99).copy()
    ev[77, 2] += 500.0 * float(ev[:, 2].std())
    ref = fitted_params(pkg, oracle64, ev, K, iters=2)
    soa = oracle64.transpose(ev)
    with pkg.Engine(ev, K) as eng:
        eng.seed(K)
        eng.set_clusters(K, ref)
        eng.estep(K)
        eng.mstep(K)
        eng.constants(K)
        got = eng.get_clusters(K)
        p = eng.profile()
        assert p["mstep_tensor_launches"] == 0 and p["mstep_simt_launches"] == 1
    oracle64.estep(soa, ref, K)
    oracle64.mstep(soa, ref, K)
    oracle64.constants(ref, K)
    assert_params_close(got, ref, K)
    with pkg.Engine(ev, K) as eng:
        eng.set_option("path", pkg.PATH_TENSOR)
        with pytest.raises(pkg.GmmError):
            eng.seed(K)


@pytest.mark.parametrize("path", PATHS)
def test_seed_parity(loaded, oracle64, path):
    pkg = loaded
    ev = pkg.synth.make_blobs(10_000, 4, 8)
    K = 8
    ref = pkg.Clusters(K, 4, ev.shape[0])
    oracle64.seed(ev, K, ref)
    with pkg.Engine(ev, K) as eng:
        eng.set_option("path", path_id(pkg, path))
        got = eng.seed(K)
    np.testing.assert_array_equal(got.means, ref.means)
    np.testing.assert_array_equal(got.N, ref.N)
    np.testing.assert_allclose(got.avgvar, ref.avgvar, rtol=1e-5)
    assert_params_close(got, ref, K)


@pytest.mark.parametrize("path", PATHS)
def test_em_config1_100_iters(loaded, oracle64, path):
    """BASELINE config 1: N=10k, D=4, K=8, the reference's fixed 100 iterations."""
    pkg = loaded
    cfg = pkg.synth.CONFIGS["c1"]
    ev = pkg.synth.make_blobs(cfg["N"], cfg["D"], cfg["K"])
    K = cfg["K"]
    ref = pkg.Clusters(K, cfg["D"], cfg["N"])
    oracle64.seed(ev, K, ref)
    ll_ref, it_ref = oracle64.em(oracle64.transpose(ev), ref, K, 100, 100)
    with pkg.Engine(ev, K) as eng:
        eng.set_option("path", path_id(pkg, path))
        eng.seed(K)
        ll, it = eng.em(K, 100, 100)
        got = eng.get_clusters(K, with_memberships=True)
    assert it == it_ref == 100
    assert abs(ll - ll_ref) <= 1e-5 * abs(ll_ref)
    run_level_check(got, ref, K, path)


@pytest.mark.parametrize("path", PATHS)
def test_em_config2_slice(loaded, oracle64, path):
    """BASELINE config 2 shape (D=16, K=32) on a 100k-event slice, 10 iterations
    (the oracle finishes in seconds); the full 1M/50-iteration run is covered by
    the size-independent properties below."""
    pkg = loaded
    N, D, K = 100_000, 16, 32
    ev = pkg.synth.make_blobs(N, D, K)
    ref = pkg.Clusters(K, D, N)
    oracle64.seed(ev, K, ref)
    ll_ref, _ = oracle64.em(oracle64.transpose(ev), ref, K, 10, 10)
    with pkg.Engine(ev, K) as eng:
        eng.set_option("path", path_id(pkg, path))
        eng.seed(K)
        ll, it = eng.em(K, 10, 10)
        got = eng.get_clusters(K, with_memberships=True)
    assert it == 10
    assert abs(ll - ll_ref) <= 1e-5 * abs(ll_ref)
    run_level_check(got, ref, K, path)


@pytest.mark.parametrize("path", PATHS)
def test_em_config5_slice(loaded, oracle64, path):
    """BASELINE config 5 shape (D=24, K=128: two 64-cluster passes on the tensor path) on a
    40k-event slice, 5 iterations.  128 clusters on 32 blobs: four clusters compete for each blob, so a
    handful of boundary events (3 of 5.1M on a B200) move by up to 1.2e-2 on the tensor path
    (scripts/exp_gsplit.py); parameters stay inside the run-level bars."""
    pkg = loaded
    N, D, K = 40_000, 24, 128
    ev = pkg.synth.make_blobs(N, D, 32, seed=55)
    ref = pkg.Clusters(K, D, N)
    oracle64.seed(ev, K, ref)
    ll_ref, _ = oracle64.em(oracle64.transpose(ev), ref, K, 5, 5)
    with pkg.Engine(ev, K) as eng:
        eng.set_option("path", path_id(pkg, path))
        eng.seed(K)
        ll, it = eng.em(K, 5, 5)
        got = eng.get_clusters(K, with_memberships=True)
    assert it == 5
    assert abs(ll - ll_ref) <= 1e-5 * abs(ll_ref)
    # 128 clusters on 32 blobs (~300 events each, four clusters per blob): EM is near-degenerate here — the reference's
    # OWN FP32 arithmetic moves responsibilities by 2.0e-4 (1.6x the 1e-3 / 1e-5 bar) against exact arithmetic in these
    # 5 iterations, a 1e-7 per-call perturbation (SIMT path) grows to 2e-4, the tensor path's 2e-6 to 1.3e-3.
    run_level_check(got, ref, K, path, memb=dict(rtol=1e-3, atol=1e-5 if path == "simt" else 3e-3), rtol=5e-4)


@pytest.mark.parametrize("path", PATHS)
def test_em_convergence_rule(loaded, oracle64, path):
    """min_iters < max_iters: the epsilon test of gaussian.cu:532 decides."""
    pkg = loaded
    ev = pkg.synth.make_blobs(6_000, 3, 3, seed=4)
    K = 3
    ref = pkg.Clusters(K, 3, ev.shape[0])
    oracle64.seed(ev, K, ref)
    ll_ref, it_ref = oracle64.em(oracle64.transpose(ev), ref, K, 2, 60)
    with pkg.Engine(ev, K) as eng:
        eng.set_option("path", path_id(pkg, path))
        eng.seed(K)
        ll, it = eng.em(K, 2, 60)
    assert 2 <= it_ref < 60
    assert it == it_ref
    assert abs(ll - ll_ref) <= 1e-5 * abs(ll_ref)


@pytest.mark.parametrize("path", PATHS)
def test_fit_order_reduction(loaded, oracle64, path):
    """gmm_fit: final cluster count integer-exact, best configuration equal."""
    pkg = loaded
    ev = pkg.synth.make_blobs(8_000, 4, 4, seed=12)
    K0 = 8
    c, s = pkg.Clusters(K0, 4, ev.shape[0]), pkg.Clusters(K0, 4, ev.shape[0])
    ideal_ref, mr_ref = oracle64.fit(ev, K0, 0, 20, 20, c, s)
    with pkg.Engine(ev, K0) as eng:
        eng.set_option("path", path_id(pkg, path))
        ideal, mr, saved = eng.fit(K0, 0, 20, 20, with_memberships=True)
    assert ideal == ideal_ref
    assert abs(mr - mr_ref) <= 1e-5 * abs(mr_ref)
    assert_params_close(saved, s, ideal, rtol=5e-4)
    assert_memb_close(saved.memberships[:ideal], s.memberships[:ideal], **RUN_MEMB)
    # explicit target
    ideal_ref3, _ = oracle64.fit(ev, K0, 3, 20, 20, c, s)
    with pkg.Engine(ev, K0) as eng:
        eng.set_option("path", path_id(pkg, path))
        ideal3, _, saved3 = eng.fit(K0, 3, 20, 20)
    assert ideal3 == ideal_ref3 == 3
    assert_params_close(saved3, s, 3, rtol=5e-4)


@pytest.mark.parametrize("path", PATHS)
def test_fit_config5_shape(loaded, oracle64, path):
    """Order-reduction loop at the config-5 shape (D=24, more than 64 clusters, reduced to a target):
    the tensor path runs the two-pass E-step while K > 64 and the single-pass one afterwards."""
    pkg = loaded
    N, D, K0, target = 12_000, 24, 72, 60
    ev = pkg.synth.make_blobs(N, D, 24, seed=77)
    c, s = pkg.Clusters(K0, D, N), pkg.Clusters(K0, D, N)
    ideal_ref, mr_ref = oracle64.fit(ev, K0, target, 3, 3, c, s)
    with pkg.Engine(ev, K0) as eng:
        eng.set_option("path", path_id(pkg, path))
        ideal, mr, saved = eng.fit(K0, target, 3, 3)
    assert ideal == ideal_ref
    assert abs(mr - mr_ref) <= 1e-4 * abs(mr_ref)
    # ~170 events per cluster for 325 moments each, 13 model orders
    assert_params_close(saved, s, ideal, rtol=5e-4 if path == "simt" else 2e-3, rtol_N=5e-4 if path == "simt" else 2e-3)


@pytest.mark.parametrize("path", PATHS)
def test_full_size_properties_config2(loaded, path):
    """Config 2 at full size (N=1M, D=16, K=32): size-independent properties —
    responsibilities sum to 1, sum_k N_k = N, covariances symmetric positive
    definite, log-likelihood non-decreasing (up to the regulariser), rerun
    bit-stable in the parameters to 1e-6."""
    pkg = loaded
    cfg = pkg.synth.CONFIGS["c2"]
    ev = pkg.synth.make_blobs(cfg["N"], cfg["D"], cfg["K"])
    K, N = cfg["K"], cfg["N"]
    with pkg.Engine(ev, K) as eng:
        eng.set_option("path", path_id(pkg, path))
        eng.seed(K)
        lls = []
        for i in range(6):
            ll, _ = eng.em(K, 1, 1) if i else (eng.estep(K), 0)
            lls.append(ll)
        got = eng.get_clusters(K, with_memberships=True)
    assert all(b >= a - 1e-5 * abs(a) for a, b in zip(lls, lls[1:])), lls
    np.testing.assert_allclose(got.memberships.sum(0), 1.0, atol=1e-5)
    assert abs(float(got.N.astype(np.float64).sum()) - N) < 1e-4 * N
    for k in range(K):
        np.testing.assert_array_equal(got.R[k], got.R[k].T)
        assert np.all(np.linalg.eigvalsh(got.R[k].astype(np.float64)) > 0)
    np.testing.assert_allclose(got.pi.sum(), 1.0, rtol=1e-5)


def test_upload_events_equals_fresh_context(loaded):
    """gmm_upload_events replaces the shard in place: same results as a new context."""
    pkg = loaded
    ev = pkg.synth.make_blobs(30_000, 16, 6, seed=31)
    K = 6
    with pkg.Engine(ev, K) as eng:
        eng.seed(K)
        ll_a, _ = eng.em(K, 4, 4)
        a = eng.get_clusters(K)
    with pkg.Engine(np.zeros_like(ev), K) as eng:
        eng.seed(K)                                   # moments of the placeholder data must not survive
        eng.upload_events(ev)
        eng.seed(K)
        ll_b, _ = eng.em(K, 4, 4)
        b = eng.get_clusters(K)
    assert ll_a == ll_b
    for f in ("N", "means", "R", "Rinv", "constant", "pi"):
        np.testing.assert_array_equal(getattr(a, f), getattr(b, f))


def test_reference_binary_matches_oracle_and_engine(loaded, oracle64):
    """The output of the UNMODIFIED reference program (oracle/_ref/gaussianMPI_ref) on a B200 — config 1, 20 iterations,
    stored as tests/golden/ref_c1_it20.summary and the responsibilities of the first 2000 events,
    ref_c1_it20.memberships.npy (tests/golden/make_ref_golden.sh) — against the oracle and the engine: pins both to the
    reference."""
    pkg = loaded
    import sys
    sys.path.insert(0, os.path.dirname(__file__))
    from test_oracle import GOLDEN, _parse_summary
    N, D, K, iters = 10_000, 4, 8, 20
    ev = pkg.synth.make_blobs(N, D, K)
    golden = _parse_summary(os.path.join(GOLDEN, "ref_c1_it20.summary"))
    assert len(golden) == K
    memb_ref = np.load(os.path.join(GOLDEN, "ref_c1_it20.memberships.npy"))
    assert memb_ref.shape == (2000, K)
    cl = pkg.Clusters(K, D, N)
    oracle64.seed(ev, K, cl)
    oracle64.em(oracle64.transpose(ev), cl, K, iters, iters)
    with pkg.Engine(ev, K) as eng:
        eng.seed(K)
        eng.em(K, iters, iters)
        got = eng.get_clusters(K, with_memberships=True)
    for who, c in (("oracle", cl), ("engine", got)):
        for k in range(K):
            g = golden[k]
            assert abs(c.pi[k] - g["pi"]) < 2e-5, who
            np.testing.assert_allclose(c.means[k], g["means"], atol=2e-3, err_msg=who)
            np.testing.assert_allclose(c.R[k], np.array(g["R"]), atol=2e-3, err_msg=who)
        np.testing.assert_allclose(c.memberships[:, :2000].T, memb_ref, rtol=1e-3, atol=1e-5 + 1e-6, err_msg=who)


def test_cli_end_to_end(loaded, oracle64, tmp_path):
    pkg = loaded
    exe = os.path.join(ROOT, "cuda-gmm-mpi_b200", "gaussianMPI_b200")
    N, D, K0 = 5_000, 3, 5
    ev = pkg.synth.make_blobs(N, D, 3, seed=6)
    data = tmp_path / "d.bin"
    pkg.synth.write_bin(str(data), ev)
    env = dict(os.environ, GMM_ITERS="15", GMM_GPUS="1")
    r = subprocess.run([exe, str(K0), str(data), str(tmp_path / "out"), "3"], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    import sys
    sys.path.insert(0, os.path.dirname(__file__))
    from test_oracle import _parse_summary
    got = _parse_summary(str(tmp_path / "out.summary"))
    c, s = pkg.Clusters(K0, D, N), pkg.Clusters(K0, D, N)
    ideal = oracle64.fit(ev, K0, 3, 15, 15, c, s)[0]
    assert ideal == 3 == len(got)
    for k in range(3):
        np.testing.assert_allclose(got[k]["means"], s.means[k], atol=2e-3)
        np.testing.assert_allclose(np.array(got[k]["R"]), s.R[k], atol=2e-3)
    rows = open(tmp_path / "out.results").read().splitlines()
    assert len(rows) == N
    m = np.array([float(v) for v in rows[17].split("\t")[1].split(",")])
    np.testing.assert_allclose(m, s.memberships[:3, 17], atol=2e-4)


def test_cli_csv_input_equals_bin(loaded, tmp_path):
    """The CLI's two input routes — `.bin` streamed from the file to the device shard by shard, anything else parsed as
    comma-separated text with one header line into host memory (readData.cpp:49-129) — give the same output files."""
    pkg = loaded
    exe = os.path.join(ROOT, "cuda-gmm-mpi_b200", "gaussianMPI_b200")
    N, D, K0 = 3_000, 4, 4
    ev = pkg.synth.make_blobs(N, D, 3, seed=16)
    # values that survive the text round trip exactly (atof of %.9g is the same float)
    pkg.synth.write_bin(str(tmp_path / "d.bin"), ev)
    with open(tmp_path / "d.csv", "w") as f:
        f.write(",".join(f"col{i}" for i in range(D)) + "\n")
        for row in ev:
            f.write(",".join("%.9g" % float(v) for v in row) + "\n")
    env = dict(os.environ, GMM_ITERS="8", GMM_GPUS="1")
    outs = []
    for name in ("d.bin", "d.csv"):
        r = subprocess.run([exe, str(K0), str(tmp_path / name), str(tmp_path / ("out_" + name)), "3"], capture_output=True, text=True,
                           env=env, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
        outs.append((open(str(tmp_path / ("out_" + name)) + ".summary").read(), open(str(tmp_path / ("out_" + name)) + ".results").read()))
    assert outs[0][0] == outs[1][0]
    assert outs[0][1] == outs[1][1]


@pytest.mark.skipif(gpu_count() < 2, reason="needs >= 2 GPUs")
def test_cli_two_gpus_equals_one(loaded, tmp_path):
    """Sharded run == single-GPU run (one NCCL all-reduce of the packed statistics)."""
    pkg = loaded
    exe = os.path.join(ROOT, "cuda-gmm-mpi_b200", "gaussianMPI_b200")
    ev = pkg.synth.make_blobs(20_001, 4, 4, seed=2)
    data = tmp_path / "d.bin"
    pkg.synth.write_bin(str(data), ev)
    import sys
    sys.path.insert(0, os.path.dirname(__file__))
    from test_oracle import _parse_summary
    outs = {}
    for g in (1, 2):
        env = dict(os.environ, GMM_ITERS="10", GMM_GPUS=str(g))
        r = subprocess.run([exe, "4", str(data), str(tmp_path / f"o{g}"), "4"], capture_output=True, text=True, env=env, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
        outs[g] = _parse_summary(str(tmp_path / f"o{g}.summary"))
    assert len(outs[1]) == len(outs[2]) == 4
    for a, b in zip(outs[1], outs[2]):          # only the summation order differs between the two runs
        assert abs(a["N"] - b["N"]) <= 1e-4 * a["N"]
        assert abs(a["pi"] - b["pi"]) <= 2e-6
        np.testing.assert_allclose(a["means"], b["means"], atol=1.1e-3)
        np.testing.assert_allclose(np.array(a["R"]), np.array(b["R"]), atol=1.1e-3)


@pytest.mark.parametrize("N,D,K", [(70_001, 24, 64), (33_333, 8, 5)])
def test_tensor_steps_rerun_bit_stable(loaded, N, D, K):
    """Stress of the asynchronous hand-overs inside the tensor kernels (TMA stage release, operand stages, accumulator
    drains, the E-step's TMEM hand-over): 40 E-step + M-step repetitions from identical inputs must be bit-identical —
    a refill that overtakes a pending load, or a drain that races an MMA, shows up as run-to-run differences (the
    stage-release race of round 1 did)."""
    pkg = loaded
    ev = pkg.synth.make_blobs(N, D, min(K, 8), seed=321)
    with pkg.Engine(ev, K) as eng:
        eng.set_option("path", pkg.PATH_TENSOR)
        start = eng.seed(K)
        first = None
        for rep in range(40):
            eng.set_clusters(K, start)
            ll = eng.estep(K)
            eng.mstep(K)
            got = eng.get_clusters(K, with_memberships=(rep % 10 == 0))
            cur = (ll, got.N.copy(), got.means.copy(), got.R.copy())
            if first is None:
                first, memb0 = cur, got.memberships.copy()
            else:
                assert cur[0] == first[0], rep
                for a, b in zip(cur[1:], first[1:]):
                    np.testing.assert_array_equal(a, b, err_msg=f"repetition {rep}")
                if got.memberships is not None:
                    np.testing.assert_array_equal(got.memberships, memb0, err_msg=f"repetition {rep}")
