"""CPU tests of the product's GPU-free parts: the C-ABI library loads and exports
everything include/gmm.h declares, host numerics (inverse, M-step finalisation,
Rissanen, order reduction) against the oracle, file formats, CLI argument rules."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, random_spd_params, assert_params_close


def test_abi_exports_every_declared_symbol(pkg):
    hdr = open(os.path.join(ROOT, "include", "gmm.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = set(re.findall(r"\b(gmm_[a-z0-9_]+)\s*\(", hdr))
    assert len(names) >= 25
    lib = pkg.load_library()
    missing = [n for n in sorted(names) if not hasattr(lib, n)]
    assert not missing, missing
    out = subprocess.check_output(["nm", "-D", "--defined-only", pkg.library_path()], text=True)
    exported = set(re.findall(r" T (gmm_[a-z0-9_]+)", out))
    assert names <= exported


def test_no_oracle_in_product(pkg):
    """The product must never route through the oracle or any CPU fallback."""
    src_dir = os.path.join(ROOT, "cuda-gmm-mpi_b200")
    for root, _, files in os.walk(src_dir):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                txt = open(os.path.join(root, f)).read()
                assert "gmm_oracle" not in txt and "oracle/" not in txt, f
    out = subprocess.check_output(["ldd", pkg.library_path()], text=True)
    assert "oracle" not in out


def test_compute_fails_loudly_without_gpu(pkg):
    """No visible GPU (none installed, or CUDA_VISIBLE_DEVICES empty): creating a context raises GMM_ERR_CUDA. Run in a
    child process with the devices hidden, so that a machine with a GPU checks it too."""
    code = """if True:
        import sys
        sys.path.insert(0, sys.argv[1])
        import numpy as np
        import __graft_entry__ as entry
        pkg = entry.load_package()
        try:
            pkg.Engine(np.zeros((16, 4), np.float32), 2)
        except pkg.GmmError as ex:
            print("GmmError", ex.code)
    """
    r = subprocess.run([sys.executable, "-c", code, ROOT], capture_output=True, text=True, timeout=300,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.strip().splitlines()[-1] == "GmmError 4", r.stdout + r.stderr


def test_host_invert(pkg, oracle64):
    rng = np.random.default_rng(0)
    for n in (1, 2, 5, 16, 24, 32):
        A = rng.standard_normal((n, n))
        M = (A @ A.T / n + 0.5 * np.eye(n)).astype(np.float32)
        inv, ld = pkg.host_invert(M)
        oinv, old = oracle64.invert(M)
        np.testing.assert_allclose(inv, oinv, rtol=2e-3, atol=2e-4)
        assert abs(ld - old) < 1e-4 * max(1.0, abs(old))
        _, ld10 = pkg.host_invert(M, use_log10=True)
        _, old10 = oracle64.invert(M, use_log10=True)
        if n > 1:
            assert abs(ld10 - old10) < 1e-4 * max(1.0, abs(old10))


def numpy_stats(pkg, ev, memb, shift, K):
    """Packed statistics [K][F] + LL slot, computed in double with numpy."""
    N, D = ev.shape
    x = ev.astype(np.float64) - shift
    F = 1 + D + D * (D + 1) // 2
    stats = np.zeros(K * F + 1)
    tri = [(i, j) for i in range(D) for j in range(i + 1)]
    for k in range(K):
        g = memb[k].astype(np.float64)
        s = stats[k * F:(k + 1) * F]
        s[0] = g.sum()
        s[1:1 + D] = g @ x
        M2 = (x * g[:, None]).T @ x
        s[1 + D:] = [M2[i, j] for i, j in tri]
    return stats


@pytest.mark.parametrize("N,D,K", [(2000, 4, 5), (1500, 1, 3), (3000, 7, 4), (1200, 24, 3)])
def test_host_finalize_matches_oracle_mstep(pkg, oracle64, N, D, K):
    ev = pkg.synth.make_blobs(N, D, K, seed=21)
    ref = random_spd_params(pkg, K, D, np.random.default_rng(4))
    ref.memberships = np.zeros((K, N), np.float32)
    oracle64.constants(ref, K)
    soa = oracle64.transpose(ev)
    oracle64.estep(soa, ref, K)
    memb = ref.memberships.copy()
    got = ref.copy()
    oracle64.mstep(soa, ref, K)
    oracle64.constants(ref, K)
    shift = ev.astype(np.float64).mean(0)
    pkg.host_finalize(numpy_stats(pkg, ev, memb, shift, K), shift, got, K)
    assert_params_close(got, ref, K)


def test_host_finalize_empty_cluster_rules(pkg, oracle64):
    """N < 0.5 -> means 0, R = I, pi = 1e-10; 0.5 < N < 1 -> covariance zeroed
    before the regulariser (gaussian.cu:614-679, gaussian_kernel.cu:658-675,185)."""
    N, D, K = 800, 3, 4
    ev = pkg.synth.make_blobs(N, D, 2, seed=3)
    ref = random_spd_params(pkg, K, D, np.random.default_rng(8))
    ref.memberships = np.zeros((K, N), np.float32)
    memb = ref.memberships
    memb[0] = 0.7; memb[1] = 0.3 - 1e-3
    memb[2] = 0.0; memb[2, 5] = 0.3                      # N = 0.3  (< 0.5)
    memb[3] = 0.0; memb[3, 7] = 0.45; memb[3, 9] = 0.3   # N = 0.75 (0.5 < N < 1.0)
    got = ref.copy()
    soa = oracle64.transpose(ev)
    oracle64.mstep(soa, ref, K)
    oracle64.constants(ref, K)
    shift = ev.astype(np.float64).mean(0)
    pkg.host_finalize(numpy_stats(pkg, ev, memb, shift, K), shift, got, K)
    assert_params_close(got, ref, K)
    np.testing.assert_array_equal(got.R[2], np.eye(D, dtype=np.float32))
    np.testing.assert_array_equal(got.means[2], 0)
    assert got.pi[2] == np.float32(1e-10)


def test_rissanen_epsilon(pkg, oracle64):
    for (D, N, K, ll) in [(4, 10_000, 8, -1.2e5), (24, 10_000_000, 64, -3.3e8), (16, 1_000_000, 32, -2.0e7)]:
        assert pkg.host_epsilon(D, N) == pytest.approx(oracle64.epsilon(D, N), rel=1e-6)
        assert pkg.host_rissanen(ll, K, D, N) == pytest.approx(oracle64.rissanen(ll, K, D, N), rel=1e-6)


def test_reduce_order_matches_oracle(pkg, oracle64):
    N, D, K = 3000, 4, 7
    ev = pkg.synth.make_blobs(N, D, 4, seed=13)
    ref = pkg.Clusters(K, D, N)
    oracle64.seed(ev, K, ref)
    oracle64.em(oracle64.transpose(ev), ref, K, 5, 5)
    ref.N[2] = 0.2                                    # force an "empty" cluster
    got = ref.copy()
    newK_ref, pair_ref = oracle64.reduce_order(ref, K)
    newK, pair = pkg.host_reduce_order(got, K)
    assert newK == newK_ref == K - 2
    assert pair == pair_ref
    assert_params_close(got, ref, newK)


def test_shard_range(pkg):
    for N, G in [(10, 3), (10_000_000, 8), (7, 7), (5, 1)]:
        tot = 0
        for r in range(G):
            b, n = pkg.shard_range(N, G, r)
            assert b == (N // G) * r
            tot += n
        assert tot == N
        assert pkg.shard_range(N, G, G - 1)[1] == N // G + N % G      # remainder to the last shard


def test_read_bin_and_csv(pkg, tmp_path):
    ev = pkg.synth.make_blobs(37, 5, 2, seed=1)
    p = tmp_path / "d.bin"
    pkg.synth.write_bin(str(p), ev)
    np.testing.assert_array_equal(pkg.read_data(str(p)), ev)
    c = tmp_path / "d.csv"
    with open(c, "w") as f:
        f.write("a,b,c,d,e\n")
        for row in ev:
            f.write(",".join(f"{v:.9g}" for v in row) + "\n")
        f.write("\n")
    np.testing.assert_allclose(pkg.read_data(str(c)), ev, rtol=1e-6)
    bad = tmp_path / "bad.csv"
    bad.write_text("a,b,c\n1,2,3\n4,5\n")
    with pytest.raises(pkg.GmmError):
        pkg.read_data(str(bad))


def test_writers_format(pkg, tmp_path):
    K, D, N = 2, 3, 4
    cl = pkg.Clusters(K, D, N)
    cl.pi[:] = [0.25, 0.75]; cl.N[:] = [1, 3]
    cl.means[...] = np.arange(K * D).reshape(K, D)
    cl.R[...] = np.eye(D)
    cl.memberships[...] = np.array([[0.25] * N, [0.75] * N])
    ev = np.arange(N * D, dtype=np.float32).reshape(N, D)
    pkg.write_summary(str(tmp_path / "o.summary"), cl, K)
    pkg.write_results(str(tmp_path / "o.results"), ev, cl, K)
    s = (tmp_path / "o.summary").read_text().splitlines()
    assert s[0] == "Cluster #0" and s[1] == "Probability: 0.250000" and s[2] == "N: 1.000000"
    assert s[3] == "Means: 0.000 1.000 2.000 "
    assert s[5] == "R Matrix:" and s[6] == "1.000 0.000 0.000 "
    r = (tmp_path / "o.results").read_text().splitlines()
    assert r[0] == "0.000000,1.000000,2.000000\t0.250000,0.750000"
    assert len(r) == N


def test_cli_argument_rules(pkg, tmp_path):
    exe = os.path.join(ROOT, "cuda-gmm-mpi_b200", "gaussianMPI_b200")
    assert os.path.exists(exe)
    ev = pkg.synth.make_blobs(64, 2, 2, seed=1)
    data = tmp_path / "d.bin"
    pkg.synth.write_bin(str(data), ev)
    run = lambda *a: subprocess.run([exe, *a], capture_output=True, text=True)
    r = run()
    assert r.returncode == 1 and "Usage:" in r.stdout
    assert run("0", str(data), "out").returncode == 1          # K out of range
    assert run("513", str(data), "out").returncode == 1
    r = run("4", str(tmp_path / "missing.bin"), "out")
    assert r.returncode == 1 and "Invalid infile" in r.stdout
    r = run("4", str(data), "out", "5")
    assert r.returncode == 1 and "target_num_clusters must be less than equal" in r.stdout
    from conftest import have_gpu
    if not have_gpu():
        r = run("4", str(data), str(tmp_path / "out"))
        assert r.returncode == 255 and "No CUDA capable GPUs" in r.stdout     # main returns -1


def test_host_finalize_is_shift_invariant(pkg):
    """The packed statistics may be taken about any centre: the finalised N / means / covariances
    must not depend on the shift (the engine uses the float-rounded global mean)."""
    rng = np.random.default_rng(21)
    N, D, K = 4000, 6, 3
    ev = (rng.standard_normal((N, D)) * rng.uniform(0.5, 2.0, D) + rng.uniform(-30, 30, D)).astype(np.float32)
    memb = rng.dirichlet(np.ones(K), size=N).T.astype(np.float32)
    outs = []
    for shift in (np.zeros(D), ev.mean(0).astype(np.float64), ev.mean(0).astype(np.float64) + 3.0):
        cl = pkg.Clusters(K, D, 0)
        cl.avgvar[:] = 0.01
        pkg.host_finalize(numpy_stats(pkg, ev, memb, shift, K), shift, cl, K)
        outs.append(cl)
    for o in outs[1:]:
        np.testing.assert_allclose(o.N, outs[0].N, rtol=1e-7)
        np.testing.assert_allclose(o.means, outs[0].means, rtol=1e-6, atol=1e-5)
        np.testing.assert_allclose(o.R, outs[0].R, rtol=2e-4, atol=2e-4)      # shift 0 cancels |mu|^2 ~ 900 against sigma^2 ~ 1
        np.testing.assert_allclose(o.constant, outs[0].constant, rtol=1e-4)


def test_results_writer_matches_printf(pkg, tmp_path):
    """gmm_write_results formats with its own "%f" routine (parallel, buffered): digit for digit what printf gives,
    ties, carries, signed zeros, huge values, inf / nan included (gaussian.cu:1044-1058 uses fprintf "%f")."""
    rng = np.random.default_rng(1)
    N, D, K = 5000, 5, 7
    ev = (rng.standard_normal((N, D)) * 10.0 ** rng.integers(-8, 9, (N, 1))).astype(np.float32)
    ev[0] = [0.0, -0.0, 1e-7, -1e-7, 0.9999995]
    ev[1] = [2.5e-7, 3.5e-7, 0.0000005, 1.0000005, 123456789.0]
    ev[2] = [1e14, -1e14, 3e15, 1e20, float("inf")]
    ev[3] = [0.5e-6, 1.5e-6, 2.5e-6, -0.5e-6, -2.5e-6]
    ev[4] = [3.4e38, -3.4e38, float("nan"), 1e-45, 16777216.0]
    ev[5:105] = rng.integers(-3, 3, (100, D)) + 0.5
    ev[105:205] = rng.integers(0, 1000, (100, D)) / 64.0
    cl = pkg.Clusters(K, D, N)
    cl.memberships[...] = rng.random((K, N)).astype(np.float32)
    path = str(tmp_path / "t.results")
    pkg.write_results(path, ev, cl, K)
    lines = open(path).read().splitlines()
    assert len(lines) == N
    for i in range(N):
        exp = ",".join("%f" % float(v) for v in ev[i]) + "\t" + ",".join("%f" % float(v) for v in cl.memberships[:, i])
        assert lines[i] == exp, i


def test_host_worker_team_selftest(pkg):
    """The persistent worker team of the per-iteration host finalisation: thousands of back-to-back parallel loops of
    varying size (and team re-creation, and sleeping workers) — every item exactly once, no lost wake-up, no deadlock."""
    lib = pkg.load_library()
    for threads, jobs, n in ((1, 50, 7), (2, 3000, 64), (8, 3000, 80), (16, 1500, 5)):
        assert lib.gmm_host_pool_selftest(threads, jobs, n) == 0, lib.gmm_last_error()


def test_every_runtime_option_is_documented():
    """Every key gmm_set_option accepts (csrc/gmm_api.cu) is described in the C header and in INTEGRATION.md."""
    import os
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = open(os.path.join(root, "cuda-gmm-mpi_b200", "csrc", "gmm_api.cu")).read()
    body = src[src.index("int gmm_set_option("):]
    body = body[:body.index("\n}\n")]
    keys = set(re.findall(r'k == "([a-z_]+)"', body))
    assert {"path", "finalize", "allreduce", "host_threads", "profile"} <= keys
    header = open(os.path.join(root, "include", "gmm.h")).read()
    integ = open(os.path.join(root, "INTEGRATION.md")).read()
    for k in keys:
        assert f'"{k}"' in header, f"option {k} is not documented in include/gmm.h"
        if k != "finalize_fault_iter":                 # test hook: header only
            assert f"`{k}`" in integ, f"option {k} is not documented in INTEGRATION.md"
