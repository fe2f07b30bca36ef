"""CPU tier: the C-ABI library loads and exports every symbol include/gprc.h declares, fails loudly without a GPU,
the product never touches the oracle, and the host-side logic (kernel closures, reshape rules, optimisers, sharding)
behaves like the reference."""
import ast
import math
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "gaussian-process-regression_b200")


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "gprc.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(gprc_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(gprc):
    lib = gprc._lib.load()
    names = declared_symbols()
    assert len(names) >= 40
    for n in names:
        assert hasattr(lib, n), "libgprc.so does not export %s" % n
    # and the ctypes table binds exactly the header
    assert sorted(gprc._lib.SIGNATURES) == names
    assert lib.gprc_version() == 100


def test_alias_survives_importing_every_test_module(gprc):
    """Round 1's GPU tier went red because `from gprc_b200.fit import ...` in a test module re-imported fit.py under the
    alias and rebound the package attribute `fit` from the function to a module.  Import every test module in pytest's
    collection order (alphabetical) and check that the alias and the real package are still one set of objects."""
    import importlib
    real = importlib.import_module("gaussian-process-regression_b200")
    tests_dir = os.path.join(ROOT, "tests")
    if tests_dir not in sys.path:
        sys.path.insert(0, tests_dir)
    for f in sorted(os.listdir(tests_dir)):
        if f.startswith("test_") and f.endswith(".py"):
            importlib.import_module(f[:-3])
            assert callable(gprc.fit) and not isinstance(gprc.fit, type(os)), "gprc.fit rebound after importing " + f
    assert gprc is real
    assert gprc.Objective is importlib.import_module("gaussian-process-regression_b200.fit").Objective
    for name, mod in list(sys.modules.items()):
        if name.startswith("gprc_b200.") and mod is not None:
            assert mod is sys.modules["gaussian-process-regression_b200" + name[len("gprc_b200"):]], name
    for attr in ("fit", "GPR", "GPC", "cov_func", "multistart", "optim_until_error"):
        assert callable(getattr(gprc, attr)), attr


def test_no_gpu_fails_loudly(gprc):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(gprc.GprcError, match="no CUDA device"):
        gprc.Context(0)
    with pytest.raises(gprc.GprcError):
        gprc.GPR(np.array([[1.0, 2.0]]), np.array([0.0, 1.0]), 1.0, gprc.cov_func(gprc.sqrexp, l=1.0))


def test_sass_has_fp64_tensor_and_tma_instructions():
    so = os.path.join(PKG, "libgprc.so")
    out = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True).stdout
    assert "DMMA.8x8x4" in out, "no FP64 tensor-core instructions in libgprc.so"
    assert "UBLKCP" in out, "no TMA bulk copies in libgprc.so"
    assert "SYNCS.ARRIVE.TRANS64" in out, "no mbarrier transactions in libgprc.so"


def test_product_never_imports_the_oracle():
    for dirpath, _, files in os.walk(PKG):
        for f in files:
            if f.endswith(".py"):
                tree = ast.parse(open(os.path.join(dirpath, f)).read())
                for node in ast.walk(tree):
                    mods = []
                    if isinstance(node, ast.Import):
                        mods = [a.name for a in node.names]
                    elif isinstance(node, ast.ImportFrom):
                        mods = [node.module or ""]
                    assert not any(m.split(".")[0] == "oracle" for m in mods), (f, mods)
    for f in os.listdir(os.path.join(PKG, "csrc")):
        assert "oracle" not in open(os.path.join(PKG, "csrc", f)).read()


def test_cov_func_carries_kernel_spec(gprc):
    k = gprc.cov_func(gprc.rationalquadratic, l=1.5, alpha=0.5)
    assert k.gprc_kernel.name == "rationalquadratic" and k.gprc_kernel.params == dict(l=1.5, alpha=0.5)
    k = gprc.cov_func(gprc.gammaexp, 2.0, 1.5)  # positional (l, gamma), the order fit() uses (R/fit.R:118)
    assert k.gprc_kernel.params == dict(l=2.0, gamma=1.5)
    kc, _ = k.gprc_kernel.to_c()
    assert kc.id == 4 and kc.l == 2.0 and kc.gamma == 1.5
    assert gprc.cov_func(lambda x, y: x, 1).gprc_kernel is None      # opaque closure -> host evaluation
    assert gprc.cov_func(gprc.sqrexp).gprc_kernel is None            # parameters missing -> not a complete spec
    x = np.array([[0.0, 1.0], [0.0, 1.0]])
    np.testing.assert_allclose(gprc.cov_func(gprc.sqrexp, l=1.0)(x, x[:, ::-1]), np.exp(-1.0) * np.ones(2))


def test_host_kernels_match_oracle(gprc, oracle):
    rng = np.random.default_rng(0)
    x, y = rng.standard_normal((3, 7)), rng.standard_normal((3, 7))
    for name, args in [("constant", (2.0,)), ("linear", (0.5,)), ("polynomial", (0.3, 3.0)), ("sqrexp", (0.7,)),
                       ("gammaexp", (1.2, 1.5)), ("rationalquadratic", (0.9, 2.0))]:
        np.testing.assert_array_equal(getattr(gprc, name)(x, y, *args), getattr(oracle, name)(x, y, *args))
        assert getattr(gprc, name)(x[:, 0], y[:, 0], *args) == pytest.approx(getattr(oracle, name)(x[:, 0], y[:, 0], *args))


def test_host_optimisers(gprc):
    from importlib import import_module
    opt = import_module("gaussian-process-regression_b200._optim")
    x = opt.brent_fmin(lambda t: math.cos(t), 0.0, 10.0, math.sqrt(opt.EPS))
    assert abs(x - math.pi) < 1e-6
    r = opt.r_optim([1.0], lambda p: -(p[0] - 3.0) ** 2, method="Brent", lower=0.0, upper=10.0)  # fnscale = -1: maximise
    assert abs(r["par"][0] - 3.0) < 1e-6 and abs(r["value"]) < 1e-10
    f = lambda p: -((p[0] - 1) ** 2 + 2 * (p[1] + 0.5) ** 2)
    g = lambda p: np.array([-2 * (p[0] - 1), -4 * (p[1] + 0.5)])
    r = opt.r_optim([0.0, 0.0], f, gr=g, method="BFGS")
    np.testing.assert_allclose(r["par"], [1.0, -0.5], atol=1e-6)


def test_optim_until_error_policy(gprc):
    from importlib import import_module
    opt = import_module("gaussian-process-regression_b200._optim")

    def f(p):  # errors on part of the domain score -10000 (R/fit.R:50)
        if p[0] > 6.0:
            raise opt.OptimError("chol failed")
        return -(p[0] - 5.0) ** 2
    r = gprc.optim_until_error([1.0], f, method="Brent", lower=0.0, upper=10.0)
    assert abs(r["par"][0] - 5.0) < 1e-4

    calls = []

    def f2(p):
        calls.append(tuple(p))
        return -float(np.sum((np.asarray(p) - 2.0) ** 2))

    def bad_gradient(p):  # optim() itself throws -> best recorded evaluation is returned (R/fit.R:58-66)
        raise opt.OptimError("system is computationally singular")
    r = gprc.optim_until_error([1.0, 1.0], f2, gr=bad_gradient, method="BFGS")
    np.testing.assert_array_equal(r["par"], [1.0, 1.0])
    assert r["value"] == -2.0


def test_simulation_helpers(gprc, oracle):
    np.testing.assert_array_equal(gprc.combine_all([[1.0, 2.0], [3.0, 4.0, 5.0]]), oracle.combine_all([[1.0, 2.0], [3.0, 4.0, 5.0]]))
    noise = gprc.iid_noise(lambda n, sd: np.full(n, sd), sd=0.1)
    np.testing.assert_array_equal(noise(np.zeros((3, 5))), np.full(5, 0.1))


@pytest.mark.gpu
def test_multivariate_normal(gprc):
    # mean + t(chol(Sigma)) %*% Z on the device; singular Sigma takes the reference's eigen fallback (R/GPRclass.R:363-368)
    cov = np.array([[1.0, 0.5], [0.5, 1.0]])
    z = gprc.multivariate_normal(4, [0.0, 1.0], cov, rng=np.random.default_rng(0))
    Z = np.random.default_rng(0).standard_normal((2, 4))
    np.testing.assert_allclose(z, np.array([[0.0], [1.0]]) + np.linalg.cholesky(cov) @ Z, rtol=1e-13, atol=1e-14)
    rng = np.random.default_rng(3)
    G = rng.standard_normal((300, 300))
    S = G @ G.T / 300 + 0.1 * np.eye(300)
    z = gprc.multivariate_normal(7, np.arange(300.0), S, rng=np.random.default_rng(1))
    Z = np.random.default_rng(1).standard_normal((300, 7))
    np.testing.assert_allclose(z, np.arange(300.0)[:, None] + np.linalg.cholesky(S) @ Z, rtol=1e-10, atol=1e-10)
    z = gprc.multivariate_normal(3, [0.0, 0.0], np.ones((2, 2)), rng=np.random.default_rng(0))  # singular: eigen path
    np.testing.assert_allclose(z[0], z[1], atol=1e-7)


def _worker(rank, world, port, q):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    import gprc_b200 as g
    from importlib import import_module
    fitmod = import_module("gaussian-process-regression_b200.fit")
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    seen = []

    class FakeObjective:  # stands in for the GPU objective: the sharding/merge logic is what is under test
        def __init__(self, *a, **k):
            pass

    def fake_fit_one(obj, cov, engine="host"):
        seen.append(cov)
        score = {"sqrexp": -3.0, "gammaexp": -2.5, "constant": -9.0, "linear": -1.0, "polynomial": -4.0,
                 "rationalquadratic": -2.0}[cov]
        return dict(par=np.array([len(cov) * 1.0]), value=score)
    fitmod.Objective = FakeObjective
    fitmod._fit_one = fake_fit_one
    r = fitmod.fit(np.zeros((1, 3)), np.zeros(3), 0.1, group=dist.group.WORLD, verbose=False)
    q.put((rank, r["cov"], [float(s) for s in r["score"]], sorted(seen), float(r["par"][0])))
    dist.destroy_process_group()


def test_fit_shards_kernel_families_over_ranks_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 1000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    names = ["sqrexp", "gammaexp", "constant", "linear", "polynomial", "rationalquadratic"]
    assert res[0][3] == sorted(names[0::2]) and res[1][3] == sorted(names[1::2])   # dealt round-robin, no overlap
    for rank, cov, score, _, par in res:
        assert cov == "linear" and par == 6.0                                       # which.max over the merged scores
        assert score == [-3.0, -2.5, -9.0, -1.0, -4.0, -2.0]                        # in cov_names order on every rank


def test_bench_test_point_shards_cover_exactly():
    m = 1000000
    for world in (1, 2, 4, 8, 3):
        cuts = [(r * m // world, (r + 1) * m // world) for r in range(world)]
        assert cuts[0][0] == 0 and cuts[-1][1] == m
        assert all(a[1] == b[0] for a, b in zip(cuts, cuts[1:]))


def _build_c_client(tmp_path):
    exe = str(tmp_path / "c_abi_smoke")
    subprocess.run(["gcc", "-std=c11", "-Wall", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "c_abi_smoke.c"),
                    "-L" + PKG, "-lgprc", "-lm", "-o", exe], check=True)
    return exe


def test_plain_c_client_links_against_the_abi(tmp_path):
    """include/gprc.h is a C header and libgprc.so links into a C program with no C++/Python/R in sight; without a GPU
    the client reports the loud failure of gprc_ctx_create."""
    exe = _build_c_client(tmp_path)
    import torch
    if torch.cuda.is_available():
        pytest.skip("covered by the gpu test")
    r = subprocess.run([exe], env=dict(os.environ, LD_LIBRARY_PATH=PKG), capture_output=True, text=True)
    assert r.returncode == 2 and "no CUDA device" in r.stdout


@pytest.mark.gpu
def test_plain_c_client_reproduces_known_answers(tmp_path):
    exe = _build_c_client(tmp_path)
    r = subprocess.run([exe], env=dict(os.environ, LD_LIBRARY_PATH=PKG), capture_output=True, text=True)
    assert r.returncode == 0, r.stdout
    assert "all known answers reproduced through the C ABI" in r.stdout


def test_int8_digit_arithmetic_host_selftest():
    """csrc/ozaki.cuh: the fixed-point digit split used by the INT8 variance pass, compiled for the host by
    tools/oz_test: exact reconstruction, int8 digit range, overflow flag, int32 headroom of the drain interval,
    shared-memory / TMEM budgets -- for 6, 7 and 8 digits."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    tool = os.path.join(root, "tools", "oz_test")
    if not os.path.exists(tool):
        import __graft_entry__ as ge
        ge.build()
    out = subprocess.run([tool, "digits"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    assert out.stdout.count(" 0 failures") == 5, out.stdout


@pytest.mark.parametrize("path,tile,trtri", [(4, 2, 0.0), (4, 1, 0.0), (4, 64, 0.0), (4, 128, 0.0), (2, 64, 0.0), (1, 64, 1200.0)])
def test_bench_roofline_block_is_serialisable(path, tile, trtri):
    """bench.roofline_block (pure function): the INT8 pass reports against the INT8 pipe (measured peak of the run when
    given, frac < 1) with the FP64 view beside it; the FP64 passes against cuBLAS Dgemm; no pasted traffic constants.
    Guards the last lines of a minutes-long GPU run."""
    import json
    import types
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if root not in sys.path:
        sys.path.insert(0, root)
    import bench
    args = types.SimpleNamespace(ozaki_digits=7, int8_tile=tile)
    timers = dict(build_k=9.0, chol=1240.0, solve=19.0, trtri=trtri, build_ks=400.0, var=22000.0, newton=0.0, predict=22500.0)
    n, m = 50000, 1000000
    flops = float(n) * n * m
    achieved = flops / (timers["var"] * 1e-3) / 1e12
    peak = dict(burst_tops=4700.0, sustained_tops=3900.0, clk_per_mma=128.4, seconds=2.0)
    r = bench.roofline_block(args, path, timers, achieved, 35.5, flops, timers["var"], 24.0, n, m_local=m, int8_peak=peak,
                             variant=tile, chunks=14)
    line = json.loads(json.dumps(dict(roofline=r)))["roofline"]
    for key in ("kernel", "bound", "achieved", "peak", "unit", "frac", "traffic", "predict_path", "ms_per_step",
                "algorithmic_bytes_per_step"):
        assert key in line, key
    assert line["bound"] == "tensor" and line["unit"] == "TFLOP/s"
    assert abs(line["frac"] - line["achieved"] / line["peak"]) < 1e-12
    assert abs(line["algorithmic_bytes_per_step"] - (14 * 8 * n * n / 2 + 16.0 * n * m)) < 1.0
    if path == 4:
        assert line["peak"] == 3900.0 and "of measured" in line["peak_source"]
        assert line["frac"] < 1.0 and line["fp64_equivalent"]["frac"] > 1.5
        assert set(line["peaks"]) == {"measured_sustained", "measured_burst", "proxy_2x_bf16_sustained", "nominal"}
        assert line["int8_products_per_fp64_product"] == 28
        assert ("update128" in line["kernel"]) == (tile == 128) and ("stack" in line["kernel"]) == (tile in (1, 2))
        # V digits cross HBM once per 256 rows of L on cluster pairs, once per 128 otherwise
        assert line["v_digit_stream_bytes"] == pytest.approx({2: 0.5, 1: 1.0, 64: 1.0, 128: 10 / 7}[tile] * 7 * m * 128 *
                                                              sum(range(391)), rel=1e-12)
        proxy = bench.roofline_block(args, path, timers, achieved, 35.5, flops, timers["var"], 24.0, n, variant=tile)
        assert "proxy" in proxy["peak_source"] or "fallback" in proxy["peak_source"]
    else:
        assert "fp64_equivalent" not in line and abs(line["achieved"] - achieved) < 1e-9
    assert bench.roofline_block(args, path, timers, None, 35.5, flops, timers["var"], 24.0, n, variant=tile)["frac"] is None


def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs: the caller's arrays of the last step as float64 .npy files, every test point while they
    fit the size limit, beyond it the same seeded sample in every run."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if root not in sys.path:
        sys.path.insert(0, root)
    import bench
    m = 1000
    mean, var = np.linspace(-2.0, 3.0, m), np.linspace(0.0, 1.0, m)
    bench.dump_outputs(str(tmp_path / "out"), mean, var, -1.5, 0, m, 0, 1)
    for name, want in (("mean", mean), ("var", var), ("logp", [-1.5])):
        got = np.load(tmp_path / "out" / (name + ".npy"))
        assert got.dtype == np.float64
        np.testing.assert_array_equal(got, want)
    big = bench.DUMP_LIMIT // 8
    idx = bench.dump_index(big)
    assert 0.99 * bench.DUMP_LIMIT < 16 * len(idx) < bench.DUMP_LIMIT - 1024
    assert np.all(np.diff(idx) > 0) and idx[-1] < big
    np.testing.assert_array_equal(idx, bench.dump_index(big))


def _load_protocol_sim(mutate=None):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = open(os.path.join(root, "tools", "oz_protocol_sim.py")).read()
    if mutate is not None:
        old, new = mutate
        assert old in src
        src = src.replace(old, new)
    ns = {}
    exec(compile(src, "oz_protocol_sim", "exec"), ns)
    return ns


def test_int8_kernel_barrier_protocols_model():
    """tools/oz_protocol_sim.py: the producer / MMA / drain roles of the INT8 kernels (single CTA, wide two-pass, and the
    cluster-pair kernel with multicast V stages) replayed with the kernels' slot / phase / count arithmetic under random
    latencies: no deadlock, every MMA reads the k-step it expects in every CTA, no stage overwritten or ring re-partitioned
    under outstanding reads, accumulators never written during a drain."""
    assert _load_protocol_sim()["campaign"](10) == []


@pytest.mark.parametrize("mutation", [
    ('            if passes == 2 and r > 0:\n                yield ("wait", pass_done[c], (r - 1) & 1)', "            pass"),
    ("                if need_wait:", "                if False:"),
    ("EMPTY_COUNT = 2 ", "EMPTY_COUNT = 1 "),   # cluster pairs: a slot refilled after ONE CTA's commit instead of both
])
def test_protocol_model_detects_injected_bugs(mutation):
    """The model must have teeth: dropping the pass_done wait or the empty wait, or letting the cluster pair refill a slot
    after only one CTA's commit, is caught."""
    assert len(_load_protocol_sim(mutation)["campaign"](3)) > 0


def test_bench_cpu_arms_run_at_reduced_size():
    """bench.py's CPU legs (the only places outside tests/ that may execute oracle/): the bounded sample of the GPU arm and
    the --impl reference pass, at sizes that take seconds, checked for internal consistency (the reference pass reproduces
    the oracle's logp on its sample; generous <= literal; scaling laws of the phases)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if root not in sys.path:
        sys.path.insert(0, root)
    import bench
    from oracle import gprc_oracle as o
    s = bench.cpu_sample(4000, 20000, 8, 1024, 256)
    assert s["kind"] == "port" and s["cores"] >= 1 and 0 < s["value"] <= s["literal_value"]
    assert "scaled, not run" in s["sample"]
    r = bench.cpu_reference_full(3000, 20000, 8, 512, n_train=1536)
    assert r["value"] > 0 and r["literal_value"] > r["value"] and "REDUCED from 3000" in r["sample"]
    X, y, Xs = bench.make_inputs(3000, 20000, 8)
    ref = o.GPR(X[:, :1536], y[:1536], 0.01, o.cov_func(o.sqrexp, l=1.0))
    got = float(r["sample"].rsplit("logp of the sample ", 1)[1])
    assert abs(got - float(ref.logp)) <= 1e-6 * abs(float(ref.logp))
