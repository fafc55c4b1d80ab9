"""Host-side logic that needs no GPU: kernel recognition (duck typing of the reference's kernel
objects), descriptor filling, argument parsing of the two recombination signatures, shard maths."""
import math

import pytest
import torch

from basq_b200 import _lib, _rchq, kernels, sharded
from oracle import gp_kernels as ogp


def _model(noise=1e-4, mean_const=0.3, family="rbf"):
    return ogp.make_gp(3, 12, family=family, lengthscale=1.3, outputscale=0.7, noise=noise, mean_const=mean_const)


def test_describe_reference_kernel_objects():
    m = _model()
    cases = [
        (ogp.VanillaGP(m).predictive_kernel, _lib.PRED_COV),
        (ogp.WsabiGP(m, alpha=0.2).predictive_kernel, _lib.PRED_COV),
        (ogp.WsabiGP(m, alpha=0.2).wsabil_kernel, _lib.WSABI_L),
        (ogp.WsabiGP(m, alpha=0.2).wsabim_kernel, _lib.WSABI_M),
        (ogp.ScaleMmltGP(m).gspace_kernel, _lib.MMLT_G),
        (ogp.ScaleMmltGP(m).hspace_kernel, _lib.PRED_COV),
        (ogp.Kernel(m, "predictive_covariance"), _lib.PRED_COV),
        (ogp.Kernel(m, "weighted_predictive_covariance"), _lib.WSABI_L),
        (ogp.Kernel(m, "kernel"), _lib.PLAIN),
        (m.covar_module.forward, _lib.PLAIN),
        (m.covar_module, _lib.PLAIN),
    ]
    for k, mode in cases:
        spec = kernels.describe_kernel(k)
        assert spec.mode == mode and spec.family == _lib.RBF
        assert abs(spec.outputscale - 0.7) < 1e-12 and abs(float(spec.lengthscale[0]) - 1.3) < 1e-12
        if mode != _lib.PLAIN:
            assert abs(spec.noise - 1e-4) < 1e-15 and abs(spec.mean_const - 0.3) < 1e-12
            W, Xobs, _ = ogp.get_cov_cache(m)
            assert torch.allclose(spec.W, W) and spec.Xobs is Xobs
    assert kernels.describe_kernel(ogp.WsabiGP(m, alpha=0.2).wsabil_kernel).offset == 0.2
    quirk = kernels.describe_kernel(ogp.VanillaGP(m, add_noise_diag=True).predictive_kernel)
    assert quirk.noise_diag and quirk.diag_add == 0.0 and quirk.noise == pytest.approx(1e-4)
    assert not kernels.describe_kernel(ogp.VanillaGP(m).predictive_kernel).noise_diag
    # the noise enters the covariance before the warping, the jitter after it (BASQ/_wsabi.py:216-224)
    wm = kernels.describe_kernel(ogp.WsabiGP(m, jitter=1e-3, add_noise_diag=True).wsabim_kernel)
    assert wm.noise_diag and wm.diag_add == pytest.approx(1e-3)
    mat = _model(family="matern")
    assert kernels.describe_kernel(mat.covar_module.forward).family == _lib.MATERN25


def test_unknown_callable_is_rejected():
    with pytest.raises(TypeError, match="no generic"):
        kernels.describe_kernel(lambda x, y: x @ y.T)
    with pytest.raises(ValueError):
        kernels.describe_kernel(ogp.Kernel(_model(), "nonsense"))


def test_descriptor_fields():
    m = _model()
    spec = kernels.describe_kernel(ogp.VanillaGP(m).predictive_kernel)
    desc, keep = spec.to_desc(3, torch.device("cpu"), torch.float32)
    assert (desc.family, desc.mode, desc.dtype, desc.d, desc.n_obs) == (_lib.RBF, _lib.PRED_COV, _lib.F32, 3, 12)
    assert [desc.lengthscale[i] for i in range(3)] == [1.3, 1.3, 1.3]
    assert keep[0].dtype == torch.float32 and keep[1].dtype == torch.float64
    with pytest.raises(ValueError):
        spec.to_desc(4, torch.device("cpu"), torch.float32)
    with pytest.raises(TypeError):
        spec.to_desc(3, torch.device("cpu"), torch.float16)


def test_recombination_signatures(monkeypatch):
    seen = {}

    def fake(samp, pt, s, kernel, device, mu=None, use_obj=True, calc_obj=None):
        seen.update(dtype=samp.dtype, mu=mu, s=s, calc_obj=calc_obj)
        return torch.arange(2), torch.ones(2)

    monkeypatch.setattr(_rchq, "rc_kernel_svd", fake)
    X, Z = torch.randn(20, 2), torch.randn(5, 2)
    w0 = torch.rand(20)
    _rchq.recombination(X, Z, 4, "k", "cpu")                                   # BASQ, default init_weights=0
    assert seen["mu"] is None and seen["dtype"] == torch.float32
    _rchq.recombination(X, Z, 4, "k", "cpu", w0)                               # BASQ ignores weights (:53)
    assert seen["mu"] is None
    _rchq.recombination(X, Z, 4, "k", "cpu", init_weights=w0)
    assert seen["mu"] is None
    _rchq.recombination(X, Z, 4, "k", "cpu", torch.float64, w0)                # SOBER honours them
    assert seen["mu"] is w0 and seen["dtype"] == torch.float64
    _rchq.recombination(X, Z, 4, "k", "cpu", dtype=torch.float64, init_weights=None, calc_obj=None)
    assert seen["mu"] is None
    monkeypatch.setattr(_rchq, "HONOUR_INIT_WEIGHTS_IN_BASQ_SIGNATURE", True)
    _rchq.recombination(X, Z, 4, "k", "cpu", w0)
    assert seen["mu"] is w0
    with pytest.raises(ValueError):
        _rchq.recombination(X, Z, 4, "k", "cpu", torch.float64, torch.rand(7))
    f = lambda x: x[:, 0]
    _rchq.recombination(X, Z, 4, "k", "cpu", torch.float64, None, f)           # SOBER's calc_obj is forwarded
    assert seen["calc_obj"] is f
    _rchq.recombination(X, Z, 4, "k", "cpu")
    assert seen["calc_obj"] is None


def test_shard_bounds_and_survivor_counts():
    for N, W in [(10, 3), (7, 8), (1000, 4)]:
        spans = [sharded.shard_bounds(N, W, r) for r in range(W)]
        assert spans[0][0] == 0 and spans[-1][1] == N
        assert all(spans[i][1] == spans[i + 1][0] for i in range(W - 1))
    # kept_before equals a brute-force count
    S, R = 8, 53
    keep = torch.tensor([1, 0, 1, 1, 0, 0, 1, 0])
    prefix = torch.zeros(S + 1, dtype=torch.int64); prefix[1:] = torch.cumsum(keep, 0)
    K = int(prefix[S])
    brute = [sum(int(keep[g % S]) for g in range(p)) for p in range(R + 1)]
    assert [sharded.kept_before(p, S, prefix, K) for p in range(R + 1)] == brute


def test_level_tree_bookkeeping():
    """sharded.LevelTree (mirror of LevelTree in csrc/api.cu): node ids, parent columns and factors of
    a pass with F = 4 cells per set, checked against the definition - node u of level l = cells
    u + k S 2^l; children u (low) and u + S 2^l (high); a cell's factor = product along its path."""
    import numpy as np
    S, F, R = 6, 4, 1000
    tree = sharded.LevelTree(S, F, R)
    factor = torch.zeros(F * S, dtype=torch.float64)
    assert tree.columns() == S and list(tree.node) == list(range(S)) and tree.lvl == 0
    # level 0: keep sets 1, 3, 4 with factors 2, 3, 5
    om0 = np.array([0.0, 2.0, 0.0, 3.0, 5.0, 0.0])
    more, kept = tree.advance(om0, factor)
    assert more and kept == 3 and tree.lvl == 1
    assert list(tree.node) == [1, 3, 4] and list(tree.ppos) == [1, 3, 4] and list(tree.fpar) == [2.0, 3.0, 5.0]
    assert list(tree.act) == [1, 3, 4, 1 + S, 3 + S, 4 + S]              # low halves, then high halves
    # level 1: keep low(1), high(3), high(4)
    om1 = np.array([0.5, 0.0, 0.0, 0.0, 2.0, 1.0])
    more, kept = tree.advance(om1, factor)
    assert more and kept == 3 and tree.lvl == 2
    assert list(tree.node) == [1, 3 + S, 4 + S] and list(tree.ppos) == [0, 4, 5]
    assert list(tree.fpar) == [1.0, 6.0, 5.0]
    assert list(tree.act) == [1, 3 + S, 4 + S, 1 + 2 * S, 3 + 3 * S, 4 + 3 * S]
    # level 2 (cells): keep three of the six
    om2 = np.array([1.0, 0.0, 0.25, 0.0, 1.5, 0.0])
    more, kept = tree.advance(om2, factor)
    assert not more and kept == 3
    expect = torch.zeros(F * S, dtype=torch.float64)
    expect[1] = 1.0; expect[4 + S] = 1.25; expect[3 + 3 * S] = 9.0
    assert torch.equal(factor, expect)
    # fewer live points than sets: only min(S, R) columns at level 0
    assert sharded.LevelTree(S, 1, 4).columns() == 4


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours) prints one JSON line with
    the contract's keys on a CPU-only box; tiny sizes so that it takes seconds."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--cpu-sample", "2000", "--M", "200", "--n", "40", "--n-obs", "22"],
                         capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["value"] > 0 and line["cpu_baseline"]["kind"] == "port"
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and "workload" in line["config"]
    # same `config` keys as our arm (the driver compares them), the bounded sample is named beside the number
    assert set(line["config"]) == {"workload", "N_total", "parallelism", "l2_policy"}
    assert "N=2000" in line["cpu_baseline"]["sample"] and line["cpu_baseline"]["cores"] >= 1
    ex = line["extrapolation"]
    assert ex["N_full"] == 10_000_000 and ex["n_large"] == 2000 and ex["seconds_full"] > 0


def test_bench_reference_arm_uses_all_threads_under_torchrun_env():
    """torch.distributed.run exports OMP_NUM_THREADS=1; the CPU arm must still use every host core, and
    ranks other than 0 exit without work."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    args = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "20",
            "--warmup", "0", "--cpu-sample", "2000", "--M", "200", "--n", "40", "--n-obs", "22", "--cpu-budget", "5"]
    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="2", LOCAL_RANK="0")
    out = subprocess.run(args, capture_output=True, text=True, timeout=300, cwd=root, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    cores = len(os.sched_getaffinity(0))
    assert line["cpu_baseline"]["cores"] == cores and line["n_gpus"] == 2
    assert line["config"]["parallelism"] == "dp2" and 1 <= line["steps"] <= 20
    assert "N=2000" in line["cpu_baseline"]["sample"]          # the sample is never shrunk by --steps
    env["RANK"] = "1"
    out = subprocess.run(args, capture_output=True, text=True, timeout=300, cwd=root, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_bench_rejects_zero_steps():
    """--steps is the number of timed steps: zero would leave nothing to time."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "0"],
                         capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 2 and "--steps" in out.stderr
