"""bench.py's reference arm runs without a GPU (it times the oracle port on the host cores): check the
JSON contract of its line on the small C1 workload."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c1",
                        "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "VB-MLP train samples/sec" and d["unit"] == "samples/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 2 and d["warmup"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 8 and d["cpu_baseline"]["sample"]   # config.lua:5
    # C1 fits: the full minibatch is timed, nothing is extrapolated, and ms_per_step is time really spent
    assert d["estimated"] is False and d["cpu_baseline"]["rows_timed"] == 100
    assert abs(d["ms_per_step"] - 1e3 * 100 / d["value"]) < 0.5 * d["ms_per_step"]
    assert d["config"]["global_batch"] == 100 and d["config"]["sizes"] == [784, 100, 10]
    assert d["e2e"] == dict(value=d["value"], unit="samples/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0)


def test_dump_outputs_is_refused_before_any_work(tmp_path):
    """Only the single-GPU vbnn arm dumps, and never into a directory that already holds arrays (they would pass
    for this run's)."""
    stale = tmp_path / "stale"
    stale.mkdir()
    (stale / "layer4_weight.npy").write_bytes(b"")
    for out, extra, msg in ((tmp_path / "a", ["--impl", "reference"], "needs --impl vbnn on one GPU"),
                            (tmp_path / "b", ["--gpus", "2"], "needs --impl vbnn on one GPU"),
                            (stale, [], "already holds .npy files")):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", str(out)] + extra,
                           capture_output=True, text=True, timeout=60, cwd=ROOT)
        assert r.returncode == 2 and msg in r.stderr, (extra, r.stderr[-500:])
    assert sorted(os.listdir(tmp_path)) == ["stale"] and os.listdir(stale) == ["layer4_weight.npy"]


def test_dump_outputs_samples_large_arrays_at_fixed_indices(tmp_path):
    """dump_outputs on a stand-in for vbnn_b200.MLP (CPU tensors behind the same attributes): arrays up to
    DUMP_MAX_ELEMS keep their shape, larger ones become the elements at the same seeded indices in every run."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    from vbnn_b200 import _lib as VL

    class Layer:
        def __init__(self, kind, O, I):
            g = torch.Generator().manual_seed(O * 7 + I)
            self.kind, self.bias = kind, torch.randn(O, generator=g)
            if kind == VL.KIND_VB:
                self.means, self.lvars = torch.randn(O, I, generator=g), torch.randn(O, I, generator=g)
            else:
                self.weight = torch.randn(O, I, generator=g)

    class Net:
        opt = dict(S=2)
        _res = torch.tensor([2.5, 40.0])
        model = [Layer(VL.KIND_VB, 600, 500), Layer(VL.KIND_LINEAR, 10, 600)]

        def outputs(self, s):
            return torch.full((100, 10), -float(s + 1))

    net = Net()
    for d in ("a", "b"):
        bench.dump_outputs(net, str(tmp_path / d))
    names = ["layer0_bias", "layer0_lvars", "layer0_means", "layer1_bias", "layer1_weight", "logp", "result"]
    assert sorted(f[:-4] for f in os.listdir(tmp_path / "a")) == names
    a = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in names}
    assert all(v.dtype == np.float32 and np.array_equal(v, np.load(tmp_path / "b" / f"{n}.npy")) for n, v in a.items())
    assert a["logp"].shape == (2, 100, 10) and (a["logp"][1] == -2).all() and a["layer1_weight"].shape == (10, 600)
    n = 600 * 500
    assert n > bench.DUMP_MAX_ELEMS and a["layer0_means"].shape == (bench.DUMP_MAX_ELEMS,)
    idx = np.sort(np.random.default_rng(0).choice(n, bench.DUMP_MAX_ELEMS, replace=False))
    assert np.array_equal(a["layer0_means"], net.model[0].means.reshape(-1).numpy()[idx])
    assert np.array_equal(a["layer0_lvars"], net.model[0].lvars.reshape(-1).numpy()[idx])


def test_flops_per_sample_matches_survey():
    sys.path.insert(0, ROOT)
    import bench
    assert bench.flops_per_sample(bench.WORKLOADS["c1"]) == 319600                 # SURVEY.md 8(d)
    assert bench.flops_per_sample(bench.WORKLOADS["c2"]) == 124752000
    assert bench.flops_per_sample(bench.WORKLOADS["c3"]) == 762773504               # plain nn.Linear output layer


def test_both_arms_describe_the_same_config():
    sys.path.insert(0, ROOT)
    import bench
    for name in ("c1", "c2", "c3"):
        w = bench.WORKLOADS[name]
        a = bench.config_dict(w, 1, w["N"], "weak")
        assert a["workload"] == w["desc"] and a["global_batch"] == w["N"] and a["flops_per_sample"] == bench.flops_per_sample(w)
    c = bench.config_dict(bench.WORKLOADS["c3"], 8, 1024, "strong")
    assert c["global_batch"] == 8192 and c["per_gpu_batch"] == 1024 and c["parallelism"] == "dp8" and c["scaling"] == "strong"
