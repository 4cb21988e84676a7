"""bench.py --dump-outputs on the GPU: the arrays the last timed minibatch left the caller are written as float32
.npy files, the same arguments give the same arrays, and --steps reaches every timed loop (one more minibatch moves
the parameters; the C1 / C2 extra workloads time --steps minibatches too)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bench_dump(out, steps, *extra):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                        "--warmup", "3", "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(out)] + list(extra),
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["steps"] == steps
    arrays = {f[:-4]: np.load(os.path.join(out, f)) for f in sorted(os.listdir(out))}
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in arrays.values())
    assert sum(os.path.getsize(os.path.join(out, f"{k}.npy")) for k in arrays) <= 64 << 20
    return line, arrays


@pytest.mark.gpu
def test_dump_outputs_is_reproducible_and_follows_steps(tmp_path):
    c1 = ("--workload", "c1", "--no-extra")
    _, a = bench_dump(tmp_path / "a", 4, *c1)
    _, b = bench_dump(tmp_path / "b", 4, *c1)
    _, c = bench_dump(tmp_path / "c", 5, *c1)
    # C1: 784-100-10, batch 100, one weight sample, nn.Linear output layer
    shapes = dict(result=(2,), logp=(1, 100, 10), layer0_means=(100, 784), layer0_lvars=(100, 784), layer0_bias=(100,),
                  layer1_weight=(10, 100), layer1_bias=(10,))
    assert {k: v.shape for k, v in a.items()} == shapes
    for k in shapes:
        assert np.allclose(a[k], b[k], rtol=1e-5, atol=1e-6), k
    assert not np.allclose(a["layer0_means"], c["layer0_means"], rtol=1e-5, atol=1e-6)


@pytest.mark.gpu
def test_c3_dump_is_sampled_and_extra_workloads_follow_steps(tmp_path):
    """The default workload (C3, 4096-4096x4-1000, batch 8192) with its C1 / C2 extra workloads: the extras time
    --steps minibatches after their own 20 warm-up minibatches, and every array above 2^18 elements is sampled."""
    line, a = bench_dump(tmp_path / "c3", 3)
    assert {k: (v["steps"], v["warmup"]) for k, v in line["extra_workloads"].items()} == {"c1": (3, 20), "c2": (3, 20)}
    big = [f"layer{k}_{n}" for k in range(4) for n in ("means", "lvars")] + ["layer4_weight", "logp"]
    small = {f"layer{k}_bias": (4096,) for k in range(4)}
    small.update(layer4_bias=(1000,), result=(2,))
    assert {k: v.shape for k, v in a.items()} == dict(small, **{k: (1 << 18,) for k in big})
