"""The Philox + Box-Muller noise against fp64 on every uniform value it can draw (pytest -m gpu; -s prints the report).

Every normal libvbnn draws comes from one device function, philox_normal4 (csrc/philox.cuh).  tests/noise_reference.py
restates it on the device: Philox bit for bit, the transform in fp64 with a per-element bound derived from the
documented accuracy of __logf, rsqrt.approx and sin / cos.approx.  Each uniform sits on a grid of 2^24 values, so
2^29 consecutive counters (2^30 Box-Muller pairs) visit every grid value of u0 and of u1 about 64 times:
  (a) the whole domain, drawn by vbnn_philox_normal and compared element by element with the restatement;
  (b) counters whose u0 is among the 64 lowest or highest grid values (u0 near 1 is where the true log is smaller than
      __logf's error) or whose u1 sits at a quadrant boundary, each drawn alone: bit-identical to (a), within the bound;
  (c) the call sites that can be read back bit for bit: k_sample_w's epsilon in a weight-mode fp32 layer, and the
      normals of k_init_normal behind vbnn_mlp_init_params.  The epsilon / zeta regenerated in the GEMM epilogues
      (epilogue.cuh, epilogue_tc.cuh, gemm_tc.cu) is compared with draw_noise, element by element, in
      test_gpu_edge_values.py and test_gpu_multiwave.py, and draw_noise is the k_philox_matrix checked here;
  (d) quad counters past 2^32 - 1 wrap to 0 on the device and in the restatement alike."""
import ctypes as C

import numpy as np
import pytest
import torch

import noise_reference as NR

pytestmark = pytest.mark.gpu

SEED, STEP, STREAM, SAMPLE = 0x5EED0000000B, 7, NR.STREAM_ZETA | 3, 2
TOTAL, CHUNK = 1 << 29, 1 << 25          # counters of (a), drawn cols = 4 (one counter per row)
EDGE = 64                                # grid values at each end of u0 that (b) draws alone
MIN_COUNT = 16                           # of each grid value over (a); the expectation is 2^30 / 2^24 = 64
REGIONS = {"u0 > 1/2": lambda k: k >= NR.HALF, "u0 <= 1/2": lambda k: k < NR.HALF,
           f"top {EDGE} u0": lambda k: k >= NR.GRID - EDGE}


def draw(ctx, rows, cols, row0, seed=SEED, step=STEP, stream=STREAM, sample=SAMPLE):
    from vbnn_b200 import _lib as L
    out = torch.empty(rows, cols, device="cuda")
    L.check(L.lib().vbnn_philox_normal(ctx.handle, C.c_uint64(seed), step, stream, sample, rows, cols, row0,
                                       C.c_void_p(out.data_ptr())))
    return out


def check_bound(dev, ref):
    """finite, within the per-element bound, |n| <= R_MAX + bound, and the radius not negative: the sign of n agrees
    with cos / sin wherever those are larger than their error.  Returns the failing elements' mask."""
    d = dev.double()
    return (~torch.isfinite(dev) | ~((d - ref.n).abs() <= ref.bound) | ~(d.abs() <= NR.R_MAX + ref.bound)
            | ((ref.trig.abs() > ref.trig_err) & (d * ref.trig < 0)))


def near_quadrant(k):
    """u1 grid values at the quadrant boundaries 0, 1/4, 1/2, 3/4, 1: the two on each side of j 2^22"""
    return ((k + 2) % (1 << 22)) < 4


@pytest.fixture(scope="module")
def whole_domain(ctx):
    cnt = [torch.zeros(NR.GRID, dtype=torch.int64, device="cuda") for _ in range(2)]
    s = dict(nonfinite=0, over_bound=0, over_rmax=0, neg_radius=0, failures=[],
             err={r: 0.0 for r in REGIONS}, ratio={r: 0.0 for r in REGIONS}, hazard={})
    picks = {}
    for row0 in range(0, TOTAL, CHUNK):
        dev = draw(ctx, CHUNK, 4, row0)
        ref = NR.philox_normal4(torch.arange(row0, row0 + CHUNK, device="cuda"), SEED, STREAM, SAMPLE, STEP)
        k0, k1 = ref.k_u0[:, 0::2], ref.k_u1[:, 0::2]                 # [CHUNK x 2]: one per Box-Muller pair
        cnt[0] += torch.bincount(k0.reshape(-1), minlength=NR.GRID)
        cnt[1] += torch.bincount(k1.reshape(-1), minlength=NR.GRID)
        d = dev.double()
        err = (d - ref.n).abs()
        s["nonfinite"] += int((~torch.isfinite(dev)).sum())
        s["over_bound"] += int((~(err <= ref.bound)).sum())
        s["over_rmax"] += int((~(d.abs() <= NR.R_MAX + ref.bound)).sum())
        s["neg_radius"] += int(((ref.trig.abs() > ref.trig_err) & (d * ref.trig < 0)).sum())
        bad = check_bound(dev, ref)
        for i in torch.nonzero(bad)[:8 - len(s["failures"])].tolist():
            s["failures"].append(dict(idx4=row0 + i[0], j=i[1], k_u0=int(ref.k_u0[i[0], i[1]]),
                                      k_u1=int(ref.k_u1[i[0], i[1]]), dev=float(dev[i[0], i[1]]),
                                      ref=float(ref.n[i[0], i[1]]), bound=float(ref.bound[i[0], i[1]])))
        for name, sel in REGIONS.items():
            m = sel(ref.k_u0)
            s["err"][name] = max(s["err"][name], float(torch.where(m, err, 0.0).max()))
            s["ratio"][name] = max(s["ratio"][name], float(torch.where(m, err / ref.bound, 0.0).max()))
        # the device's radius where |ln u0| is below __logf's error: its projection on (cos, sin)
        for a in range(2):
            hz = torch.nonzero(NR.hazard_u0(k0[:, a])).flatten()
            r_dev = d[hz, 2 * a] * ref.trig[hz, 2 * a] + d[hz, 2 * a + 1] * ref.trig[hz, 2 * a + 1]
            for k, r in zip(k0[hz, a].tolist(), r_dev.tolist()):
                lo, hi, c = s["hazard"].get(k, (r, r, 0))
                s["hazard"][k] = (min(lo, r), max(hi, r), c + 1)
        # (b): the first counter of each grid value at the ends of u0 and at the quadrant boundaries of u1
        for kind, kk, mask in (("u0", k0, (k0 < EDGE) | (k0 >= NR.GRID - EDGE)), ("u1", k1, near_quadrant(k1))):
            rows = torch.nonzero(mask)[:, 0]
            for r, k in zip(rows.tolist(), kk[mask].tolist()):
                if (kind, k) not in picks:
                    picks[(kind, k)] = (row0 + r, dev[r].clone())
        del dev, ref, d, err, bad, k0, k1
    s["coverage"] = [int(c.min()) for c in cnt]
    print(f"\nnoise over {TOTAL} counters ({2 * TOTAL} Box-Muller pairs): fewest draws of one grid value "
          f"u0 {s['coverage'][0]}, u1 {s['coverage'][1]} (expected 64)")
    for name in REGIONS:
        print(f"  {name:>12}: max |n_dev - n_fp64| {s['err'][name]:.3e}, max error / bound {s['ratio'][name]:.3f}")
    print(f"  non-finite {s['nonfinite']}, beyond the bound {s['over_bound']}, |n| > R_MAX + bound {s['over_rmax']}, "
          f"negative radius {s['neg_radius']}")
    ref_r = NR.box_muller(torch.tensor(sorted(s["hazard"])), torch.zeros(len(s["hazard"]), dtype=torch.int64))
    for (k, (lo, hi, c)), r in zip(sorted(s["hazard"].items()), ref_r.n_cos.tolist()):
        print(f"  u0 = {float(NR.unit_f32(torch.tensor(k))):.9f} (k = 2^24 - {NR.GRID - k}): fp64 radius {r:.3e}, "
              f"device radius in [{lo:.3e}, {hi:.3e}] over {c} pairs")
    return s, picks


def test_whole_domain_within_fp64_bound(whole_domain):
    s, _ = whole_domain
    assert min(s["coverage"]) >= MIN_COUNT, s["coverage"]
    assert len(s["hazard"]) == 7, sorted(s["hazard"])
    assert (s["nonfinite"], s["over_bound"], s["over_rmax"], s["neg_radius"]) == (0, 0, 0, 0), s["failures"]


def test_targeted_counters_drawn_alone(ctx, whole_domain):
    _, picks = whole_domain
    assert sum(kind == "u0" for kind, _ in picks) == 2 * EDGE
    assert sum(kind == "u1" for kind, _ in picks) == 2 + 4 * 3 + 2
    keys = sorted(picks)
    idx4 = torch.tensor([picks[k][0] for k in keys], device="cuda")
    alone = torch.cat([draw(ctx, 1, 4, int(i)) for i in idx4.tolist()])
    seen = torch.stack([picks[k][1] for k in keys])
    assert torch.equal(alone.view(torch.int32), seen.view(torch.int32))
    ref = NR.philox_normal4(idx4, SEED, STREAM, SAMPLE, STEP)
    for i, (kind, k) in enumerate(keys):
        assert k in (ref.k_u0 if kind == "u0" else ref.k_u1)[i].tolist()
    bad = check_bound(alone, ref)
    assert not bad.any(), [keys[i] for i in torch.nonzero(bad)[:, 0].tolist()]


def hazards_in(ctr, seed, stream, sample, step):
    """the counters put u0 = 1.0 and another u0 within __logf's error of 1 into at least one pair each"""
    k = NR.grid_indices(ctr, seed, stream, sample, step)[:, 0::2]
    return bool((k == NR.GRID - 1).any()) and bool((NR.hazard_u0(k) & (k != NR.GRID - 1)).any())


def vb_net(ctx, I, O):
    import vbnn_b200
    opt = vbnn_b200.default_opt(input_size=I, hidden=[O], classes=[str(i) for i in range(10)], S=1, B=10.0,
                                reparam="weight", precision="fp32", strict_reference=True, batchSize=8, log=False)
    return vbnn_b200.MLP(opt, ctx, max_batch=8)


def test_weight_sample_eps_is_the_noise(ctx):
    """k_sample_w's epsilon in a weight-mode fp32 layer.  The layer keeps epsilon (VBLinear.e, BUF_EPS: k_sample_w's
    eps_out) only when the caller injects it, so no option makes it keep the epsilon it draws.  With mu = 0 and the
    strict-reference sigma cache at 1 the sampled weight is fmaf(1, eps, 0) = eps exactly, which reads it back."""
    from vbnn_b200 import _lib as L
    I = O = 2048                                        # 2^20 counters: about 0.9 hazardous u0 values per step
    net = vb_net(ctx, I, O)
    lyr = net.model[0]                                  # layer 0 of an mlp: Philox stream kStreamEps | 0
    ctr = NR.matrix_counters(O, I, device="cuda")
    step = next(s for s in range(1000, 1500) if hazards_in(ctr, ctx.seed, NR.STREAM_EPS, 0, s))
    lyr.set(L.BUF_MEANS, torch.zeros(O, I))
    lyr.set(L.BUF_STDV, torch.ones(O, I))
    step0 = ctx.get_step()
    try:
        ctx.set_step(step)
        net.sample(sample_idx=0)
        w = lyr.weight.cuda()
    finally:
        ctx.set_step(step0)
    assert torch.equal(w, lyr.draw_noise(step, 0))
    ref = NR.philox_normal4(ctr, ctx.seed, NR.STREAM_EPS, 0, step)
    bad = check_bound(w.reshape(-1, 4), ref)
    assert NR.hazard_u0(ref.k_u0).any() and not bad.any(), int(bad.sum())


def test_init_params_normals(ctx):
    """k_init_normal behind vbnn_mlp_init_params: means = fl(std * n) with std = sqrtf(2 / I) (he_means), stream
    kStreamInit | layer, sample 1, step 0, key = the seed argument."""
    I = O = 2048
    net = vb_net(ctx, I, O)
    ctr = NR.matrix_counters(O, I, device="cuda")
    seed = next(s for s in range(1, 500) if hazards_in(ctr, s, NR.STREAM_INIT, 1, 0))
    net.init_params(seed=seed, he_means=True)
    means = net.model[0].means.clone()
    std = float(np.sqrt(np.float32(2.0) / np.float32(I)))
    assert torch.equal(means, draw(ctx, O, I, 0, seed=seed, step=0, stream=NR.STREAM_INIT, sample=1) * std)
    ref = NR.philox_normal4(ctr, seed, NR.STREAM_INIT, 1, 0)
    m = means.reshape(-1, 4).double()
    tol = std * ref.bound + NR.U32 * std * (ref.n.abs() + ref.bound)
    assert NR.hazard_u0(ref.k_u0).any()
    assert torch.isfinite(m).all() and ((m - std * ref.n).abs() <= tol).all()


def test_counters_wrap_at_2_32(ctx):
    """row0 = 2^30 - 1 with cols = 16: quad counters 2^32 - 4 .. 2^32 - 1, then 0 .. 3 (include/vbnn.h)"""
    rows, cols, row0 = 2, 16, (1 << 30) - 1
    dev = draw(ctx, rows, cols, row0)
    assert torch.equal(dev[1].view(torch.int32), draw(ctx, 1, cols, 0)[0].view(torch.int32))
    ctr = NR.matrix_counters(rows, cols, row0, device="cuda")
    assert ctr.tolist() == [(1 << 32) - 4 + c for c in range(4)] + [0, 1, 2, 3]
    ref = NR.philox_normal4(ctr, SEED, STREAM, SAMPLE, STEP)
    assert not check_bound(dev.reshape(-1, 4), ref).any()
