"""CPU tests of tests/noise_reference.py, the torch restatement of the Philox + Box-Muller noise (-m "not gpu").

They pin the restatement to Random123's known-answer vectors and to the numpy oracle bit for bit, its fp64 transform
to the oracle's fp32 one within the oracle's rounding, and check that the per-element bound is tight enough to flag a
planted error at the top of the grid and a sign flip of the radius, while accepting the oracle."""
import math

import numpy as np
import torch

import noise_reference as NR
from oracle import vbnn_oracle as O

KATS = [   # Random123 kat_vectors, philox4x32 10 rounds (as in test_oracle.py)
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
]


def test_philox_known_answer_vectors():
    for ctr, key, out in KATS:
        got = NR.philox4x32_10([torch.tensor([w]) for w in ctr], key)
        assert tuple(int(w[0]) for w in got) == out


def test_philox_matches_oracle_bit_for_bit():
    rng = np.random.RandomState(7)
    n = 1 << 14
    ctr = rng.randint(0, 1 << 32, size=(n, 4), dtype=np.uint64).astype(np.uint32)
    ctr[:64] = 0                                     # counter words at both ends of the range, in every position
    ctr[64:128] = 0xFFFFFFFF
    ctr[128:256] = np.where(rng.rand(128, 4) < 0.5, 0, 0xFFFFFFFF)
    for key in [(0, 0), (0xFFFFFFFF, 0xFFFFFFFF), (0, 0xFFFFFFFF), (0x12345678, 0x9ABCDEF0)]:
        want = O.philox4x32_10(ctr, np.array(key, dtype=np.uint32))
        got = NR.philox4x32_10([torch.from_numpy(ctr[:, j].astype(np.int64)) for j in range(4)], key)
        got = np.stack([g.numpy() for g in got], axis=1)
        assert got.min() >= 0 and got.max() <= 0xFFFFFFFF
        assert np.array_equal(got, want.astype(np.int64)), key


def test_counters_wrap_like_the_device():
    """matrix_counters takes the quad index mod 2^32, as the device's uint32 arithmetic does"""
    ctr = NR.matrix_counters(rows=2, cols=16, row0=(1 << 30) - 1)
    assert ctr.tolist() == [0xFFFFFFFC, 0xFFFFFFFD, 0xFFFFFFFE, 0xFFFFFFFF, 0, 1, 2, 3]
    a = NR.philox_normal4(ctr, 5, 1, 2, 3)
    b = NR.philox_normal4(torch.arange(4) + (1 << 32), 5, 1, 2, 3)    # 2^32 + c is counter c
    assert torch.equal(a.n[4:], b.n)


def test_uniform_grid():
    k = torch.tensor([0, 1, NR.HALF - 2, NR.HALF - 1, NR.HALF, NR.GRID - 3, NR.GRID - 2, NR.GRID - 1])
    u = NR.unit_f32(k)
    assert u.dtype == torch.float32
    # oracle: (float(k) + 0.5f) * 2^-24 in fp32, two exact-or-same roundings of the same number
    ref = (k.numpy().astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -24)
    assert np.array_equal(u.numpy(), ref)
    assert u[-1] == 1.0 and u[0] == 2.0 ** -25
    assert u[-2] == u[-3] == 1.0 - 2.0 ** -23      # halfway cases round to even: pairs of k share a value above 1/2
    assert u[2] == 0.5 - 2.0 ** -25 and u[3] == 0.5 and u[4] == 0.5 + 2.0 ** -23
    hz = NR.hazard_u0(torch.arange(NR.GRID - 64, NR.GRID))
    assert hz.sum() == 7 and hz[-7:].all()         # u0 = 1.0 and the three fp32 values below it


def test_fp64_transform_matches_oracle():
    """The oracle rounds log, sqrt, the angle and cos / sin to fp32: its error is r |fl(fl(2pi) u1) - 2pi u1| from the
    angle plus a few fp32 roundings of r and n."""
    seed, step, stream, sample, rows, cols = 5, 3, (1 << 16) | 2, 1, 256, 1024
    want = O.philox_normal_matrix(seed, step, stream, sample, rows, cols)
    ref = NR.philox_normal4(NR.matrix_counters(rows, cols), seed, stream, sample, step)
    n = NR.as_matrix(ref.n, rows, cols).numpy()
    r = np.hypot(n, NR.as_matrix(ref.n[:, [1, 0, 3, 2]], rows, cols).numpy())
    u1 = NR.unit_f32(NR.as_matrix(ref.k_u1, rows, cols)).double().numpy()
    d_arg = np.abs(np.float32(NR.TWO_PI_F32) * u1.astype(np.float32) - 2 * math.pi * u1)
    tol = r * d_arg + 8 * NR.U32 * r + NR.FLT_MIN
    err = np.abs(want - n)
    assert (err <= tol).all(), float((err / tol).max())
    assert (err <= NR.as_matrix(ref.bound, rows, cols).numpy()).all()     # the bound accepts the oracle too


def test_bound_stays_small_over_the_grid():
    """Away from u0 = 1 the bound is at the level of the intrinsics' own errors; it never exceeds 2^-10"""
    k = torch.arange(NR.GRID)
    for k1 in (0, NR.GRID // 4, NR.GRID // 2 - 1, 12345, NR.GRID - 2, NR.GRID - 1):
        p = NR.box_muller(k, torch.full_like(k, k1))
        b = torch.maximum(p.bound_cos, p.bound_sin)
        assert float(b.max()) < 2.0 ** -10, k1
        if k1 < NR.GRID - 1:
            assert float(b[:NR.HALF].max()) < 2.0 ** -16, k1
        assert float(p.n_cos.abs().max()) <= NR.R_MAX


def test_bound_flags_planted_errors():
    ctr = torch.arange(1 << 16)
    ref = NR.philox_normal4(ctr, 9, 0, 0, 0)
    n32 = ref.n.float()                               # the fp64 value rounded to fp32: a faithful device
    assert ((n32.double() - ref.n).abs() <= ref.bound).all()
    # 2^-9 on the top-of-grid u0 values, one element of each pair with u0 = 1.0 and u0 = 1 - 2^-23
    for kk in (NR.GRID - 1, NR.GRID - 2):
        p = NR.box_muller(torch.tensor([kk] * 4), torch.tensor([0, NR.GRID // 8, NR.GRID // 4, NR.GRID - 1]))
        for n, b in ((p.n_cos, p.bound_cos), (p.n_sin, p.bound_sin)):
            for planted in (n + 2.0 ** -9, n - 2.0 ** -9):
                assert ((planted - n).abs() > b).all(), kk
    # sign flip of the radius: flagged wherever |n| exceeds half the bound, which is almost everywhere
    bad = (-n32.double() - ref.n).abs() > ref.bound
    big = ref.n.abs() > ref.bound / 2
    assert bad[big].all() and big.float().mean() > 0.999
    # and the trigonometric factor decides the sign where it is larger than its error
    sure = ref.trig.abs() > ref.trig_err
    assert ((n32.double() * ref.trig)[sure] >= 0).all()
    assert ((-n32.double() * ref.trig)[sure & (ref.n != 0)] < 0).all()
