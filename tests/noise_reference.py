"""Device-side restatement of libvbnn's Gaussian noise (csrc/philox.cuh: philox_normal4), with a per-element bound.

Philox4x32-10 runs on int64 torch tensors (CUDA or CPU) holding uint32 words.  Each 32 x 32 -> 64 product is built
from 16-bit limbs, so every intermediate stays below 2^50 and nothing relies on int64 overflow.  The counter layout is
philox.cuh's and oracle.philox_normal_matrix's: (idx4, stream, sample, step), key = (seed_lo, seed_hi).

The uniforms are u = ((x >> 8) + 0.5) 2^-24 rounded once to fp32, as u32_to_unit forms them: the grid index
k = x >> 8 takes 2^24 values, and the top one, k = 2^24 - 1, rounds to exactly 1.0.  The Box-Muller transform of
those fp32 values is evaluated in fp64.

The device computes t = -2 __logf(u0), r = t * rsqrt.approx.ftz(max(t, 1e-30)), (s, c) = __sincosf(fl(2pi_f u1)),
n = (r c, r s).  The bound on |n_device - n_fp64| comes from the documented accuracy of each step, not from
measured errors:
  * __logf: absolute error 2^-21.41 for u0 in [0.5, 2], otherwise 3 ulp (CUDA C++ Programming Guide, "Intrinsic
    Functions", single precision).  Near u0 = 1 the true log is smaller than that absolute error, so the spec allows
    t of either sign there; the bound is that of the intended r = sqrt(max(t, 0)), so a device that turns a negative t
    into a large or negative radius fails it.
  * -2 * l is exact in fp32.
  * rsqrt.approx.f32: relative error 2^-22.9 over the entire range (PTX ISA, rsqrt); the product t * rsqrt adds one
    fp32 rounding.  Where max(t, 1e-30) clamps, r = t 1e15 lies between 0 and sqrt(t): inside the same interval.
  * sin.approx.f32 / cos.approx.f32 (what __sincosf issues): absolute error 2^-20.5 on [-2pi, 2pi] and 2^-14.7 on
    [-100pi, 100pi] (PTX ISA, sin / cos).  The device's argument fl(fl(2pi) u1) is known exactly, so the bound adds
    |fl(fl(2pi) u1) - 2pi u1| (|d cos|, |d sin| <= |d arg|) to the intrinsic's figure.  Arguments run from 2^-25 2pi
    up to fl(2pi) = 6.28318548..., which exceeds 2pi: only that one point (u1 = 1.0) needs the [-100pi, 100pi] figure.
  * n = r * c: one more fp32 rounding, plus FLT_MIN for a product flushed to zero.
Every range the transform uses is covered by one of these documented figures, so no engineering budget is needed.
The resulting bound is below 2^-16 for u0 <= 1/2 (except at u1 = 1.0), grows as u0 -> 1 (where __logf's absolute
error is all of t) and stays below 2^-10 everywhere (test_noise_reference_cpu.py).
The fp64 evaluation error of the reference itself (~1e-15 relative) is far below every term and is not counted.
|n| <= sqrt(-2 ln 2^-25) = 5.887 by construction of the grid (the smallest u0 is 2^-25), up to the bound."""
import math
from typing import NamedTuple

import numpy as np
import torch

MASK32 = 0xFFFFFFFF
_M0, _M1 = 0xD2511F53, 0xCD9E8D57          # Philox4x32 multipliers
_W0, _W1 = 0x9E3779B9, 0xBB67AE85          # Weyl key increments
GRID = 1 << 24                              # uniform grid values per 32-bit word
HALF = (1 << 23) + 1                        # k >= HALF <=> u > 1/2 (k = 2^23 rounds to exactly 1/2)

STREAM_EPS, STREAM_ZETA, STREAM_INIT = 0 << 16, 1 << 16, 2 << 16   # philox.cuh kStream*

U32 = 2.0 ** -24                            # fp32 unit roundoff
FLT_MIN = 2.0 ** -126
LOGF_ABS = 2.0 ** -21.41                    # __logf, u0 in [0.5, 2]: absolute error
LOGF_ULP = 3.0                              # __logf elsewhere: ulp error
RSQ_REL = 2.0 ** -22.9                      # rsqrt.approx.f32: relative error
TRIG_ABS_2PI = 2.0 ** -20.5                 # sin/cos.approx.f32 on [-2pi, 2pi]: absolute error
TRIG_ABS_100PI = 2.0 ** -14.7               # sin/cos.approx.f32 on [-100pi, 100pi]: absolute error
TWO_PI_F32 = float(np.float32(2.0 * math.pi))   # the device's 6.283185307179586f
R_MAX = math.sqrt(-2.0 * math.log(2.0 ** -25))  # 5.887: largest radius the grid can produce


def _mulhilo(a: int, b: torch.Tensor):
    """(hi, lo) 32-bit words of the exact product of the constant a < 2^32 and uint32 words b (int64 tensor)."""
    p_lo = a * (b & 0xFFFF)                     # < 2^48
    p_hi = a * (b >> 16)                        # < 2^48; the product is p_hi 2^16 + p_lo
    s = p_lo + ((p_hi & 0xFFFF) << 16)          # < 2^49
    return (p_hi >> 16) + (s >> 32), s & MASK32


def philox4x32_10(ctr, key):
    """ctr: 4 uint32 words as int64 tensors or ints (broadcast against each other); key: (k0, k1) ints.
    Returns the 4 output words as int64 tensors."""
    dev = next((c.device for c in ctr if torch.is_tensor(c)), torch.device("cpu"))
    c = [torch.as_tensor(w, dtype=torch.int64, device=dev) & MASK32 for w in ctr]
    c = list(torch.broadcast_tensors(*c))
    k0, k1 = int(key[0]) & MASK32, int(key[1]) & MASK32
    for _ in range(10):
        hi0, lo0 = _mulhilo(_M0, c[0])
        hi1, lo1 = _mulhilo(_M1, c[2])
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0 = (k0 + _W0) & MASK32
        k1 = (k1 + _W1) & MASK32
    return c


def unit_f32(k: torch.Tensor) -> torch.Tensor:
    """u32_to_unit of grid index k = x >> 8: (k + 0.5) 2^-24 rounded once to fp32 (exact in fp64 before the cast)."""
    return ((k.to(torch.float64) + 0.5) * 2.0 ** -24).to(torch.float32)


def _logf_err(u: torch.Tensor, lg: torch.Tensor) -> torch.Tensor:
    """documented |__logf(u) - ln u| for fp32 u (as fp64) with fp64 ln u = lg"""
    _, e = torch.frexp(lg)                      # |lg| = m 2^e, m in [0.5, 1): ulp = 2^(e - 24)
    ulp = torch.ldexp(torch.ones_like(lg), e - 24)
    return torch.where((u >= 0.5) & (u <= 2.0), torch.full_like(lg, LOGF_ABS), LOGF_ULP * ulp)


class Pair(NamedTuple):
    """The fp64 Box-Muller of one (u0, u1) pair: n_cos = r cos, n_sin = r sin, each with its bound, and the
    trigonometric factor with its own error (for the sign of the radius)."""
    n_cos: torch.Tensor
    n_sin: torch.Tensor
    bound_cos: torch.Tensor
    bound_sin: torch.Tensor
    cos: torch.Tensor
    sin: torch.Tensor
    trig_err: torch.Tensor


def box_muller(k0: torch.Tensor, k1: torch.Tensor) -> Pair:
    """fp64 Box-Muller of the fp32 uniforms of grid indices k0 (radius) and k1 (angle), with the bounds derived in the
    module docstring."""
    u0 = unit_f32(k0).to(torch.float64)
    u1 = unit_f32(k1).to(torch.float64)
    lg = torch.log(u0)
    t = -2.0 * lg
    dt = 2.0 * _logf_err(u0, lg)
    r = torch.sqrt(t)
    e_r = RSQ_REL + U32 + RSQ_REL * U32
    r_hi = torch.sqrt(t + dt) * (1.0 + e_r)
    r_lo = torch.sqrt(torch.clamp(t - dt, min=0.0)) * (1.0 - e_r)
    dr = torch.maximum(r_hi - r, r - r_lo)

    arg = 2.0 * math.pi * u1
    arg_dev = (TWO_PI_F32 * u1).to(torch.float32).to(torch.float64)   # 24 x 24-bit product: exact before the cast
    trig_err = torch.where(arg_dev <= 2.0 * math.pi, torch.full_like(arg, TRIG_ABS_2PI),
                           torch.full_like(arg, TRIG_ABS_100PI)) + (arg_dev - arg).abs()
    co, si = torch.cos(arg), torch.sin(arg)

    def bound(f):
        mag = f.abs() + trig_err
        return dr * mag + r * trig_err + U32 * (r + dr) * mag + FLT_MIN

    return Pair(r * co, r * si, bound(co), bound(si), co, si, trig_err)


class Normals(NamedTuple):
    """philox_normal4 restated for a vector of counters; every field is [n x 4], column j the normal 4q + j:
    k_u0 / k_u1 are the grid indices of the element's pair (x0, x1) for j = 0, 1 and (x2, x3) for j = 2, 3."""
    k_u0: torch.Tensor
    k_u1: torch.Tensor
    n: torch.Tensor
    bound: torch.Tensor
    trig: torch.Tensor
    trig_err: torch.Tensor


def words(idx4, seed: int, stream: int, sample: int, step: int):
    """Philox output words of quad counters idx4 (int64 tensor; taken mod 2^32 as the device's uint32 counter)."""
    return philox4x32_10((idx4, stream, sample, step), (seed & MASK32, (seed >> 32) & MASK32))


def grid_indices(idx4, seed: int, stream: int, sample: int, step: int) -> torch.Tensor:
    """[n x 4] grid indices x >> 8 of the four words of each counter: columns 0 and 2 are the radii's u0."""
    return torch.stack([w >> 8 for w in words(idx4, seed, stream, sample, step)], dim=1)


def philox_normal4(idx4, seed: int, stream: int, sample: int, step: int) -> Normals:
    k = grid_indices(idx4, seed, stream, sample, step)
    a, b = box_muller(k[:, 0], k[:, 1]), box_muller(k[:, 2], k[:, 3])
    st = lambda *c: torch.stack(c, dim=1)
    return Normals(k_u0=st(k[:, 0], k[:, 0], k[:, 2], k[:, 2]), k_u1=st(k[:, 1], k[:, 1], k[:, 3], k[:, 3]),
                   n=st(a.n_cos, a.n_sin, b.n_cos, b.n_sin), bound=st(a.bound_cos, a.bound_sin, b.bound_cos, b.bound_sin),
                   trig=st(a.cos, a.sin, b.cos, b.sin), trig_err=st(a.trig_err, a.trig_err, b.trig_err, b.trig_err))


def matrix_counters(rows: int, cols: int, row0: int = 0, device="cpu") -> torch.Tensor:
    """[rows * ceil(cols/4)] quad counters of a rows x cols matrix drawn by k_philox_matrix / draw_noise, mod 2^32"""
    q = (cols + 3) // 4
    r = torch.arange(row0, row0 + rows, dtype=torch.int64, device=device)[:, None]
    return ((r * q + torch.arange(q, dtype=torch.int64, device=device)[None, :]).reshape(-1)) & MASK32


def as_matrix(t: torch.Tensor, rows: int, cols: int) -> torch.Tensor:
    """[rows * q x 4] per-counter values -> the rows x cols matrix they fill"""
    return t.reshape(rows, -1)[:, :cols]


def hazard_u0(k: torch.Tensor) -> torch.Tensor:
    """u0 grid values where |ln u0| is within __logf's documented absolute error, so t = -2 __logf(u0) may be <= 0:
    u0 = 1.0 and the three fp32 values below it (k >= 2^24 - 7)."""
    u = unit_f32(k).to(torch.float64)
    return -torch.log(u) <= LOGF_ABS
