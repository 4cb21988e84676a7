"""fp64 reference with the device's conventions at degenerate values, and per-element error bounds.

Values come from the CPU oracle's layer methods (oracle/vbnn_oracle.py), as in tests/custom_loss_reference.py, with two
conventions of libvbnn that the oracle does not follow:
  * local reparameterisation: R := 0 where V = X^2 s2^T == 0 (an all-zero input row; include/vbnn.h next to
    VBNN_REPARAM_LOCAL).  The oracle divides by 2 sqrt(0) and gets +-inf, and NaN downstream.
  * ClassNLL targets outside 1..C add 0 to the loss, no -1 to the gradient and never count as correct, and the
    predicted class is the lowest index among tied maxima (include/vbnn.h next to vbnn_mlp_step).

Every value is paired with a bound E on |device - reference|, element by element, derived from how the device
computes it rather than fitted to what it returns:
  * one fp32-accumulated contraction of m non-zero products (adding an exact zero is exact, so a row of zeros has
    no rounding at all): C_ACC * m * 2^-24 * (|A| |B|) + m * 2^-150.  C_ACC = 2 allows every addition a full ulp,
    which covers truncating tensor-core adders as well as round-to-nearest FMA chains; 2^-150 is the absolute
    rounding error in fp32's subnormal range.  Errors already on the operands (E_A, E_B) pass through as
    E_A |B| + |A| E_B + E_A E_B.
  * storing a value in a narrower type: exact where the input is exact (both sides round the same number), else
    E + unit * (2 |v| + E), since the two sides may then round to neighbouring values (unit 2^-24 fp32, 2^-8 bf16).
  * __expf: (2 + floor(1.173 |x|)) ulps (CUDA C Programming Guide, intrinsic functions); results below FLT_MIN
    are flushed to zero, an absolute error of the result itself.
  * MUFU rsqrt: 2^-21 relative.
  * the bias gradient (fp32 atomics over N rows) is a contraction of G with a ones vector: C_ACC * N * 2^-24 * sum|G|.
  * exact operands: where every term of a contraction or fp32 sum is an integer known without error and the sum of
    the terms' magnitudes is below 2^24, every partial sum is an integer fp32 holds exactly, in any order, tile
    shape, K-split or atomic order: the bound is 0 (exactness rule, `exact_sum`).  Rounding such a value to bf16
    rounds the same number on both sides.  So ternary inputs and dL/dY, integer means and biases and log-variances
    whose __expf flushes to 0 (sigma = 0) make logits, dX and every gradWeight and gradBias bit-exact.
A bound of +inf marks an element whose value the device's rounding can legitimately change by any amount (for
example R where V is within its own error of 0); such elements are only checked to be finite."""
import math

import numpy as np
import torch

from oracle import vbnn_oracle as O

U32 = 2.0 ** -24          # fp32 unit roundoff
UBF = 2.0 ** -8           # bf16 unit roundoff
U16 = 2.0 ** -11          # fp16 unit roundoff (the bf16 weight mode keeps eps as fp16 for the dW epilogue)
ETA16 = 2.0 ** -25        # |rounding error| in fp16's subnormal range (|eps| < 2^-14)
ETA = 2.0 ** -150         # |rounding error| in fp32's subnormal range
ETA_BF = 2.0 ** -134      # the same for bf16
RSQ = 2.0 ** -21          # rsqrt.approx relative error
FLT_MIN = 2.0 ** -126
C_ACC = 2.0
EXACT = 2.0 ** 24         # integer partial sums below this are exact in fp32
LN_FLUSH = -90.0          # __expf(x) = ex2.approx.ftz(x log2 e) is exactly 0 below about -87.3: flushed, no error
INF = float("inf")


# ---------------------------------------------------------------- error-bound algebra
def _abs(t):
    return t.abs() if isinstance(t, torch.Tensor) else abs(t)


def mul_err(a, ea, b, eb):
    """|a' b' - a b| for |a' - a| <= ea, |b' - b| <= eb (0 * inf taken as 0: an exact zero times anything is 0)."""
    out = ea * _abs(b) + _abs(a) * eb + ea * eb
    return torch.nan_to_num(out, nan=0.0, posinf=INF)


def round_err(v, e, unit, tiny=None):
    """Bound after both sides store their value in a type of unit roundoff `unit`: v is the reference's stored value,
    e the bound on the difference before the store.  Where e == 0 both round the same number."""
    tiny = (ETA if unit <= U32 else ETA_BF) if tiny is None else tiny
    return torch.where(e > 0, e + unit * (2.0 * v.abs() + e) + tiny, torch.zeros_like(e))


def is_int(t):
    """Element-wise: an integer value (finite)."""
    return torch.isfinite(t) & (t == t.round())


def exact_sum(err, terms_mag, *ints):
    """The exactness rule, element-wise: True where the terms carry no error (`err` == 0), every tensor of `ints`
    (broadcast) is integer-valued and the terms' magnitudes sum below 2^24, so that the fp32 sum is exact."""
    ok = (err == 0) & (terms_mag < EXACT)
    for t in ints:
        ok = ok & is_int(t)
    return ok


def _zero_where(ok, e):
    return torch.where(ok, torch.zeros_like(e), e)


def _exact_rows(T, eT):
    """[rows] bool: every element of the row an integer with no operand error."""
    ok = is_int(T).all(dim=1)
    return ok if eT is None else ok & (eT == 0).all(dim=1)


def expf_err(x):
    """Bound on |__expf(x) - exp(x)|, x in fp64 (already the fp32 argument)."""
    v = torch.exp(x)
    e = v * (2.0 + torch.floor(1.173 * x.abs())) * 2.0 ** -23
    return torch.where(v < FLT_MIN, v, e)


def contraction_bound(A, B, eA=None, eB=None):
    """Bound on |got - A @ B^T| per element for one fp32-accumulated contraction over the last dimension.  A, B are the
    reference's operands as the device rounds them; eA, eB (optional, same shapes) bound the device's operands'
    distance from them."""
    aA, aB = A.abs(), B.abs()
    exact = _exact_rows(A, eA)[:, None] & _exact_rows(B, eB)[None, :]
    if eA is not None or eB is not None:
        eA = torch.zeros_like(aA) if eA is None else eA
        eB = torch.zeros_like(aB) if eB is None else eB
        nzA, nzB = ((aA + eA) > 0).double(), ((aB + eB) > 0).double()
        m = nzA @ nzB.t()
        big = torch.nan_to_num((aA + eA) @ (aB + eB).t(), posinf=INF)
        prop = torch.nan_to_num(eA @ aB.t() + aA @ eB.t() + eA @ eB.t(), nan=0.0, posinf=INF)
        prop = torch.where(m > 0, prop, torch.zeros_like(prop))
        out = prop + C_ACC * m * U32 * big + m * ETA
    else:
        m = (aA > 0).double() @ (aB > 0).double().t()
        big = aA @ aB.t()
        out = C_ACC * m * U32 * big + m * ETA
    return torch.where(exact & (big < EXACT), torch.zeros_like(out), out)


def violations(got, ref, bound):
    """Indices where |got - ref| > bound, or got is not finite.  Returns a list of (index tuple, got, ref, bound)."""
    got = torch.as_tensor(np.asarray(got, dtype=np.float64))
    ref = torch.as_tensor(ref, dtype=torch.float64)
    bound = torch.as_tensor(bound, dtype=torch.float64)
    bad = ~torch.isfinite(got) | ((got - ref).abs() > bound)
    idx = bad.nonzero().tolist()
    return [(tuple(i), float(got[tuple(i)]), float(ref[tuple(i)]), float(bound[tuple(i)])) for i in idx[:8]] + (
        [("...", int(bad.sum()))] if len(idx) > 8 else [])


# ---------------------------------------------------------------- one layer, values and bounds
class LayerPass:
    """One VBLinear / Linear layer of the oracle run forward and backward with the device's conventions, each value
    with its bound.  bf: VBNN_PREC_BF16 (operands rounded to bf16; the oracle must hold operand_round=round_bf16)."""

    def __init__(self, lyr, bf, strict=True):
        self.l, self.bf, self.strict = lyr, bf, strict
        self.unit = UBF if bf else U32
        self.vb = isinstance(lyr, O.VBLinearOracle)
        self.lrt = self.vb and lyr.lrt

    def _store(self, v, e):
        """A value the device keeps in the operand type (bf16 or fp32) after an fp32 computation."""
        return round_err(v, e, UBF) if self.bf else e

    def sample_bound(self, eps):
        """Bound on the device's sampled weight q(mu + sd * eps), sd = __expf(0.5 lvars)."""
        l = self.l
        half = 0.5 * l.lvars
        sd = torch.exp(half)
        pre = l.means + sd * eps
        e = eps.abs() * expf_err(half) + U32 * pre.abs() + ETA
        # sigma flushed to 0 on the device: it samples q(mu) exactly, and so does the reference here
        e = _zero_where((half < LN_FLUSH) & (l.weight == l.q(l.means)), e)
        return self._store(l.weight, e) if self.bf else e

    def forward(self, x, ex, noise=None):
        """x: the layer input as the reference holds it (operand-rounded), ex its bound.  noise: eps (weight mode,
        already passed to sample()) or zeta (LRT).  Returns (Y, E_Y) of the pre-activation output in fp32."""
        l = self.l
        self.x, self.ex = x, ex
        if self.lrt:
            Y = l.updateOutput(x, noise)
            q = l.q
            self.s2 = q(torch.exp(l.lvars))
            self.es2 = self._store(self.s2, expf_err(l.lvars))
            if self.bf:
                # bf16 rounding is monotonic: where both ends of __expf's error interval round to the reference's
                # bf16 value (sigma^2 = 2^-10, or a flushed 0), the device stores that same value
                ev, ee = torch.exp(l.lvars), expf_err(l.lvars)
                self.es2 = _zero_where((q(ev - ee) == self.s2) & (q(ev + ee) == self.s2), self.es2)
            self.mu = q(l.means)
            self.X2 = q(x * x)
            e2 = mul_err(x, ex, x, ex)
            if self.bf:
                e2 = e2 + torch.where((x * x < FLT_MIN) & (x != 0), ETA, 0.0)
                self.eX2 = round_err(self.X2, e2, UBF)
            else:
                self.eX2 = e2 + U32 * self.X2 + torch.where(x != 0, ETA, 0.0)
            M = x @ self.mu.t() + l.bias
            eM = contraction_bound(x, self.mu, ex, None)
            V = self.X2 @ self.s2.t()
            eV = contraction_bound(self.X2, self.s2, self.eX2, self.es2)
            # the convention: R := 0 where V == 0 (the oracle's zeta / (2 sqrt 0) is +-inf or NaN)
            zeta = l.zeta
            sqV = V.sqrt()
            l._R = torch.where(V == 0, torch.zeros_like(V), l._R)
            Y = torch.where(V == 0, M, Y)
            l.output = Y
            Vlo = (V - eV).clamp(min=0)
            esq_exact = torch.where(V > 0, eV / (sqV + Vlo.sqrt()), eV.sqrt())
            esq = torch.where((V > 0) | (eV > 0), esq_exact + RSQ * (sqV + esq_exact) + U32 * sqV + ETA, torch.zeros_like(V))
            ers = torch.where(Vlo > 0, esq_exact / (sqV * Vlo.sqrt()) + RSQ / Vlo.sqrt().clamp(min=1e-300),
                              torch.where((V == 0) & (eV == 0), torch.zeros_like(V), torch.full_like(V, INF)))
            eR = 0.5 * zeta.abs() * ers + U32 * l._R.abs()
            eR = torch.nan_to_num(eR, nan=0.0, posinf=INF)
            self.eR = round_err(l._R, eR, UBF) if self.bf else eR
            # the epilogue's adds round only where the accumulators are not exactly 0 (0 + b + 0 * zeta = b)
            eY = eM + mul_err(sqV, esq, zeta, 0.0) + self._live(x, ex) * (U32 * (M.abs() + Y.abs()) + ETA)
            # M exact, sqrt(0) zeta = 0, an integer bias: the epilogue's adds are exact
            eY = _zero_where(exact_sum(eM + eV, Y.abs(), Y, l.bias) & (V == 0), eY)
            self.V, self.eV = V, eV
            return Y, eY
        Y = l.updateOutput(x)
        W = l.weight if self.vb else l.q(l.weight)
        self.W = W
        if not hasattr(self, "eW"):
            self.eW = torch.zeros_like(W)
        eC = contraction_bound(x, W, ex, self.eW)
        eY = _zero_where(exact_sum(eC, Y.abs(), Y, l.bias), eC + self._live(x, ex) * U32 * Y.abs())
        return Y, eY

    @staticmethod
    def _live(x, ex):
        """[N x 1]: 1 for rows with a non-zero (or uncertain) input, 0 for rows the device knows are all zero."""
        return (((x.abs() + ex) > 0).any(dim=1, keepdim=True)).to(x.dtype)

    def backward(self, g, eg, eps=None):
        """g: dL/d(output) as the reference holds it (operand-rounded), eg its bound.  Accumulates this sample's
        gradWeight / gradSum / gradBias (and their bounds) and returns (gradInput, its bound), both fp32."""
        l, x, ex = self.l, self.x, self.ex
        gi = l.updateGradInput(x, g)
        before_w, before_s = l.gradWeight.clone(), (l.gradSum.clone() if self.vb else None)
        l.accGradParameters(x, g, 1.0)
        dW = l.gradWeight - before_w
        edW = contraction_bound(g.t(), x.t(), eg.t(), ex.t())
        ones = torch.ones(1, g.shape[0], dtype=g.dtype)
        edB = contraction_bound(g.t(), ones, eg.t(), None)[:, 0]
        if self.lrt:
            H = l.q(g * l._R)
            eH = mul_err(g, eg, l._R, self.eR) + U32 * (g * l._R).abs()
            eH = round_err(H, eH, UBF) if self.bf else eH
            a1e = contraction_bound(g, self.mu.t(), eg, None)
            a2 = H @ self.s2
            a2e = contraction_bound(H, self.s2.t(), eH, self.es2.t())
            egi = a1e + 2.0 * mul_err(x, ex, a2, a2e) + U32 * (2.0 * (x * a2).abs() + gi.abs()) + ETA
            egi = _zero_where((a1e == 0) & (a2 == 0) & (a2e == 0), egi)      # G mu exact, + 2 X .* 0
            dS = l.gradSum - before_s
            edS = contraction_bound(H.t(), self.X2.t(), eH.t(), self.eX2.t())
            mS = H.abs().t() @ self.X2.abs()
        else:
            W = self.W
            egi = contraction_bound(g, W.t(), eg, self.eW.t())
            if self.vb:
                dS = l.gradSum - before_s
                e16 = U16 * eps.abs() + ETA16 if self.bf else 0.0
                edS = edW * eps.abs() + dW.abs() * e16 + U32 * dS.abs()
                mS = dS.abs()
            else:
                dS = edS = mS = None
        self.acc = getattr(self, "acc", [])
        # (value, bound, the magnitudes of its terms): the device may sum the samples' terms in one fp32 accumulator
        self.acc.append((dW, edW, g.abs().t() @ x.abs(), dS, edS, mS, g.sum(0), edB, g.abs().sum(0)))
        return gi, egi

    def grad_bounds(self):
        """(gradWeight, gradSum, gradBias) bounds of the samples accumulated so far: each sample's bound, plus the
        fp32 accumulation across samples."""
        S = len(self.acc)
        out = []
        for j in (0, 3, 6):
            if self.acc[0][j] is None:
                out.append(None)
                continue
            e = sum(a[j + 1] for a in self.acc)
            mag = sum(a[j].abs() for a in self.acc)
            terms = sum(a[j + 2] for a in self.acc)
            out.append(_zero_where(exact_sum(e, terms, *[a[j] for a in self.acc]), e + C_ACC * S * U32 * mag))
        return out


def relu_store(ps, y, ey):
    """nn.ReLU and the store of the next layer's operand: (a, E_a)."""
    a = ps.l.q(torch.clamp(y, min=0))
    ea = round_err(a, ey, UBF) if ps.bf else ey
    return a, torch.where(y + ey <= 0, torch.zeros_like(ea), ea)     # the device's y <= 0 too: both store 0


def relu_backward(ps, a, ea, gi, egi):
    """ReLU backward on the stored activation a (bound ea): the mask x > 0 is uncertain where a is within its bound
    of 0, and there the whole gradient is uncertain.  Then the gradient operand's store."""
    q = ps.l.q
    mask = (a > 0).to(a.dtype)
    g = q(gi * mask)
    unsure = ((a > 0) & (a <= ea)) | ((a == 0) & (ea > 0))
    eg = torch.where(unsure, gi.abs() + egi, egi * mask)
    return g, (round_err(g, eg, UBF) if ps.bf else eg)


def mlp_minibatch(ref, x, G, noise, lrt, bf, strict, opt):
    """One split minibatch (vbnn_mlp_forward_train with the chosen dL/dY = G [S x N x C], then the backward of
    vbnn_mlp_backward_update) through the oracle net `ref` with the device's conventions.  x: the network input as
    fp64 holding fp32 values.  Returns dict of (value, bound): logits [S x N x C], dX, and per layer gW / gS / gB.
    The parameters are not updated."""
    S = opt["S"]
    layers = ref.vb + [ref.out]
    passes = [LayerPass(l, bf, strict) for l in layers]
    ref.resetGradients()
    x = ref.q(x)
    ex0 = torch.zeros_like(x)
    Y, EY, dX, EdX = [], [], 0, 0
    dX_mag, dX_err = 0, 0             # the dX sum's terms, sum over samples of |G| |W| of the first layer; their bounds
    for s in range(S):
        if not lrt:
            ref.sample(noise[s])
            for k, ps in enumerate(passes):
                if ps.vb:
                    ps.eW = ps.sample_bound(noise[s][k])
        acts, eacts = [x], [ex0]
        for k, ps in enumerate(passes):
            z = noise[s][k] if (lrt and ps.vb) else None
            y, ey = ps.forward(acts[-1], eacts[-1], z)
            if k < len(passes) - 1:
                a, ea = relu_store(ps, y, ey)
                acts.append(a); eacts.append(ea)
        Y.append(y); EY.append(ey)
        g = ref.q(G[s])
        eg = torch.zeros_like(g)
        for k in range(len(passes) - 1, -1, -1):
            ps = passes[k]
            gi, egi = ps.backward(g, eg, None if lrt or not ps.vb else noise[s][k])
            if k > 0:
                g, eg = relu_backward(passes[k - 1], acts[k], eacts[k], gi, egi)
            else:
                dX, EdX = dX + gi, EdX + egi + C_ACC * U32 * gi.abs()
                dX_mag, dX_err = dX_mag + g.abs() @ (ps.mu if ps.lrt else ps.W).abs(), dX_err + egi
    EdX = _zero_where(exact_sum(dX_err, dX_mag, dX), EdX)
    out = dict(logits=(torch.stack(Y), torch.stack(EY)), dX=(dX, EdX))
    for k, ps in enumerate(passes):
        ew, es, eb = ps.grad_bounds()
        l = ps.l
        out[f"gW{k}"] = (l.gradWeight.clone(), ew)
        out[f"gB{k}"] = (l.gradBias.clone(), eb)
        if ps.vb:
            out[f"gS{k}"] = (l.gradSum.clone(), es)
    return out


# ---------------------------------------------------------------- the loss with the device's target rule
def first_argmax(Y):
    """Lowest index among tied maxima, per row."""
    return torch.from_numpy(np.argmax(np.asarray(Y, dtype=np.float64), axis=-1))


def classnll_device(Y, t1):
    """LogSoftMax + ClassNLL (size-averaged) of one sample's logits Y [N x C] under the device's target rule.
    t1: 1-based targets (any integer).  Returns (error, accuracy %, dL/dY, logp)."""
    N, C = Y.shape
    logp = O.log_softmax(Y)
    tgt = t1.long() - 1
    valid = (tgt >= 0) & (tgt < C)
    rows = torch.arange(N)[valid]
    err = float(-logp[rows, tgt[valid]].sum() / N)
    acc = float((first_argmax(Y)[valid] == tgt[valid]).sum()) / N * 100.0
    g = torch.exp(logp) / N
    g[rows, tgt[valid]] -= 1.0 / N
    return err, acc, g, logp


# ---------------------------------------------------------------- exact operands: the whole minibatch in fp64 torch
def bf16(t):
    return t.to(torch.bfloat16).to(t.dtype)


def exact_minibatch(X, params, G, lrt, vb, eps=None):
    """The split minibatch of a bf16 net whose log-variances flush sigma to 0 (lvars < LN_FLUSH), in plain fp64 torch
    on any device: the ReLU chain a <- bf16(relu(a W^T + b)) forward and g <- bf16((g W) .* (a > 0)) back, W the means
    (or the Linear weight).  X [N x I0], params [(W, b)] per layer, G [S x N x C] = dL/dY, vb[k]: layer k is a
    VBLinear, eps[s][k]: weight-mode epsilon [O x I] of VB layer k in sample s (for gradSum).  Operands must be
    integer-valued: every value is then exact, and the 2^24 condition of the exactness rule is asserted on every
    contraction and sum, so the device must reproduce logits, dX, gW and gB bit for bit.  Returns dict of (value,
    bound) with bound 0, except weight-mode gradSum sum_s dW_s .* eps_s: its bound allows eps in fp16 and the fp32
    products and sums.  Under local reparameterisation gradSum is exactly 0."""
    S, nl = G.shape[0], len(params)
    assert is_int(X).all() and is_int(G).all() and all(is_int(W).all() and is_int(b).all() for W, b in params)
    worst = {}

    def note(name, mag):
        worst[name] = max(worst.get(name, 0.0), float(mag.max()))

    out = {f"gW{k}": 0 for k in range(nl)}
    out.update({f"gB{k}": 0 for k in range(nl)})
    gS = {k: 0 for k in range(nl) if vb[k]}
    eS = {k: 0 for k in range(nl) if vb[k]}
    mS = {k: 0 for k in range(nl) if vb[k]}
    mW = [0] * nl
    mB = [0] * nl
    logits, dX, mX = [], 0, 0
    for s in range(S):
        acts = [bf16(X)]
        for k, (W, b) in enumerate(params):
            y = acts[-1] @ W.t() + b
            note(f"fwd{k}", acts[-1].abs() @ W.abs().t() + b.abs())
            if k < nl - 1:
                acts.append(bf16(y.clamp(min=0)))
        logits.append(y)
        g = bf16(G[s])
        for k in range(nl - 1, -1, -1):
            W, a = params[k][0], acts[k]
            dW = g.t() @ a
            out[f"gW{k}"] = out[f"gW{k}"] + dW
            out[f"gB{k}"] = out[f"gB{k}"] + g.sum(0)
            mW[k] = mW[k] + g.abs().t() @ a.abs()
            mB[k] = mB[k] + g.abs().sum(0)
            if vb[k] and not lrt:
                dS = dW * eps[s][k]
                gS[k] = gS[k] + dS
                eS[k] = eS[k] + dW.abs() * (eps[s][k].abs() * U16 + ETA16) + U32 * dS.abs()
                mS[k] = mS[k] + dS.abs()
            gi = g @ W
            mag = g.abs() @ W.abs()
            if k > 0:
                note(f"dx{k}", mag)
                g = bf16(gi * (acts[k] > 0))
            else:
                dX, mX = dX + gi, mX + mag
    for k in range(nl):
        note(f"dW{k}", mW[k])
        note(f"gB{k}", mB[k])
    note("dX", mX)
    over = {n: w for n, w in worst.items() if w >= EXACT}
    assert not over, ("the 2^24 condition fails: fp32 is not exact on", over)
    z = lambda v: (v, torch.zeros_like(v))
    res = dict(logits=z(torch.stack(logits)), dX=z(dX))
    for k in range(nl):
        res[f"gW{k}"] = z(out[f"gW{k}"])
        res[f"gB{k}"] = z(out[f"gB{k}"])
        if vb[k]:
            W = params[k][0]
            res[f"gS{k}"] = z(torch.zeros_like(W)) if lrt else (gS[k], eS[k] + C_ACC * S * U32 * mS[k])
    res["worst"] = worst
    return res
