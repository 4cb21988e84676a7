"""CPU checks behind the live hyper-parameters (vbnn_layer_set_opts, VBLinear.set_opt / MLP.set_opt):
  * under a schedule that changes every live value at every step, tests/update_reference.py fed each step's values
    agrees with the oracle's VBLinear.update whose optimiser tables and opt.B are rewritten the same way (the Torch7
    idiom), so both stay valid references for the GPU tests of tests/test_gpu_update_schedule.py;
  * set_opt maps the config dict as buildModel does and keeps every key but the live ones in the net's opt;
  * the "{k}.opts" checkpoint key survives checkpoint.save_net / load_net."""
import math

import numpy as np
import torch

import update_reference as R
from oracle import vbnn_oracle as O
from vbnn_b200 import _lib as L
from vbnn_b200 import checkpoint
from vbnn_b200.config import default_opt, opts_struct, with_live

F = np.float32

# one row per step: B, lr_bias, lr_mu, lr_var, beta1, beta2, eps -- every value changes at every step
SCHEDULE = [
    (10.0, 1e-3, 1e-4, 0.05, 0.9, 0.999, 1e-8),
    (25.0, 5e-4, 3e-4, 0.02, 0.8, 0.99, 1e-6),
    (60.0, 2e-3, 5e-5, 0.08, 0.95, 0.995, 1e-7),
    (200.0, 1e-4, 1e-3, 0.01, 0.5, 0.9, 1e-5),
    (1e6, 0.0, 0.0, 0.0, 0.0, 0.0, 1e-8),
]


def ref_opt(row, S, lrt):
    B, lr_bias, lr_mu, lr_var, b1, b2, eps = row
    return dict(B=B, S=S, lr_bias=lr_bias, lr_mu=lr_mu, lr_var=lr_var, beta1=b1, beta2=b2, eps=eps, lrt=lrt)


def set_tables(ol, oo, row):
    """What a Torch7 user writes between minibatches: opt.B and the layer's optimiser tables."""
    B, lr_bias, lr_mu, lr_var, b1, b2, eps = row
    oo["B"] = B
    ol.biasState["learningRate"] = lr_bias
    for st, lr in ((ol.meanState, lr_mu), (ol.varState, lr_var)):
        st.update(learningRate=lr, beta1=b1, beta2=b2, epsilon=eps)


def test_reference_follows_a_schedule_like_the_oracle():
    """Each step from the oracle's own state: the reference fed that step's values equals the oracle's update to within
    the bound plus 2e-5 per element (the fp32 constants, as test_update_reference_cpu.py states)."""
    O_, I, S, nth = 6, 11, 3, 8
    rng = np.random.RandomState(0)
    for lrt in (False, True):
        oo = dict(var_init=1e-3, mu_init=0, B=1.0, S=S, state=dict(learningRate=0.0), meanState=dict(learningRate=0.0),
                  varState=dict(learningRate=0.0), reparam="local" if lrt else "weight")
        ol = O.VBLinearOracle(I, O_, oo)
        ol.means.copy_(torch.from_numpy(F(rng.randn(O_, I) * 0.2).astype(np.float64)))
        ol.lvars.copy_(torch.from_numpy(F(rng.uniform(math.log(1e-3), math.log(1e-1), (O_, I))).astype(np.float64)))
        for t, row in enumerate(SCHEDULE):
            gW = torch.from_numpy(F(rng.randn(O_, I)).astype(np.float64))
            gS = torch.from_numpy(F(rng.randn(O_, I) * 10).astype(np.float64))
            gB = torch.from_numpy(F(rng.randn(O_)).astype(np.float64))
            z = torch.zeros(O_, I, dtype=torch.float64)
            st = dict(mu=ol.means.clone(), lv=ol.lvars.clone(), bias=ol.bias.clone(), gW=gW, gS=gS, gB=gB, t=t,
                      m_mu=ol.meanState.get("m", z).clone(), v_mu=ol.meanState.get("v", z).clone(),
                      m_var=ol.varState.get("m", z).clone(), v_var=ol.varState.get("v", z).clone())
            opt = ref_opt(row, S, lrt)
            ref = R.update(st, opt, R.Prior("empirical", terms=R.update_terms(O_, I, 1, nth)))
            set_tables(ol, oo, row)
            ol.gradWeight.copy_(gW); ol.gradSum.copy_(gS); ol.gradBias.copy_(gB)
            ol.update(oo)
            got = dict(mu=ol.means, lv=ol.lvars, m_mu=ol.meanState["m"], v_mu=ol.meanState["v"],
                       m_var=ol.varState["m"], v_var=ol.varState["v"], bias=ol.bias)
            for k, v in got.items():
                r, b = ref[k]
                tol = b + 2e-5 * r.abs()
                assert ((v - r).abs() <= tol).all(), (lrt, t, k, float((v - r).abs().max()), float(tol.max()))


def test_a_schedule_changes_the_reference():
    """The schedule is not a no-op in the reference: the same gradients under the first row and under the second give
    different means, log-variances and bias."""
    rng = np.random.RandomState(1)
    d = lambda a: torch.from_numpy(np.asarray(a, F).astype(np.float64))
    st = dict(mu=d(rng.randn(5, 8)), lv=d(rng.uniform(-6, -2, (5, 8))), bias=d(rng.randn(5)), gW=d(rng.randn(5, 8)),
              gS=d(rng.randn(5, 8)), gB=d(rng.randn(5)), t=2, m_mu=d(rng.randn(5, 8) * 0.1),
              v_mu=d(rng.rand(5, 8) * 0.1), m_var=d(rng.randn(5, 8) * 0.1), v_var=d(rng.rand(5, 8) * 0.1))
    pr = R.Prior("empirical", terms=R.update_terms(5, 8, 1, 8))
    a = R.update(st, ref_opt(SCHEDULE[0], 2, False), pr)
    b = R.update(st, ref_opt(SCHEDULE[1], 2, False), pr)
    for k in ("mu", "lv", "bias"):
        assert not torch.equal(a[k][0], b[k][0]), k


def _fields(o):
    return {f: getattr(o, f) for f, _ in L.VbnnOpts._fields_}


def test_set_opt_keeps_the_fixed_keys_and_takes_the_live_ones():
    """set_opt passes opts_struct(opt) -- buildModel's mapping -- and stores with_live(net.opt, opt) as the net's opt:
    the live keys (B and the three optimiser tables) are the new dict's, every other key stays the net's, and mapping
    the stored dict gives what was passed on every live field."""
    built = default_opt(B=123.0, S=4, var_init=0.02, mu_init=1, reparam="local", precision="bf16", hidden=[7, 9],
                        strict_reference=False, state=dict(learningRate=0.003), varState=dict(learningRate=0.07),
                        meanState=dict(learningRate=2e-4, beta1=0.85, beta2=0.99, epsilon=1e-6))
    new = default_opt(B=9.0, S=1, reparam="weight", hidden=[3], state=dict(learningRate=0.01),
                      varState=dict(learningRate=0.002), meanState=dict(learningRate=5e-5, beta1=0.7, epsilon=1e-7))
    kept = with_live(built, new)
    for k in built:
        if k not in ("B", "state", "meanState", "varState"):
            assert kept[k] == built[k], k
    got, passed, before = _fields(opts_struct(kept)), _fields(opts_struct(new)), _fields(opts_struct(built))
    for f in got:
        assert got[f] == (passed[f] if f in L.LIVE_OPTS else before[f]), f
    # meanState without beta2: optim.adam's default, as at creation
    assert got["adam_beta2"] == F(0.999) and got["adam_beta1"] == F(0.7)
    assert built["meanState"]["beta2"] == 0.99                  # the net's dict itself is not modified
    # a layer's report (field -> value) maps back to the same values
    live = {f: passed[f] for f in L.LIVE_OPTS}
    back = _fields(opts_struct(with_live(built, live)))
    assert all(back[f] == live[f] for f in L.LIVE_OPTS)


class _Net:
    """What checkpoint.save_net / load_net use of an MLP."""
    def __init__(self, sd, opt):
        self.sd, self.opt, self.loaded = sd, opt, None

    def state_dict(self):
        return self.sd

    def load_state_dict(self, sd):
        self.loaded = sd


def test_opts_key_round_trips_through_a_checkpoint(tmp_path):
    live = torch.tensor(SCHEDULE[1], dtype=torch.float32)
    sd = {"sizes": [3, 4, 2], "step": 7, "0.t": 2, "0.opts": live, "1.opts": live * 2}
    net = _Net(sd, default_opt(B=25.0))
    checkpoint.save_net(net, str(tmp_path))
    back = _Net(None, None)
    opt = checkpoint.load_net(back, str(tmp_path))
    assert opt["B"] == 25.0
    for k in ("0.opts", "1.opts"):
        assert back.loaded[k].dtype == torch.float32 and torch.equal(back.loaded[k], sd[k]), k
    assert len(L.LIVE_OPTS) == live.numel() == 7
