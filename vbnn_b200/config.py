"""config.lua restated (reference config.lua:1-68): the same keys with the same shipped values,
plus the keys the B200 build adds (SURVEY.md section 5: reparam, precision, seed, ngpu)."""
from __future__ import annotations

from . import _lib as L


def default_opt(**over):
    opt = dict(
        threads=8, network_to_load="", network_name="exp", type="vb", dataset="mnist",
        cuda=True, batchSize=1, testBatchSize=100,                      # config.lua:5-12
        trainSize=100, testSize=1000, classes=list("0123456789"),       # config.lua:15-17
        geometry=(28, 28), input_size=28 * 28,                          # config.lua:18-19
        plot=True, B=1000000.0, hidden=[10], S=30, testSamples=30,      # config.lua:28-33
        quicktest=False, log=True,                                      # config.lua:34-35
        mu_init=0, var_init=0.001, msr_init=False,                      # config.lua:43-45
        state=dict(learningRate=0.001),                                 # config.lua:51-54
        varState=dict(learningRate=0.05),                               # config.lua:55-59
        meanState=dict(learningRate=0.0001),                            # config.lua:60-64
        # new keys
        reparam="weight",        # 'weight' = reference sampling, 'local' = local reparameterisation
        precision="fp32",        # 'fp32' (exact-parity CUDA-core GEMM) or 'bf16' (tcgen05)
        strict_reference=True,   # reproduce quirks Q1/Q6
        vb_output=False,         # convnet.lua:30: VBLinear output layer instead of nn.Linear
        seed=3,                  # config.lua:40 torch.manualSeed(3)
        ngpu=1,
    )
    opt.update(over)
    return opt


def opts_struct(opt) -> L.VbnnOpts:
    """buildModel's mapping of the config dict to vbnn_opts; set_opt passes the same mapping to vbnn_*_set_opts,
    which refuses a change of any field but the live ones (L.LIVE_OPTS)."""
    o = L.VbnnOpts()
    L.lib().vbnn_opts_default(o)
    o.var_init = float(opt["var_init"])
    o.msr_init = 1 if opt.get("msr_init") else 0
    o.mu_init = float(opt["mu_init"])
    o.S = int(opt["S"])
    _live_fields(o, opt)
    o.reparam = L.REPARAM_LOCAL if opt.get("reparam", "weight") == "local" else L.REPARAM_WEIGHT
    o.precision = L.PREC_BF16 if opt.get("precision", "fp32") == "bf16" else L.PREC_FP32
    o.strict_reference = 1 if opt.get("strict_reference", True) else 0
    return o


def _live_fields(o, opt):
    o.B = float(opt["B"])
    o.lr_bias = float(opt["state"]["learningRate"])
    o.lr_mu = float(opt["meanState"]["learningRate"])
    o.lr_var = float(opt["varState"]["learningRate"])
    o.adam_beta1 = float(opt["meanState"].get("beta1", 0.9))
    o.adam_beta2 = float(opt["meanState"].get("beta2", 0.999))
    o.adam_eps = float(opt["meanState"].get("epsilon", 1e-8))


def with_live(opt, src):
    """A copy of the config dict opt whose live keys -- B and the optimiser tables state / meanState / varState, the
    keys opts_struct reads the live fields from -- are src's.  src: a config dict, or {field: value} over L.LIVE_OPTS
    (what a layer reports).  Every other key keeps opt's value."""
    out = dict(opt)
    if all(f in src for f in L.LIVE_OPTS):
        out["B"] = src["B"]
        out["state"] = dict(opt["state"], learningRate=src["lr_bias"])
        out["meanState"] = dict(opt["meanState"], learningRate=src["lr_mu"], beta1=src["adam_beta1"],
                                beta2=src["adam_beta2"], epsilon=src["adam_eps"])
        out["varState"] = dict(opt["varState"], learningRate=src["lr_var"])
        return out
    out["B"] = src["B"]
    for k in ("state", "meanState", "varState"):
        out[k] = dict(src[k])
    return out
