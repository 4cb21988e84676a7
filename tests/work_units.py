"""Work units of one tcgen05 GEMM launch on a given tile shape, as gemm_tc.cu's launch_cfg counts them: one unit per
(128 * cg) x bn output tile, times the batch unless one unit walks every z (the dW modes accumulate the samples in
one tile; the sample-summing dX form K-concatenates them).  A persistent CTA (cg = 1) or CTA pair (cg = 2) runs
units / (#SM / cg) of them on average; from the second one on it carries its pipeline state across tiles."""


def ceil_div(a, b):
    return -(-a // b)


def units(M, N, bn, cg, batch=1, z_once=False):
    """Work units of an M x N output on (128 * cg) x bn tiles."""
    return ceil_div(M, 128 * cg) * ceil_div(N, bn) * (1 if z_once else batch)


def per_slot(M, N, bn, cg, sms, batch=1, z_once=False):
    """Units per resident CTA (cg = 1) or CTA pair (cg = 2)."""
    return units(M, N, bn, cg, batch, z_once) / (sms // cg)
