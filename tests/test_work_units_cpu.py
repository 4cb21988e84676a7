"""The work-unit count the multi-wave GPU tests assert on (tests/work_units.py), pinned to the C3 step's GEMMs."""
from work_units import per_slot, units


def test_c3_units():
    # C3 (4096-4096x4-1000, N = 8192, S = 1) on 256 x 256 CTA-pair tiles, 74 pair slots of 148 SMs
    assert units(8192, 4096, 256, 2) == 512                          # hidden forward / dx: M = N, N = O
    assert round(per_slot(8192, 4096, 256, 2, 148), 1) == 6.9
    assert units(4096, 4096, 256, 2, z_once=True) == 256               # hidden dW: M = O, N = I
    assert round(per_slot(4096, 4096, 256, 2, 148, z_once=True), 1) == 3.5
    # the ragged raw GEMM: 1024 single-CTA units, 256 pair units
    assert units(2000, 1960, 128, 1, batch=4) == 1024
    assert units(2000, 1960, 256, 2, batch=4) == 256
    # batch multiplies the units unless one unit walks every z
    assert units(4096, 4096, 128, 1, batch=2) == 2 * units(4096, 4096, 128, 1, batch=2, z_once=True)
