"""Run by tests/test_gpu_parity.py::test_batch_splitting_paths in a subprocess with B200_WS_BUDGET_MB=1, which forces the
rarely-taken sub-batching loops of the host-buffer MSM and NTT entry points (one column per device call) and of evaluate_h's
coefficient-column transforms (three columns per group)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

from ezkl_b200 import _native as nat  # noqa: E402
from ezkl_b200 import evaluation as ev  # noqa: E402
from ezkl_b200 import halo2 as h2  # noqa: E402
from oracle import oracle as orc  # noqa: E402

assert os.environ.get("B200_WS_BUDGET_MB") == "1"
nat.init(-1)
n, k = 1 << 11, 11
bases_np = orc.gen_bases(n, seed=91)
bases = h2.Bases(bases_np, window_bits=9)
cols = [orc.gen_scalars(n, seed=92 + i) for i in range(5)]
got = h2.best_multiexp_batch(cols, bases)
for c, g in zip(cols, got):
    assert np.array_equal(g[:8], orc.msm(c, bases_np, 4))
dom = h2.EvaluationDomain(5, k)
coeffs = dom.lagrange_to_coeff_batch(cols)
for c, v in zip(coeffs, cols):
    assert np.array_equal(c, orc.lagrange_to_coeff(v, k, 4))
exts = dom.coeff_to_extended_batch(coeffs)
for e, c in zip(exts, coeffs):
    assert np.array_equal(e, orc.coeff_to_extended(c, dom.extended_k, 4))
# five coefficient columns around one extended column: groups of three (a full group with a gap in its column indices, then the rest)
ext_col = orc.gen_scalars(1 << dom.extended_k, seed=97)
polys = coeffs[:2] + [ext_col] + coeffs[2:]
cosets = exts[:2] + [ext_col] + exts[2:]
prog = ev.QuotientProgram(ev.fold_y([ev.Query(0) * ev.Query(1, 1) - ev.Query(2, -1), ev.Query(3) * ev.Query(4) + ev.Query(5, 2)], 0x77))
loads, consts, instrs = prog.arrays()
num = orc.quotient_eval(cosets, k, dom.extended_k, loads, consts, instrs, threads=4)
want = orc.extended_to_coeff(orc.divide_by_vanishing(num, k, dom.extended_k), dom.extended_k, 4)
assert np.array_equal(ev.evaluate_h_from_polys(prog, polys, dom, finish=True), want)
print("split paths OK")
