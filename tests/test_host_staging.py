"""Host-pointer entry points at sizes where caller memory moves through the pinned bounce buffers (8 MiB and more, in 16 MiB
chunks): results must match the oracle exactly, including a final partial chunk."""
import ctypes as C

import numpy as np
import pytest

from ezkl_b200 import _native as nat
from ezkl_b200 import evaluation as ev
from ezkl_b200 import halo2 as h2
from oracle import oracle as orc
from tests import helpers as H

pytestmark = pytest.mark.gpu
THREADS = orc.host_threads()
N_CHUNK_AND_TAIL = (1 << 19) + 3          # 16 MiB + 96 B of Fr: one full bounce chunk and a partial one


@pytest.fixture(scope="module", autouse=True)
def _init():
    nat.init(-1)
    yield


def test_divide_by_vanishing_poly_across_bounce_chunks():
    dom = h2.EvaluationDomain(5, 17)
    n, period = N_CHUNK_AND_TAIL, dom.t_evaluations.shape[0]
    a = orc.gen_scalars(n, seed=190)
    got = a.copy()
    nat.check(nat.lib().b200_poly_scale_cycle(nat.ptr(got), C.c_size_t(n), nat.ptr(dom.t_evaluations), C.c_uint32(period)))
    want = orc.poly_op("mul", a, np.ascontiguousarray(np.tile(dom.t_evaluations, (n // period + 1, 1))[:n]), threads=THREADS)
    assert np.array_equal(got, want)


def test_g_to_lagrange_of_exactly_8_mib():
    """k = 17: 2^17 affine points are 8 MiB, the smallest copy that takes the bounce path.  Known answer: the trapdoor SRS's
    g_lagrange, built by fixed-base multiplication of L_i(s) without the group FFT."""
    params = h2.ParamsKZG.setup(17, 0x5EED17)
    assert params.g.nbytes == 8 << 20
    assert np.array_equal(h2.g_to_lagrange(params.g, 17), params.g_lagrange)


def test_bases_registered_from_host_across_bounce_chunks():
    n = (1 << 17) + 5
    pts = orc.gen_bases(n, seed=191, threads=THREADS)
    sc = orc.gen_scalars(n, seed=192)
    bases = h2.Bases(pts)
    try:
        got = h2.best_multiexp(sc, bases)
    finally:
        bases.release()
    assert np.array_equal(got[:8], orc.msm(sc, pts, THREADS))


def test_lookup_multiplicities_over_8_mib():
    n_table, n_rows, n_inputs = 1 << 17, 1 << 17, 2               # 4 MiB of table and 8 MiB of inputs
    table = orc.gen_scalars(n_table, seed=193)
    rng = np.random.default_rng(194)
    idx = [rng.integers(0, n_table, n_rows) for _ in range(n_inputs)]
    inputs = [np.ascontiguousarray(table[i]) for i in idx]
    counts = np.bincount(np.concatenate(idx), minlength=n_table)
    want = H.fr_array(range(int(counts.max()) + 1))[counts]
    assert np.array_equal(ev.lookup_multiplicities(table, inputs, n_rows), want)
