"""GPU parity tests: the CUDA path (through the C ABI / the halo2-mirror host layer) against the CPU oracle, the
reference's golden fixtures, and size-independent properties at BASELINE.json's full sizes.  Bit-exact everywhere
(integer arithmetic); run on the B200 box with `pytest -m gpu`."""
import ctypes as C
import random

import numpy as np
import pytest

from ezkl_b200 import _native as nat
from ezkl_b200 import halo2 as h2
from oracle import oracle as orc
from oracle import pyref
from tests import helpers as H

pytestmark = pytest.mark.gpu
THREADS = orc.host_threads()


@pytest.fixture(scope="module", autouse=True)
def _init():
    nat.init(-1)
    yield


def jac_to_affine(j):
    """normalised Jacobian wire [12] -> affine wire [8] ((0,1,0) -> (0,0))."""
    j = np.asarray(j, np.uint64).reshape(-1, 12)
    out = j[:, :8].copy()
    for i in range(j.shape[0]):
        if not j[i, 8:].any():
            out[i] = 0
        else:
            assert np.array_equal(j[i, 8:], np.array(H.fq_wire(1)))
    return out


# ---- layer 0: device field arithmetic and group law -------------------------------------------------------------
def test_device_field_ops():
    L = nat.lib()
    rng = random.Random(5)
    for fid, (field, mod) in enumerate((("fr", pyref.R), ("fq", pyref.P))):
        xs = [rng.randrange(mod) for _ in range(2000)] + [0, 1, mod - 1, mod - 2, 2]
        ys = [rng.randrange(mod) for _ in range(2000)] + [mod - 1, 0, mod - 1, mod - 2, mod - 1]
        a = np.stack([H.int_to_limbs(pyref.to_mont(x, mod)) for x in xs])
        b = np.stack([H.int_to_limbs(pyref.to_mont(y, mod)) for y in ys])
        for opi, op in enumerate(("add", "sub", "mul")):
            out = np.zeros_like(a)
            nat.check(nat.dbg_lib().b200_debug_field_op(fid, opi, nat.ptr(a), nat.ptr(b), nat.ptr(out), C.c_size_t(len(xs))))
            assert np.array_equal(out, orc.field_op(field, op, a, b)), (field, op)
        out = np.zeros_like(a)
        nat.check(nat.dbg_lib().b200_debug_field_op(fid, 3, nat.ptr(a), nat.ptr(b), nat.ptr(out), C.c_size_t(len(xs))))
        assert np.array_equal(out, orc.fr_inv(a) if field == "fr" else orc.fq_inv(a)), field


def test_device_group_law():
    L = nat.lib()
    rng = random.Random(6)
    bases = orc.gen_bases(256, seed=9)
    A, B = bases[:128].copy(), bases[128:].copy()
    A[0] = 0
    B[1] = 0
    A[2] = B[2]
    n = C.c_size_t(128)
    out = np.zeros_like(A)
    nat.check(nat.dbg_lib().b200_debug_g1_op(0, nat.ptr(A), nat.ptr(B), nat.ptr(out), n))
    assert np.array_equal(out, orc.g1_add_affine(A, B))
    nat.check(nat.dbg_lib().b200_debug_g1_op(1, nat.ptr(A), nat.ptr(B), nat.ptr(out), n))
    assert np.array_equal(out, orc.g1_add_affine(A, A))
    K = B.copy()
    ks = [rng.randrange(1 << 20) for _ in range(128)]
    ks[3], ks[4] = 0, 1
    for i, k in enumerate(ks):
        K[i, 0] = k
    nat.check(nat.dbg_lib().b200_debug_g1_op(2, nat.ptr(A), nat.ptr(K), nat.ptr(out), n))
    assert np.array_equal(out, orc.g1_scalar_mul(A, H.fr_array(ks)))
    nat.check(nat.dbg_lib().b200_debug_g1_op(3, nat.ptr(A), nat.ptr(B), nat.ptr(out), n))
    assert np.array_equal(out, orc.g1_add_affine(A, orc.g1_add_affine(B, B)))
    out[:] = 1
    nat.check(nat.dbg_lib().b200_debug_g1_op(4, nat.ptr(A), nat.ptr(B), nat.ptr(out), n))
    assert not out.any()


def test_device_digit_recoding():
    L = nat.lib()
    rng = random.Random(3)
    xs = [rng.randrange(pyref.R) for _ in range(500)] + [0, 1, pyref.R - 1]
    s = H.fr_array(xs)
    for c in (4, 13, 16, 20):
        W = (255 + c - 1) // c
        out = np.zeros((len(xs), W), np.int32)
        nat.check(nat.dbg_lib().b200_debug_digits(nat.ptr(s), C.c_size_t(len(xs)), C.c_int(c), out.ctypes.data_as(C.c_void_p)))
        for i, x in enumerate(xs):
            assert sum(int(out[i, w]) << (c * w) for w in range(W)) == x


# ---- NTT ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("log_n", [1, 2, 3, 6, 9, 10, 11, 12, 15, 17, 20, 21, 22])
def test_best_fft_vs_oracle(log_n):
    a = orc.gen_scalars(1 << log_n, seed=log_n)
    w = orc.omega(log_n)
    got = h2.best_fft(a, w, log_n)
    assert np.array_equal(got, orc.best_fft(a, log_n, w, THREADS))


def test_fft_batch_and_inverse_roundtrip():
    log_n = 13
    cols = [orc.gen_scalars(1 << log_n, seed=100 + i) for i in range(5)]
    dom = h2.EvaluationDomain(2, log_n)
    coeffs = dom.lagrange_to_coeff_batch(cols)
    for c, v in zip(coeffs, cols):
        assert np.array_equal(c, orc.lagrange_to_coeff(v, log_n, THREADS))
        assert np.array_equal(dom.coeff_to_lagrange(c), v)


def test_pk_fixture_known_answers():
    """The reference's proving-key fixture: values = NTT(polys), cosets = coeff_to_extended(polys) (SURVEY.md App. B)."""
    pk = H.load_pk_fixture()
    dom = h2.EvaluationDomain(9, 6)
    assert dom.extended_k == 9
    cols = [("fixed_values_%d" % c, "fixed_polys_%d" % c, "fixed_cosets_%d" % c) for c in (0, 1, 5, 37)]
    cols.append(("perm_values_0", "perm_polys_0", "perm_cosets_0"))
    for v, p, c in cols:
        assert np.array_equal(dom.coeff_to_lagrange(pk[p]), pk[v])
        assert np.array_equal(dom.lagrange_to_coeff(pk[v]), pk[p])
        assert np.array_equal(dom.coeff_to_extended(pk[p]), pk[c])
        back = dom.extended_to_coeff(pk[c])
        assert back.shape[0] == 64 * 8 and np.array_equal(back[:64], pk[p]) and not back[64:].any()
    outs = dom.coeff_to_extended_batch([pk[p] for _, p, _ in cols])
    for o, (_, _, c) in zip(outs, cols):
        assert np.array_equal(o, pk[c])


@pytest.mark.parametrize("k,j", [(8, 5), (12, 9), (17, 5)])
def test_extended_domain_vs_oracle(k, j):
    dom = h2.EvaluationDomain(j, k)
    a = orc.gen_scalars(1 << k, seed=k)
    ext = dom.coeff_to_extended(a)
    assert np.array_equal(ext, orc.coeff_to_extended(a, dom.extended_k, THREADS))
    assert np.array_equal(dom.divide_by_vanishing_poly(ext), orc.divide_by_vanishing(ext, k, dom.extended_k))
    back = dom.extended_to_coeff(ext)
    assert np.array_equal(back[: 1 << k], a) and not back[1 << k:].any()
    full = orc.gen_scalars(dom.extended_len(), seed=k + 50)
    assert np.array_equal(dom.extended_to_coeff(full), orc.extended_to_coeff(full, dom.extended_k, THREADS)[: (1 << k) * (j - 1)])


def test_fft_full_size_properties():
    """k = 22 (BASELINE configs[4]) and 2^25 (its extended domain): inverse(forward(x)) == x, and linearity."""
    for log_n in (22, 25):
        n = 1 << log_n
        a = orc.gen_scalars(n, seed=7)
        w = orc.omega(log_n)
        fa = h2.best_fft(a, w, log_n)
        w_inv = H.fr_wire(pow(pyref.omega_for(log_n), -1, pyref.R))
        back = h2.best_fft(fa, w_inv, log_n)
        n_inv = H.fr_wire(pow(n, -1, pyref.R))
        assert np.array_equal(h2.poly_op("scale", back, s=n_inv), a)
        if log_n == 22:
            b = orc.gen_scalars(n, seed=8)
            fb = h2.best_fft(b, w, log_n)
            assert np.array_equal(h2.best_fft(h2.poly_op("add", a, b), w, log_n), h2.poly_op("add", fa, fb))
            # spot-check a few outputs against direct evaluation sum_i a_i w^(ij) via the oracle's Horner
            for jdx in (0, 1, 12345, n - 1):
                x = H.fr_wire(pow(pyref.omega_for(log_n), jdx, pyref.R))
                assert np.array_equal(orc.eval_polynomial(a, x), fa[jdx])


# ---- MSM ---------------------------------------------------------------------------------------------------------
def test_srs_fixture_msm_known_answers():
    """64 MSM known answers from the reference's SRS fixture, as ONE batched call: g_lagrange[j] = MSM(n^-1 w^-ij, g)."""
    k, g, gl = H.load_srs_fixture()
    n = 1 << k
    w_inv = pow(pyref.omega_for(k), -1, pyref.R)
    n_inv = pow(n, -1, pyref.R)
    cols = [H.fr_array([pow(w_inv, i * j, pyref.R) * n_inv % pyref.R for i in range(n)]) for j in range(n)]
    for wb in (0, 4, 9):
        bases = h2.Bases(g, window_bits=wb)
        got = h2.best_multiexp_batch(cols, bases)
        assert np.array_equal(jac_to_affine(got), gl), wb
        assert np.array_equal(jac_to_affine(h2.best_multiexp(cols[5], bases))[0], gl[5])
        bases.release()
    params = h2.ParamsKZG.read(H.GOLDEN + "/kzg_k6.srs")
    ones = np.tile(orc.fr_one(), (n, 1))
    assert np.array_equal(jac_to_affine(params.commit_lagrange(ones))[0], g[0])
    assert np.array_equal(jac_to_affine(params.commit(cols[3]))[0], gl[3])


@pytest.mark.parametrize("n,wb", [(1, 0), (2, 4), (33, 5), (1000, 0), (1000, 11), (5000, 16), (1 << 14, 0), (1 << 14, 8)])
def test_msm_vs_oracle(n, wb):
    bases_np = orc.gen_bases(n, seed=n)
    sc = orc.gen_scalars(n, seed=n + 1)
    bases = h2.Bases(bases_np, window_bits=wb)
    assert np.array_equal(jac_to_affine(h2.best_multiexp(sc, bases))[0], orc.msm(sc, bases_np, THREADS))
    bases.release()


def test_msm_degenerate_inputs():
    n = 3000
    bases_np = orc.gen_bases(n, seed=77)
    bases = h2.Bases(bases_np, window_bits=10)
    rng = random.Random(1)
    cols = {
        "zeros": np.zeros((n, 4), np.uint64),
        "ones": np.tile(orc.fr_one(), (n, 1)),                                   # one heavy bucket
        "small": H.fr_array([rng.randrange(1 << 8) for _ in range(n)]),          # ezkl-like quantised witness
        "half_zero": H.fr_array([0 if i % 2 else rng.randrange(pyref.R) for i in range(n)]),
        "r_minus_1": H.fr_array([pyref.R - 1] * n),
        "equal": H.fr_array([0x1234567] * n),
        "two_values": H.fr_array([(1, pyref.R - 5)[i % 2] for i in range(n)]),
    }
    got = h2.best_multiexp_batch(list(cols.values()), bases)
    for (name, sc), g in zip(cols.items(), got):
        assert np.array_equal(jac_to_affine(g)[0], orc.msm(sc, bases_np, THREADS)), name
    assert np.array_equal(got[0], np.array([0] * 4 + list(H.fq_wire(1)) + [0] * 4, np.uint64))   # identity = (0, 1, 0)
    # fewer scalars than registered bases (ParamsKZG::commit slices the bases)
    m = 1234
    assert np.array_equal(jac_to_affine(h2.best_multiexp(cols["small"][:m], bases))[0], orc.msm(cols["small"][:m], bases_np[:m], THREADS))
    bases.release()
    # repeated and identity bases: buckets see P + P and P + identity
    dup = bases_np.copy()
    dup[1::2] = dup[0::2]
    dup[::7] = 0
    b2 = h2.Bases(dup, window_bits=6)
    for name in ("ones", "small", "half_zero"):
        assert np.array_equal(jac_to_affine(h2.best_multiexp(cols[name], b2))[0], orc.msm(cols[name], dup, THREADS)), name
    with pytest.raises(nat.B200Error):
        h2.best_multiexp(np.zeros((n + 1, 4), np.uint64), b2)
    b2.release()


@pytest.mark.parametrize("batch", [1, 2, 8, 9, 20, 21, 36, 37])
def test_msm_reduction_geometry_rows(batch):
    """The bucket reduction picks (buckets per thread, CTA size) from batch x buckets (msm.cu, msm_run): every row of that table, both
    sides of each threshold, with the bench's window (c = 16 -> 2^15 buckets per column) on a base vector small enough for the oracle.
    Scalars mix uniform columns with the skewed ones that leave most buckets empty or one bucket heavy."""
    n = 1 << 11
    bases_np = orc.gen_bases(n, seed=901)
    bases = h2.Bases(bases_np, window_bits=16)
    rng = random.Random(batch)
    cols = []
    for j in range(batch):
        if j % 5 == 3:
            cols.append(H.fr_array([rng.randrange(1 << 10) for _ in range(n)]))
        elif j % 5 == 4:
            cols.append(H.fr_array([pyref.R - 1 - (i % 3) for i in range(n)]))
        else:
            cols.append(orc.gen_scalars(n, seed=1000 * batch + j))
    got = jac_to_affine(h2.best_multiexp_batch(cols, bases))
    for j in sorted(set([0, 3, 4, batch // 2, batch - 1]) & set(range(batch))):
        assert np.array_equal(got[j], orc.msm(cols[j], bases_np, THREADS)), (batch, j)
    bases.release()


def test_msm_k17_and_linearity_k20():
    """k = 17 (BASELINE configs[1]) against the oracle; k = 20 (configs[2]) through linearity + a k=20 oracle run."""
    n = 1 << 17
    bases_np = orc.gen_bases(n, seed=17)
    sc = orc.gen_scalars(n, seed=18)
    bases = h2.Bases(bases_np)
    assert np.array_equal(jac_to_affine(h2.best_multiexp(sc, bases))[0], orc.msm(sc, bases_np, THREADS))
    bases.release()
    n = 1 << 20
    bases_np = orc.gen_bases(n, seed=20)
    a, b = orc.gen_scalars(n, seed=21), orc.gen_scalars(n, seed=22)
    bases = h2.Bases(bases_np)
    ab = h2.poly_op("add", a, b)
    got = jac_to_affine(h2.best_multiexp_batch([a, b, ab], bases))
    assert np.array_equal(orc.g1_add_affine(got[0:1], got[1:2])[0], got[2])
    assert np.array_equal(got[0], orc.msm(a, bases_np, THREADS))
    bases.release()


# ---- polynomial ops ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 7, 4096, 4097, 100000, 1 << 17, (1 << 19) + 3])      # the last moves through the 16 MiB bounce chunks
def test_poly_ops_vs_oracle(n):
    a, b = orc.gen_scalars(n, seed=n), orc.gen_scalars(n, seed=n + 1)
    s = orc.gen_scalars(1, seed=n + 2)[0]
    for op in ("add", "sub", "mul"):
        assert np.array_equal(h2.poly_op(op, a, b), orc.poly_op(op, a, b, threads=THREADS)), op
    assert np.array_equal(h2.poly_op("scale", a, s=s), orc.poly_op("scale", a, s=s, threads=THREADS))
    assert np.array_equal(h2.poly_op("axpy", a, b, s), orc.poly_op("axpy", a, b, s, threads=THREADS))
    assert np.array_equal(h2.eval_polynomial(a, s), orc.eval_polynomial(a, s))
    if n > 1:
        assert np.array_equal(h2.kate_division(a, s), orc.kate_division(a, s))
        assert np.array_equal(h2.kate_division(a, np.zeros(4, np.uint64)), orc.kate_division(a, np.zeros(4, np.uint64)))
    z = a.copy()
    z[::5] = 0
    assert np.array_equal(h2.batch_invert(z), orc.batch_invert(z))
    one = orc.fr_one()
    assert np.array_equal(h2.prefix_scan(a, one, True), orc.prefix_scan(a, one, True))
    assert np.array_equal(h2.prefix_scan(a, s, False), orc.prefix_scan(a, s, False))


def test_eval_batch():
    n = 1 << 12
    polys = [orc.gen_scalars(n, seed=i) for i in range(9)]
    xs = orc.gen_scalars(9, seed=99)
    got = h2.eval_polynomial_batch(polys, xs)
    for p, x, g in zip(polys, xs, got):
        assert np.array_equal(g, orc.eval_polynomial(p, x))


def test_error_behaviour():
    with pytest.raises(nat.B200Error):
        h2.best_fft(np.zeros((8, 4), np.uint64), orc.omega(4), 4)          # len != 2^log_n
    L = nat.lib()
    a = np.zeros((2, 4), np.uint64)
    assert L.b200_fft(nat.ptr(a), C.c_uint32(29), nat.ptr(orc.omega(1))) == -1
    out = np.zeros(12, np.uint64)
    assert L.b200_msm(C.c_uint64(987654), nat.ptr(a), C.c_size_t(2), nat.ptr(out)) == -1
    assert b"unknown bases handle" in L.b200_last_error()


def test_cpp_host_mirror():
    """include/ezkl_b200_halo2.hpp (C++ mirror of EvaluationDomain / ParamsKZG) against the reference's SRS fixture."""
    import os
    import subprocess
    exe = os.path.join(H.ROOT, "tests", "cpp", "test_mirror")
    if not os.path.exists(exe):
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(H.ROOT, "include"), "-o", exe, os.path.join(H.ROOT, "tests", "cpp", "test_mirror.cpp"),
                               "-L" + os.path.join(H.ROOT, "ezkl_b200"), "-lezkl_b200", "-Wl,-rpath," + os.path.join(H.ROOT, "ezkl_b200")])
    r = subprocess.run([exe, os.path.join(H.GOLDEN, "kzg_k6.srs")], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip().endswith("OK"), r.stdout + r.stderr


def test_sharding_layer_single_rank_device_paths():
    """world = 1 degenerate run of the multi-GPU layer on one GPU: the device implementations behind ShardedMsm /
    ShardedNtt (msm_batch -> g1_sum -> normalize; transposed batched NTTs + twiddle matrix) against the oracle."""
    import torch
    from ezkl_b200 import device as dev
    from ezkl_b200 import parallel as par
    n = 1 << 12
    bases_np = orc.gen_bases(n, seed=31)
    sc = np.stack([orc.gen_scalars(n, seed=32), orc.gen_scalars(n, seed=33)])
    sm = par.ShardedMsm(dev.from_host(bases_np), n)
    got = sm(dev.from_host(sc))
    for i in range(2):
        assert np.array_equal(jac_to_affine(got[i])[0], orc.msm(sc[i], bases_np, THREADS))
    # g1_sum of several partials: split the MSM in 4 slices by hand and add
    parts = []
    for lo in range(0, n, n // 4):
        b = dev.DeviceBases(dev.from_host(bases_np[lo:lo + n // 4]))
        parts.append(dev.msm_batch(b, dev.from_host(sc[:, lo:lo + n // 4])))
    summed = dev.g1_sum(torch.stack(parts, dim=1).contiguous())
    assert np.array_equal(dev.normalize(summed), got)
    for k in (9, 14):
        a = orc.gen_scalars(1 << k, seed=k)
        s = par.ShardedNtt(k, pyref.omega_for(k))
        out = s.gather(s.forward(s.scatter(dev.from_host(a))))
        assert np.array_equal(dev.to_host(out), orc.best_fft(a, k, orc.omega(k), THREADS))


def test_reentrancy_from_threads():
    """halo2 commits / transforms columns from Rayon worker threads: every entry point must be re-entrant (each calling thread
    gets its own stream + scratch).  Four Python threads hammer MSM / NTT / eval concurrently; results must stay exact."""
    import threading
    n, k = 1 << 12, 12
    bases_np = orc.gen_bases(n, seed=55)
    bases = h2.Bases(bases_np)
    cols = [orc.gen_scalars(n, seed=60 + i) for i in range(4)]
    exp_msm = [orc.msm(c, bases_np, THREADS) for c in cols]
    exp_ntt = [orc.best_fft(c, k, orc.omega(k), THREADS) for c in cols]
    x = orc.gen_scalars(1, seed=70)[0]
    exp_eval = [orc.eval_polynomial(c, x) for c in cols]
    errs = []

    def worker(i):
        try:
            for _ in range(6):
                assert np.array_equal(jac_to_affine(h2.best_multiexp(cols[i], bases))[0], exp_msm[i])
                assert np.array_equal(h2.best_fft(cols[i], orc.omega(k), k), exp_ntt[i])
                assert np.array_equal(h2.eval_polynomial(cols[i], x), exp_eval[i])
        except Exception as e:      # noqa: BLE001
            errs.append((i, repr(e)))

    ts = [threading.Thread(target=worker, args=(i,)) for i in range(4)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    bases.release()
    assert not errs, errs


def test_empty_and_tiny_inputs():
    L = nat.lib()
    bases_np = orc.gen_bases(8, seed=5)
    bases = h2.Bases(bases_np)
    out = np.zeros(12, np.uint64)
    nat.check(L.b200_msm(C.c_uint64(bases.handle), nat.ptr(np.zeros((1, 4), np.uint64)), C.c_size_t(0), nat.ptr(out)))     # n = 0 -> identity
    assert np.array_equal(out, np.array([0] * 4 + list(H.fq_wire(1)) + [0] * 4, np.uint64))
    assert L.b200_msm_batch(C.c_uint64(bases.handle), None, C.c_size_t(8), C.c_size_t(0), nat.ptr(out)) == -1      # NULL columns, even for batch 0
    assert h2.best_multiexp_batch([], bases).shape == (0, 12)
    one = orc.gen_scalars(1, seed=1)
    assert np.array_equal(jac_to_affine(h2.best_multiexp(one, bases))[0], orc.msm(one, bases_np[:1], 1))
    bases.release()
    a = orc.gen_scalars(2, seed=2)
    assert np.array_equal(h2.best_fft(a, orc.omega(1), 1), orc.best_fft(a, 1, orc.omega(1)))
    assert np.array_equal(h2.eval_polynomial(np.zeros((0, 4), np.uint64), one[0]), np.zeros(4, np.uint64))
    assert h2.kate_division(one, one[0]).shape == (0, 4)
    assert h2.poly_op("add", np.zeros((0, 4), np.uint64), np.zeros((0, 4), np.uint64)).shape == (0, 4)


def test_msm_k22_vs_oracle():
    """k = 22 (BASELINE configs[4]) MSM against the oracle's best_multiexp (all host cores)."""
    n = 1 << 22
    bases_np = orc.gen_bases(n, seed=22)
    sc = orc.gen_scalars(n, seed=23)
    bases = h2.Bases(bases_np)
    assert np.array_equal(jac_to_affine(h2.best_multiexp(sc, bases))[0], orc.msm(sc, bases_np, THREADS))
    bases.release()


def test_keygen_pk_reproduces_reference_proving_key_bytes(tmp_path):
    """create_keys (src/pfsys/mod.rs:376-400): from the fixture's fixed_values / permutations alone, the device keygen
    transforms must reproduce the reference pk.key's derived vectors byte for byte (polys, extended cosets, l0, l_last,
    l_active_row), for the columns carried in tests/golden/pk_k6_subset.npz."""
    pk = H.load_pk_fixture()
    key = h2.ProvingKey()
    key.k = 6
    cols = (0, 1, 5, 37)
    key.fixed_values = [pk["fixed_values_%d" % c] for c in cols]
    key.permutations = [pk["perm_values_0"]]
    out = key.keygen_pk_polys(9, 5)
    for i, c in enumerate(cols):
        assert np.array_equal(out["fixed_polys"][i], pk["fixed_polys_%d" % c])
        assert np.array_equal(out["fixed_cosets"][i], pk["fixed_cosets_%d" % c])
    assert np.array_equal(out["permutation_polys"][0], pk["perm_polys_0"])
    assert np.array_equal(out["permutation_cosets"][0], pk["perm_cosets_0"])
    assert np.array_equal(out["l0"], pk["l0"])
    assert np.array_equal(out["l_last"], pk["l_last"])
    assert np.array_equal(out["l_active_row"], pk["l_active_row"])


def test_poly_lincomb_vs_oracle():
    n = 5000
    polys = [orc.gen_scalars(n, seed=200 + i) for i in range(7)]
    sc = orc.gen_scalars(7, seed=300)
    exp = np.zeros((n, 4), np.uint64)
    for p, s_ in zip(polys, sc):
        exp = orc.poly_op("axpy", exp, p, s_)
    assert np.array_equal(h2.poly_lincomb(polys, sc), exp)


def test_msm_randomised_shapes_and_distributions():
    """Fuzz-style sweep: window bits 4..18, ragged n, small batches, and the scalar distributions ezkl produces
    (uniform, tiny quantised values, sparse, one dominant value => one giant bucket) — all against the oracle."""
    rng = random.Random(2024)
    for case in range(36):
        n = rng.choice([1, 2, 3, 31, 32, 33, 100, 257, 1000, 2048, 4099])
        c = rng.choice([0, 4, 5, 7, 9, 12, 15, 18])
        batch = rng.choice([1, 2, 5])
        bases_np = orc.gen_bases(n, seed=1000 + case)
        if case % 5 == 0 and n > 3:
            bases_np[rng.randrange(n)] = 0                       # an identity base
            bases_np[1] = bases_np[0]                            # a repeated base
        cols = []
        for b in range(batch):
            kind = rng.choice(["uniform", "small", "sparse", "dominant", "boundary"])
            if kind == "uniform":
                xs = [rng.randrange(pyref.R) for _ in range(n)]
            elif kind == "small":
                xs = [rng.randrange(1 << rng.choice([1, 8, 20])) for _ in range(n)]
            elif kind == "sparse":
                xs = [rng.randrange(pyref.R) if rng.random() < 0.1 else 0 for _ in range(n)]
            elif kind == "dominant":
                v = rng.randrange(pyref.R)
                xs = [v if rng.random() < 0.9 else rng.randrange(pyref.R) for _ in range(n)]
            else:
                xs = [rng.choice([pyref.R - 1, pyref.R - 2, 1 << 253, (1 << 128) - 1, 1]) for _ in range(n)]
            cols.append(H.fr_array(xs))
        bases = h2.Bases(bases_np, window_bits=c)
        got = jac_to_affine(h2.best_multiexp_batch(cols, bases))
        for b in range(batch):
            assert np.array_equal(got[b], orc.msm(cols[b], bases_np, THREADS)), (case, n, c, b)
        bases.release()


def test_kzg_open_identity_with_known_trapdoor():
    """End-to-end composition of the GPU primitives as a KZG opening: with an SRS g[i] = s^i * G whose trapdoor s we know,
    commit(p) - p(x) * G == (s - x) * commit(q) for q = kate_division(p, x) — checked with the oracle's group law, no pairing."""
    rng = random.Random(77)
    k = 9
    n = 1 << k
    s = rng.randrange(pyref.R)
    G = np.array(list(H.fq_wire(1)) + list(H.fq_wire(2)), np.uint64)
    powers, cur = [], 1
    for _ in range(n):
        powers.append(cur)
        cur = cur * s % pyref.R
    g = orc.g1_scalar_mul(np.tile(G, (n, 1)), H.fr_array(powers))
    bases = h2.Bases(g)
    p = orc.gen_scalars(n, seed=5)
    x = rng.randrange(pyref.R)
    xv = H.fr_wire(x)
    q = h2.kate_division(p, xv)
    px = H.fr_unwire(h2.eval_polynomial(p, xv))
    cp = jac_to_affine(h2.best_multiexp(p, bases))
    cq = jac_to_affine(h2.best_multiexp(q, bases))
    lhs = orc.g1_add_affine(cp, orc.g1_scalar_mul(G.reshape(1, 8), H.fr_array([(-px) % pyref.R])))
    rhs = orc.g1_scalar_mul(cq, H.fr_array([(s - x) % pyref.R]))
    assert np.array_equal(lhs, rhs)
    bases.release()


def test_gen_srs_and_commit_consistency():
    """gen_srs (src/pfsys/srs.rs:14-16) on the device with a known trapdoor s: g[i] = [s^i]G and g_lagrange[i] = [L_i(s)]G against
    the oracle's scalar multiplication, the fixture relation g_lagrange = n^-1 sum w^-ij g[i], and the identity that ties MSM
    and NTT together: commit_lagrange(values) == commit(lagrange_to_coeff(values)) == [p(s)]G."""
    rng = random.Random(31)
    k = 7
    n = 1 << k
    s = rng.randrange(2, pyref.R)
    params = h2.ParamsKZG.setup(k, s)
    G = np.array(list(H.fq_wire(1)) + list(H.fq_wire(2)), np.uint64)
    pw, cur = [], 1
    for _ in range(n):
        pw.append(cur)
        cur = cur * s % pyref.R
    assert np.array_equal(params.g, orc.g1_scalar_mul(np.tile(G, (n, 1)), H.fr_array(pw)))
    w = pyref.omega_for(k)
    lag = [pow(w, i, pyref.R) * (pow(s, n, pyref.R) - 1) * pow(n * (s - pow(w, i, pyref.R)), -1, pyref.R) % pyref.R for i in range(n)]
    assert np.array_equal(params.g_lagrange, orc.g1_scalar_mul(np.tile(G, (n, 1)), H.fr_array(lag)))
    vals = orc.gen_scalars(n, seed=9)
    dom = h2.EvaluationDomain(2, k)
    coeffs = dom.lagrange_to_coeff(vals)
    c1 = jac_to_affine(params.commit_lagrange(vals))[0]
    c2 = jac_to_affine(params.commit(coeffs))[0]
    ps = H.fr_unwire(h2.eval_polynomial(coeffs, H.fr_wire(s)))
    assert np.array_equal(c1, c2) and np.array_equal(c1, orc.g1_scalar_mul(G.reshape(1, 8), H.fr_array([ps]))[0])


def test_g_to_lagrange_reproduces_the_reference_srs_and_downsize():
    """The reference's own SRS fixture is a known answer for the group FFT: g_lagrange == g_to_lagrange(g) (k = 6).  Then
    ParamsKZG::downsize (src/execute.rs:1745-1748) to k = 4 against the defining relation computed with the oracle's MSM."""
    k, g, gl = H.load_srs_fixture()
    assert np.array_equal(h2.g_to_lagrange(g, k), gl)
    params = h2.ParamsKZG.read(H.GOLDEN + "/kzg_k6.srs")
    params.downsize(4)
    n = 16
    assert params.k == 4 and params.g.shape == (n, 8) and np.array_equal(params.g, g[:n])
    w_inv = pow(pyref.omega_for(4), -1, pyref.R)
    n_inv = pow(n, -1, pyref.R)
    for j in range(n):
        sc = H.fr_array([pow(w_inv, i * j, pyref.R) * n_inv % pyref.R for i in range(n)])
        assert np.array_equal(params.g_lagrange[j], orc.msm(sc, g[:n], 2)), j
    vals = orc.gen_scalars(n, seed=3)
    dom = h2.EvaluationDomain(2, 4)
    assert np.array_equal(params.commit_lagrange(vals), params.commit(dom.lagrange_to_coeff(vals)))
    # a larger transform against the trapdoor SRS: g_to_lagrange([s^i]G) == [L_i(s)]G
    p2 = h2.ParamsKZG.setup(9, 0x1234567)
    assert np.array_equal(h2.g_to_lagrange(p2.g, 9), p2.g_lagrange)


def test_batch_splitting_paths():
    """The host-buffer MSM / NTT entry points split large batches to bound device scratch; force that path with a 1 MB budget."""
    import os
    import subprocess
    import sys
    env = dict(os.environ, B200_WS_BUDGET_MB="1")
    r = subprocess.run([sys.executable, os.path.join(H.ROOT, "tests", "split_paths_check.py")], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0 and "split paths OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
