"""evaluate_h one coset part of the extended domain at a time (include/ezkl_b200_parts.h).

CPU tier: the ABI guard of the new entries, and the algorithm itself on the oracle (part transforms, per-part evaluation, the
vanishing factor per part, interleaving).  GPU tier: the part transforms against coeff_to_extended, evaluate_h_parts against
evaluate_h_from_polys byte for byte, the proof mirror through the parts path, and a k = 23 system whose full cosets could not be held."""
import json
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from ezkl_b200 import _native as nat
from ezkl_b200 import evaluation as ev
from ezkl_b200 import fields as F
from oracle import oracle as orc
from tests import helpers as H
from tests.test_cabi_guard import _PROBE

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = F.FR_MODULUS
PARTS_ENTRIES = ("b200_coeff_to_extended_part_batch", "b200_coeff_to_extended_part_dev", "b200_evaluate_h_parts", "b200_evaluate_h_parts_dev")


def test_parts_entries_check_their_guard_before_cuda():
    r = subprocess.run([sys.executable, "-c", _PROBE, nat.LIB_PATH, os.path.join(ROOT, "include", "ezkl_b200_parts.h"), ""],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    got = json.loads(r.stdout.strip().splitlines()[-1])
    assert set(got) == set(PARTS_ENTRIES)
    for name, res in got.items():
        for (rc, err), how in zip(res, ("real buffers", "NULL pointers")):
            assert rc == -3 and "not initialised" in err, "%s with %s returned %r (%s)" % (name, how, rc, err)
    lib = nat.lib()
    for name in PARTS_ENTRIES:
        assert hasattr(lib, name), name


# ---- the algorithm on the oracle -----------------------------------------------------------------------------------------------------
def part_base(k: int, ext_k: int, r: int) -> int:
    """c_r = zeta * ext_omega^r: part r of the extended domain is {c_r * omega^t : t < 2^k}."""
    ext_omega = pow(F.FR_ROOT_OF_UNITY, 1 << (F.FR_S - ext_k), R)
    return F.FR_ZETA * pow(ext_omega, r, R) % R


def oracle_part(coeffs, k: int, ext_k: int, r: int) -> np.ndarray:
    """Values of the polynomial on part r: one size-2^k transform of p_i * c_r^i (zero padded to 2^k)."""
    n = 1 << k
    p = np.zeros((n, 4), np.uint64)
    p[: coeffs.shape[0]] = coeffs
    powers = orc.prefix_scan(np.tile(H.fr_wire(part_base(k, ext_k, r)), (n, 1)), orc.fr_one(), True)      # c^i
    return orc.best_fft(orc.field_op("fr", "mul", p, powers), k, orc.omega(k))


def t_evaluations(k: int, ext_k: int) -> list:
    """1 / (c_r^n - 1) for every part r, as EvaluationDomain stores them."""
    return [pow((pow(part_base(k, ext_k, r), 1 << k, R) - 1) % R, -1, R) for r in range(1 << (ext_k - k))]


def random_program(rng, ncols: int, max_rot: int, terms: int = 6) -> ev.QuotientProgram:
    """A random folded program: products and sums of queries at rotations of both signs (some beyond d), constants, negations."""
    def leaf():
        if rng.random() < 0.2:
            return ev.Constant(rng.randrange(R))
        return ev.Query(rng.randrange(ncols), rng.randint(-max_rot, max_rot))

    def node(depth):
        if depth == 0:
            return leaf()
        a, b = node(depth - 1), node(depth - 1)
        return rng.choice([lambda: a + b, lambda: a - b, lambda: a * b, lambda: -a * b])()

    return ev.QuotientProgram(ev.fold_y([node(rng.randint(1, 3)) for _ in range(terms)], rng.randrange(R)))


@pytest.mark.parametrize("k", [4, 5, 6])
def test_parts_compose_to_the_full_quotient_on_the_oracle(k):
    rng = random.Random(900 + k)
    n = 1 << k
    for log_d in (0, 1, 2, 3):
        ext_k, d = k + log_d, 1 << log_d
        N = 1 << ext_k
        # coefficient columns of two lengths, and two columns already on the extended domain
        coeff_cols = [orc.gen_scalars(n, seed=rng.randrange(1 << 30)) for _ in range(3)] + [orc.gen_scalars(n - 3, seed=rng.randrange(1 << 30))]
        ext_cols = [orc.gen_scalars(N, seed=rng.randrange(1 << 30)) for _ in range(2)]
        full = [orc.coeff_to_extended(c, ext_k) for c in coeff_cols] + ext_cols
        for c in coeff_cols:
            for r in range(d):
                assert np.array_equal(orc.coeff_to_extended(c, ext_k)[r::d], oracle_part(c, k, ext_k, r)), (k, d, r)
        prog = random_program(rng, len(full), 2 * d + 1)
        loads, consts, instrs = prog.arrays()
        num = orc.quotient_eval(full, k, ext_k, loads, consts, instrs)
        want = orc.extended_to_coeff(orc.divide_by_vanishing(num, k, ext_k), ext_k)
        t_ev = t_evaluations(k, ext_k)
        inter = np.zeros((N, 4), np.uint64)
        for r in range(d):
            part_cols = [oracle_part(c, k, ext_k, r) for c in coeff_cols] + [np.ascontiguousarray(c[r::d]) for c in ext_cols]
            part_num = orc.quotient_eval(part_cols, k, k, loads, consts, instrs)                  # a self-contained size-n evaluate_h
            assert np.array_equal(part_num, num[r::d]), (k, d, r)
            inter[r::d] = orc.poly_op("scale", part_num, s=H.fr_wire(t_ev[r]))
        assert np.array_equal(orc.extended_to_coeff(inter, ext_k), want), (k, d)


# ---- GPU tier ---------------------------------------------------------------------------------------------------------------------------
def _domain(k: int, log_d: int):
    from ezkl_b200 import halo2 as h2
    dom = h2.EvaluationDomain((1 << log_d) + 1, k)
    assert dom.extended_k == k + log_d
    return dom


@pytest.mark.gpu
def test_coeff_to_extended_part_equals_the_strided_coset():
    import torch
    from ezkl_b200 import device as dev
    nat.init(-1)
    rng = random.Random(31)
    for k, log_d in [(3, 0), (5, 1), (6, 2), (7, 3), (5, 4), (12, 3), (14, 4), (17, 2), (20, 3)]:
        dom = _domain(k, log_d)
        n, d = 1 << k, 1 << log_d
        for n_coeffs in (n, n // 2 + 3, 1):
            polys = [orc.gen_scalars(n_coeffs, seed=rng.randrange(1 << 30)) for _ in range(2)]
            padded = [np.concatenate([p, np.zeros((n - n_coeffs, 4), np.uint64)]) for p in polys]
            fulls = dom.coeff_to_extended_batch(padded)
            parts = range(d) if k <= 14 else sorted({0, d - 1, rng.randrange(d)})
            src = torch.stack([dev.from_host(p) for p in polys])
            for r in parts:
                got = dom.coeff_to_extended_part_batch(polys, r)
                for g, f in zip(got, fulls):
                    assert np.array_equal(g, f[r::d]), (k, d, n_coeffs, r)
                got_dev = dev.to_host(dev.coeff_to_extended_part(src, dom, r)).reshape(2, n, 4)
                for g, f in zip(got_dev, fulls):
                    assert np.array_equal(g, f[r::d]), ("dev", k, d, n_coeffs, r)
    with pytest.raises(nat.B200Error):
        _domain(4, 2).coeff_to_extended_part(orc.gen_scalars(17), 0)          # more than n coefficients
    with pytest.raises(nat.B200Error):
        _domain(4, 2).coeff_to_extended_part(orc.gen_scalars(16), 4)          # part >= d


@pytest.mark.gpu
def test_coeff_to_extended_part_reproduces_the_reference_key():
    """The reference's own pk.key (k = 6, extended 2^9): part r of every stored coset is the part transform of the stored coefficients."""
    nat.init(-1)
    sub = dict(np.load(os.path.join(ROOT, "tests", "golden", "pk_k6_subset.npz")))
    dom = _domain(6, 3)
    names = sorted(k_[len("fixed_polys_"):] for k_ in sub if k_.startswith("fixed_polys_"))
    polys = [sub["fixed_polys_" + i] for i in names] + [sub["perm_polys_0"]]
    cosets = [sub["fixed_cosets_" + i] for i in names] + [sub["perm_cosets_0"]]
    l0_coeff, _, _ = dom.keygen_l_coeffs(5)
    for r in range(8):
        for g, c in zip(dom.coeff_to_extended_part_batch(polys, r), cosets):
            assert np.array_equal(g, c[r::8]), r
        assert np.array_equal(dom.coeff_to_extended_part(l0_coeff, r), sub["l0"][r::8]), r


def _device_equals_host(prog, cols, dom, finish, want):
    import torch
    from ezkl_b200 import device as dev
    tens = [dev.from_host(c) for c in cols]
    got = ev.evaluate_h_parts_device(prog, tens, dom, finish=finish)
    torch.cuda.synchronize()
    assert np.array_equal(dev.to_host(got).reshape(-1, 4), want)


@pytest.mark.gpu
def test_evaluate_h_parts_equals_evaluate_h_on_mixed_columns():
    nat.init(-1)
    rng = random.Random(4242)
    for k, log_d in [(4, 0), (5, 1), (6, 3), (8, 2), (10, 4), (12, 3)]:
        dom = _domain(k, log_d)
        n, N, d = 1 << k, 1 << (k + log_d), 1 << log_d
        cols = [orc.gen_scalars(n, seed=rng.randrange(1 << 30)) for _ in range(3)]
        cols += [orc.gen_scalars(max(1, n // 2 - 1), seed=rng.randrange(1 << 30)) for _ in range(2)]
        cols.insert(2, orc.gen_scalars(N, seed=rng.randrange(1 << 30)))
        cols.append(orc.gen_scalars(N, seed=rng.randrange(1 << 30)))
        rng.shuffle(cols)
        prog = random_program(rng, len(cols), 2 * d + 3, terms=8)
        for finish in (False, True):
            want = ev.evaluate_h_from_polys(prog, cols, dom, finish=finish)
            got = ev.evaluate_h_parts(prog, cols, dom, finish=finish)
            assert np.array_equal(got, want), (k, d, finish)
            _device_equals_host(prog, cols, dom, finish, want)
    # lengths between 2^k and 2^ext_k are neither form; a period that does not divide d is rejected
    dom = _domain(5, 2)
    prog = ev.QuotientProgram(ev.Query(0) * ev.Query(0, 1))
    with pytest.raises(nat.B200Error):
        ev.evaluate_h_parts(prog, [orc.gen_scalars(33)], dom)
    dom.t_evaluations = np.concatenate([dom.t_evaluations, dom.t_evaluations[:1]])
    with pytest.raises(nat.B200Error):
        ev.evaluate_h_parts(prog, [orc.gen_scalars(32)], dom, finish=True)


def gate_group_program(m: int) -> ev.QuotientProgram:
    """bench.py's quotient group: m coset columns and the running sum h (column m), h <- h * y + (a * b + c * a - b) with a, b, c
    read at rotations 0, +1, -1."""
    value = ev.Query(m)
    y = ev.Constant(0x1234567890ABCDEF1234567890ABCDEF)
    for t in range(m):
        a, b, c = ev.Query(t), ev.Query((t + 1) % m, 1), ev.Query((t + 2) % m, -1)
        value = value * y + (a * b + c * a - b)
    return ev.QuotientProgram(value)


@pytest.mark.gpu
def test_evaluate_h_parts_on_the_bench_group_and_the_ezkl_shaped_system():
    from tests import test_constraint_system as tcs
    nat.init(-1)
    # the bench's 33-column group at k = 17 (2^20 extended rows): 32 coefficient columns and the carried partial sum h
    k = 17
    dom = _domain(k, 3)
    cols = [orc.gen_scalars(1 << k, seed=100 + i) for i in range(32)] + [orc.gen_scalars(1 << 20, seed=99)]
    prog = gate_group_program(32)
    for finish in (False, True):
        want = ev.evaluate_h_from_polys(prog, cols, dom, finish=finish)
        assert np.array_equal(ev.evaluate_h_parts(prog, cols, dom, finish=finish), want), finish
        _device_equals_host(prog, cols, dom, finish, want)
    # the ezkl-shaped system (gates, two-chunk permutation, mv-lookup): the l-polynomials as cosets, then every column in coefficient form
    k = 7
    n = 1 << k
    dom = _domain(k, 2)
    rng = random.Random(7)
    beta, gamma, y = (rng.randrange(R) for _ in range(3))
    lookup_in = ev.Query(tcs.SEL_L) * ev.Query(tcs.A1) + (ev.Constant(1) - ev.Query(tcs.SEL_L)) * ev.Constant(rng.randrange(R))
    perm_cols = [tcs.A0, tcs.A1, tcs.B0, tcs.B1, tcs.OUT]
    terms = ev.base_op_gates(tcs.SEL, [tcs.A0, tcs.A1], [tcs.B0, tcs.B1], tcs.OUT) + \
        ev.permutation_terms(perm_cols, tcs.SIG, tcs.Z, tcs.L0, tcs.LLAST, tcs.LACT, tcs.XCOL, beta, gamma, tcs.CHUNK, tcs.BLIND) + \
        ev.mv_lookup_terms([lookup_in], ev.Query(tcs.TABLE), tcs.M, tcs.PHI, tcs.L0, tcs.LLAST, tcs.LACT, beta)
    prog = ev.QuotientProgram(ev.fold_y(terms, y))
    cols = [orc.gen_scalars(n, seed=500 + i) for i in range(tcs.NCOLS)]
    l_cos = dom.keygen_l_polys(tcs.BLIND)
    l_coeff = dom.keygen_l_coeffs(tcs.BLIND)
    for c, cos in zip(l_coeff, l_cos):
        assert np.array_equal(dom.coeff_to_extended(c), cos)
    with_cosets = list(cols)
    with_cosets[tcs.L0], with_cosets[tcs.LLAST], with_cosets[tcs.LACT] = l_cos
    coeff_only = list(cols)
    coeff_only[tcs.L0], coeff_only[tcs.LLAST], coeff_only[tcs.LACT] = l_coeff
    for finish in (False, True):
        want = ev.evaluate_h_from_polys(prog, with_cosets, dom, finish=finish)
        assert np.array_equal(ev.evaluate_h_parts(prog, with_cosets, dom, finish=finish), want), finish
        assert np.array_equal(ev.evaluate_h_parts(prog, coeff_only, dom, finish=finish), want), finish
        _device_equals_host(prog, coeff_only, dom, finish, want)


@pytest.mark.gpu
def test_create_proof_through_the_parts_quotient_reproduces_the_golden_proof():
    from ezkl_b200 import halo2 as h2
    from ezkl_b200 import prover as pv
    from tests import test_prover_mirror as tpm
    nat.init(-1)
    k, s, cs, fixed, sigmas, advice = tpm.golden_case()
    keys = pv.Keys(h2.ParamsKZG.setup(k, s), cs, fixed, sigmas, vk_repr=0x5EED)
    proof = pv.create_proof(keys, advice, rng=pv.ChaCha12Rng(bytes(32)), quotient="parts")
    golden = open(tpm.GOLDEN_PROOF, "rb").read()
    assert len(golden) == 1888 and proof == golden
    with pytest.raises(ValueError):
        pv.create_proof(keys, advice, rng=pv.ChaCha12Rng(bytes(32)), quotient="halves")


@pytest.mark.gpu
def test_quotient_at_k23_beyond_the_full_cosets():
    """k = 23, ext_k = 26, d = 8, 96 coefficient columns: their full cosets would take 96 * 2 GiB = 192 GiB, more than the device holds.
    Columns a, b, c = a * b and e = a rotated by one row, built on the device; the terms c - a * b and e - a(omega X) vanish on the
    domain, so the numerator is h(X) * (X^n - 1) with deg h <= n - 2: checked at a random point from the columns' own evaluations."""
    import torch
    from ezkl_b200 import device as dev
    nat.init(-1)
    k, log_d = 23, 3
    n, N = 1 << k, 1 << (k + log_d)
    dom = _domain(k, log_d)
    quads = 24
    coeffs = torch.empty((4 * quads, n, 4), dtype=torch.int64, device="cuda")
    lag = torch.empty((4, n, 4), dtype=torch.int64, device="cuda")
    tmp = torch.empty((4, n, 4), dtype=torch.int64, device="cuda")
    for q in range(quads):
        lag[:2] = dev.random_scalars(n, batch=2, seed=1000 + q)
        dev.poly_op("mul", lag[0], lag[1], out=lag[2])
        lag[3] = torch.roll(lag[0], -1, dims=0)                          # e[i] = a[i + 1]
        dev.ntt(lag, k, dom.omega_inv, post=[dom.ifft_divisor], out=coeffs[4 * q:4 * q + 4], tmp=tmp)
    del lag, tmp
    rng = random.Random(23)
    terms = []
    for q in range(quads):
        a, b, c, e = (ev.Query(4 * q + j) for j in range(4))
        terms += [c - a * b, e - ev.Query(4 * q, 1)]
    y = rng.randrange(R)
    expr = ev.fold_y(terms, y)
    prog = ev.QuotientProgram(expr)
    cols = [coeffs[i] for i in range(4 * quads)]
    out = ev.evaluate_h_parts_device(prog, cols, dom, finish=True)
    torch.cuda.synchronize()
    assert not out[n - 1:].any().item()                                   # deg h <= n - 2: the other 2^26 - 2^23 + 1 coefficients vanish
    x = rng.randrange(R)
    xw = x * pow(F.fr_from_limbs(dom.omega), 1, R) % R
    at_x = H.fr_list(dev.to_host(dev.eval_batch(coeffs, np.tile(H.fr_wire(x), (4 * quads, 1)))).reshape(-1, 4))
    at_xw = H.fr_list(dev.to_host(dev.eval_batch(coeffs[0::4].contiguous(), np.tile(H.fr_wire(xw), (quads, 1)))).reshape(-1, 4))
    values = {(i, 0): v for i, v in enumerate(at_x)}
    values.update({(4 * q, 1): v for q, v in enumerate(at_xw)})
    numerator = 0
    for t in terms:
        numerator = (numerator * y + _eval(t, values)) % R
    hx = H.fr_list(dev.to_host(dev.eval_batch(out[:n].unsqueeze(0).contiguous(), H.fr_wire(x).reshape(1, 4))).reshape(-1, 4))[0]
    assert numerator == hx * (pow(x, n, R) - 1) % R
    assert numerator != 0


def _eval(e, values):
    if e.kind == "constant":
        return e.args[0]
    if e.kind == "query":
        return values[e.args]
    v = [_eval(a, values) for a in e.args]
    return {"sum": lambda: v[0] + v[1], "sub": lambda: v[0] - v[1], "product": lambda: v[0] * v[1], "negated": lambda: -v[0]}[e.kind]() % R
