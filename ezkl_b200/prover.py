"""Host mirror of `halo2_proofs::plonk::create_proof` as ezkl drives it (/root/reference/src/pfsys/mod.rs:404-489: transcript init
`:435`, deterministic rng under `det-prove` `:436-439`, `create_proof` `:456`, `transcript.finalize()` `:463`; the `Snark` that
carries the bytes `:198-219`), over the C ABI.

Everything polynomial-sized runs on the device through ezkl_b200.halo2 / evaluation / multiopen (commit_lagrange, iNTT, coset
NTT, evaluate_h, grand products and sums, multiplicities, SHPLONK); the Keccak transcript, the rng and the stage sequence stay on
the host, exactly the split the Rust integration has.  Stage order restated from UPSTREAM plonk/prover.rs (SURVEY.md Appendix D4):

  vk repr, instances -> advice (blinded rows, commitments) -> theta -> lookup multiplicities m -> beta, gamma -> permutation
  z_i -> lookup phi -> vanishing random polynomial -> y -> quotient pieces h_i -> x -> evaluations (advice, fixed, random,
  sigmas, z's, phi / m) -> SHPLONK (y', v, h1, u, h2).

Proof bytes: points as x || y and scalars, 32-byte big-endian each (the layout of the reference's tests/assets/proof.json:
commitments, then evaluations, then the two SHPLONK points).  This mirror exists so that "prove time" is measured with the real
stage dependencies and so that the bytes can be diffed against `ezkl prove --features det-prove` the day a Rust toolchain is at
hand; the order of rng draws and the vk transcript representation are restated from recollection and flagged UNPINNED.
`verify_proof_with_trapdoor` replays the verifier (gate identity at x, SHPLONK equation) with the pairing replaced by the known
trapdoor of a test SRS, using the library's own MSM for the group side.
"""
from __future__ import annotations

import numpy as np

from . import evaluation as ev
from . import fields as F
from . import halo2 as h2
from . import multiopen as mo
from .evaluation import Constant, Expression, Query
from .transcript import EvmTranscriptRead, EvmTranscriptWrite

R = F.FR_MODULUS


# ---- rng: rand 0.8 `StdRng` = ChaCha12, as seeded at src/pfsys/mod.rs:437 --------------------------------------------------
class ChaCha12Rng:
    """rand_chacha's ChaCha12Rng: 256-bit key = seed, 64-bit block counter from 0, stream 0, output word by word."""

    def __init__(self, seed: bytes = bytes(32)):
        assert len(seed) == 32
        self.key = [int.from_bytes(seed[4 * i:4 * i + 4], "little") for i in range(8)]
        self.counter, self.words, self.pos = 0, [], 0

    @staticmethod
    def _block(key, counter, rounds=12):
        M = 0xFFFFFFFF
        s = [0x61707865, 0x3320646E, 0x79622D32, 0x6B206574] + key + [counter & M, (counter >> 32) & M, 0, 0]
        x = list(s)

        def qr(a, b, c, d):
            x[a] = (x[a] + x[b]) & M; x[d] ^= x[a]; x[d] = ((x[d] << 16) | (x[d] >> 16)) & M
            x[c] = (x[c] + x[d]) & M; x[b] ^= x[c]; x[b] = ((x[b] << 12) | (x[b] >> 20)) & M
            x[a] = (x[a] + x[b]) & M; x[d] ^= x[a]; x[d] = ((x[d] << 8) | (x[d] >> 24)) & M
            x[c] = (x[c] + x[d]) & M; x[b] ^= x[c]; x[b] = ((x[b] << 7) | (x[b] >> 25)) & M

        for _ in range(rounds // 2):
            qr(0, 4, 8, 12); qr(1, 5, 9, 13); qr(2, 6, 10, 14); qr(3, 7, 11, 15)
            qr(0, 5, 10, 15); qr(1, 6, 11, 12); qr(2, 7, 8, 13); qr(3, 4, 9, 14)
        return [(x[i] + s[i]) & M for i in range(16)]

    def next_u32(self) -> int:
        if self.pos == len(self.words):
            self.words, self.pos = self._block(self.key, self.counter), 0
            self.counter += 1
        v = self.words[self.pos]
        self.pos += 1
        return v

    def next_u64(self) -> int:
        lo = self.next_u32()
        return lo | (self.next_u32() << 32)


def random_fr(rng) -> int:
    """halo2curves `Fr::random`: eight next_u64 limbs read as a 512-bit little-endian integer, reduced modulo r (from_u512)."""
    return sum(rng.next_u64() << (64 * i) for i in range(8)) % R


# ---- constraint system + keys ---------------------------------------------------------------------------------------------------
def expr_degree(e: Expression) -> int:
    if e.kind == "constant":
        return 0
    if e.kind == "query":
        return 1
    d = [expr_degree(a) for a in e.args]
    return sum(d) if e.kind == "product" else max(d)


def expr_queries(e: Expression, out: list):
    """(column, rotation) pairs in first-appearance order."""
    if e.kind == "query":
        if e.args not in out:
            out.append(e.args)
    elif e.kind != "constant":
        for a in e.args:
            expr_queries(a, out)


def expr_eval(e: Expression, value_of) -> int:
    if e.kind == "constant":
        return e.args[0]
    if e.kind == "query":
        return value_of(e.args[0], e.args[1])
    v = [expr_eval(a, value_of) for a in e.args]
    return {"sum": lambda: v[0] + v[1], "sub": lambda: v[0] - v[1], "product": lambda: v[0] * v[1], "negated": lambda: -v[0]}[e.kind]() % R


class ConstraintSystem:
    """What `Circuit::configure` leaves behind, reduced to what the prover reads: columns [advice | fixed] indexed flat, gate
    polynomials, the permutation's columns, mv-lookups as (input expressions, table expression) with single-column (uncompressed)
    inputs and table.  ezkl's own BaseConfig produces exactly these pieces (/root/reference/src/circuit/ops/chip.rs)."""

    def __init__(self, num_advice: int, num_fixed: int, gates, permutation_columns, lookups, blinding_factors: int = 5):
        self.num_advice, self.num_fixed = num_advice, num_fixed
        self.gates, self.permutation_columns, self.lookups = list(gates), list(permutation_columns), list(lookups)
        self.blinding_factors = blinding_factors
        d = max([3] + [expr_degree(g) for g in self.gates] + [2 + expr_degree(t) + sum(expr_degree(f) for f in ins) for ins, t in self.lookups])
        self.degree = d
        self.chunk_len = d - 2
        q = []
        for g in self.gates:
            expr_queries(g, q)
        for ins, t in self.lookups:
            for f in ins:
                expr_queries(f, q)
            expr_queries(t, q)
        for c in self.permutation_columns:
            if (c, 0) not in q:
                q.append((c, 0))
        self.advice_queries = [x for x in q if x[0] < num_advice]
        self.fixed_queries = [x for x in q if x[0] >= num_advice]
        self.num_z = (len(self.permutation_columns) + self.chunk_len - 1) // self.chunk_len if self.permutation_columns else 0

    def column_layout(self):
        """Flat indices of the derived columns evaluate_h sees after [advice | fixed]: sigmas, z's, per lookup (m, phi), l0, l_last, l_active, X."""
        base = self.num_advice + self.num_fixed
        sig = list(range(base, base + len(self.permutation_columns)))
        zs = list(range(sig[-1] + 1 if sig else base, (sig[-1] + 1 if sig else base) + self.num_z))
        nxt = (zs[-1] + 1) if zs else ((sig[-1] + 1) if sig else base)
        lk = [(nxt + 2 * i, nxt + 2 * i + 1) for i in range(len(self.lookups))]
        nxt += 2 * len(self.lookups)
        return {"sigma": sig, "z": zs, "lookup": lk, "l0": nxt, "l_last": nxt + 1, "l_active": nxt + 2, "x": nxt + 3, "count": nxt + 4}

    def numerator(self, beta: int, gamma: int, y: int) -> Expression:
        """The folded quotient numerator in evaluate_h's order: custom gates, permutation, lookups (theta unused: single-column lookups)."""
        L = self.column_layout()
        terms = list(self.gates)
        if self.permutation_columns:
            terms += ev.permutation_terms(self.permutation_columns, L["sigma"], L["z"], L["l0"], L["l_last"], L["l_active"], L["x"], beta, gamma, self.chunk_len,
                                          self.blinding_factors)
        for (ins, t), (m_col, phi_col) in zip(self.lookups, L["lookup"]):
            terms += ev.mv_lookup_terms(ins, t, m_col, phi_col, L["l0"], L["l_last"], L["l_active"], beta)
        return ev.fold_y(terms, y)


class Keys:
    """keygen_vk + keygen_pk for the mirror (/root/reference/src/pfsys/mod.rs:376-400 `create_keys`): fixed and sigma columns in all
    three forms, the l-polynomials' cosets, the commitments the verifier needs."""

    def __init__(self, params: h2.ParamsKZG, cs: ConstraintSystem, fixed_values, sigma_values, vk_repr: int = 0):
        self.params, self.cs = params, cs
        self.domain = h2.EvaluationDomain(cs.degree, params.k)
        n = params.n
        self.fixed_values = [h2._fr(c) for c in fixed_values]
        self.sigma_values = [h2._fr(c) for c in sigma_values]
        assert len(self.fixed_values) == cs.num_fixed and len(self.sigma_values) == len(cs.permutation_columns)
        cols = self.fixed_values + self.sigma_values
        polys = self.domain.lagrange_to_coeff_batch(cols)
        cosets = self.domain.coeff_to_extended_batch(polys)
        nf = cs.num_fixed
        self.fixed_polys, self.sigma_polys = polys[:nf], polys[nf:]
        self.fixed_cosets, self.sigma_cosets = cosets[:nf], cosets[nf:]
        comm = params.commit_lagrange_batch(cols) if cols else np.zeros((0, 12), np.uint64)
        self.fixed_commitments, self.sigma_commitments = comm[:nf], comm[nf:]
        self.l0, self.l_last, self.l_active = self.domain.keygen_l_polys(cs.blinding_factors)
        x_coeff = np.zeros((n, 4), np.uint64)
        x_coeff[1] = F.fr_to_limbs(1)
        self.x_poly = x_coeff
        self.x_coset = self.domain.coeff_to_extended(x_coeff)
        self.vk_repr = vk_repr % R          # UNPINNED: upstream hashes the pinned verifying key (Blake2b of its debug string) into this scalar
        self._l_coeffs = None

    def l_polys(self):
        """(l0, l_last, l_active) in coefficient form, derived on first use: what the per-part quotient reads instead of their cosets."""
        if self._l_coeffs is None:
            self._l_coeffs = self.domain.keygen_l_coeffs(self.cs.blinding_factors)
        return self._l_coeffs


def sigma_labels(k: int, num_columns: int, cycles_next: dict) -> list:
    """Permutation columns in Lagrange form: cell (column j, row i) carries the label DELTA^j * omega^i of its successor in its
    copy-constraint cycle (`cycles_next[(j, i)]`, identity when absent) — halo2 permutation/keygen.rs build_pk."""
    n = 1 << k
    w = pow(F.FR_ROOT_OF_UNITY, 1 << (F.FR_S - k), R)
    wp = [1] * n
    for i in range(1, n):
        wp[i] = wp[i - 1] * w % R
    out = []
    for j in range(num_columns):
        col = np.zeros((n, 4), np.uint64)
        for i in range(n):
            tj, ti = cycles_next.get((j, i), (j, i))
            col[i] = F.fr_to_limbs(pow(ev.DELTA, tj, R) * wp[ti] % R)
        out.append(col)
    return out


def _wire(col_ints) -> np.ndarray:
    return np.stack([F.fr_to_limbs(v) for v in col_ints])


def _ints(col_wire) -> list:
    return [F.fr_from_limbs(r) for r in np.asarray(col_wire).reshape(-1, 4)]


# ---- the prover ---------------------------------------------------------------------------------------------------------------------
def create_proof(keys: Keys, advice, instances=(), rng=None, trace=None, quotient: str = "full") -> bytes:
    """advice: list of num_advice columns (python ints; rows >= n - blinding_factors are overwritten with blinding values).
    Returns the proof bytes (EvmTranscript stream).  `trace`, if a dict, receives the challenges and intermediate columns.
    quotient: "full" evaluates h over the whole extended domain at once (the key's cosets as columns); "parts" evaluates it one
    coset part at a time from coefficient-form columns only (evaluation.evaluate_h_parts): the same bytes, with device memory
    of about one part per column instead of one coset per column."""
    if quotient not in ("full", "parts"):
        raise ValueError("create_proof: quotient must be 'full' or 'parts', not %r" % (quotient,))
    cs, params, dom = keys.cs, keys.params, keys.domain
    n, k, bf = params.n, params.k, cs.blinding_factors
    u = n - bf - 1
    rng = rng or ChaCha12Rng()
    tr = EvmTranscriptWrite()
    L = cs.column_layout()
    # 0. vk, instances
    tr.common_scalar(keys.vk_repr)
    for col in instances:
        for v in col:
            tr.common_scalar(v)
    # 1. advice: blind the last rows, commit (the per-column Blind drawn after the rows is ignored by KZG but still consumes rng)
    adv = [[int(v) % R for v in col] for col in advice]
    assert len(adv) == cs.num_advice and all(len(c) == n for c in adv)
    for col in adv:
        for i in range(n - bf, n):
            col[i] = random_fr(rng)
    for _ in adv:
        random_fr(rng)
    adv_w = [_wire(c) for c in adv]
    for c in params.commit_lagrange_batch(adv_w):
        tr.write_ec_point(c)
    theta = tr.squeeze_challenge()
    # 2. lookups: input / table columns (Lagrange), multiplicities on the device, commit m
    fixed_i = [_ints(c) for c in keys.fixed_values]
    base_cols = adv + fixed_i

    def eval_rows(e):
        return [expr_eval(e, lambda c, rot, i=i: base_cols[c][(i + rot) % n]) for i in range(n)]

    lk = []
    for ins, t in cs.lookups:
        f_cols = [eval_rows(f) for f in ins]
        t_col = eval_rows(t)
        m_w = ev.lookup_multiplicities(_wire(t_col[:u]), [_wire(fc[:u]) for fc in f_cols], u)
        m_col = _ints(m_w) + [random_fr(rng) for _ in range(n - u)]
        lk.append({"f": f_cols, "t": t_col, "m": m_col})
    for c in (params.commit_lagrange_batch([_wire(x["m"]) for x in lk]) if lk else []):
        tr.write_ec_point(c)
    beta = tr.squeeze_challenge()
    gamma = tr.squeeze_challenge()
    # 3. permutation grand products (chunks chained through last_z), then lookup grand sums
    zs_w = []
    if cs.permutation_columns:
        blinds = [[random_fr(rng) for _ in range(bf)] for _ in range(cs.num_z)]
        zs_w = ev.permutation_products([_wire(base_cols[c]) for c in cs.permutation_columns], keys.sigma_values, k, beta, gamma, cs.chunk_len, bf, blinds)
        for c in params.commit_lagrange_batch(zs_w):
            tr.write_ec_point(c)
    phis_w = []
    for x in lk:
        phi = _ints(ev.lookup_grand_sum([_wire(fc) for fc in x["f"]], _wire(x["t"]), _wire(x["m"][:u] + [0] * (n - u)), k, beta))
        if phi[u] != 0:
            raise ValueError("create_proof: a lookup is not satisfied (grand sum does not close)")
        x["phi"] = phi[: u + 1] + [random_fr(rng) for _ in range(n - u - 1)]
        phis_w.append(_wire(x["phi"]))
    for c in (params.commit_lagrange_batch(phis_w) if phis_w else []):
        tr.write_ec_point(c)
    # 4. vanishing argument: a random polynomial of degree < n
    rand_poly = _wire([random_fr(rng) for _ in range(n)])
    random_fr(rng)
    tr.write_ec_point(params.commit(rand_poly))
    y = tr.squeeze_challenge()
    # 5. quotient: coefficients and cosets of every witness-derived column, evaluate_h, divide, split, commit
    derived = adv_w + list(zs_w)
    for x, w_phi in zip(lk, phis_w):
        derived += [_wire(x["m"]), w_phi]
    polys = dom.lagrange_to_coeff_batch(derived)
    na, nz = cs.num_advice, len(zs_w)
    adv_polys, z_polys = polys[:na], polys[na:na + nz]
    lk_polys = [(polys[na + nz + 2 * i], polys[na + nz + 2 * i + 1]) for i in range(len(lk))]
    # evaluate_h at the CPU evaluator's own boundary: witness-derived columns go in coefficient form (the library builds their cosets), the
    # key's cosets and the l-polynomials on the extended domain; one call also divides by the vanishing polynomial and converts back
    columns = [None] * L["count"]
    for i in range(na):
        columns[i] = adv_polys[i]
    for i in range(cs.num_fixed):
        columns[na + i] = keys.fixed_cosets[i]
    for i, c in enumerate(L["sigma"]):
        columns[c] = keys.sigma_cosets[i]
    for i, c in enumerate(L["z"]):
        columns[c] = z_polys[i]
    for i, (mc, pc) in enumerate(L["lookup"]):
        columns[mc], columns[pc] = lk_polys[i]
    columns[L["l0"]], columns[L["l_last"]], columns[L["l_active"]], columns[L["x"]] = keys.l0, keys.l_last, keys.l_active, keys.x_coset
    if quotient == "parts":                # the key's columns in coefficient form too: nothing of 2^ext_k elements reaches the device but the output
        for i in range(cs.num_fixed):
            columns[na + i] = keys.fixed_polys[i]
        for i, c in enumerate(L["sigma"]):
            columns[c] = keys.sigma_polys[i]
        columns[L["l0"]], columns[L["l_last"]], columns[L["l_active"]] = keys.l_polys()
        columns[L["x"]] = keys.x_poly
    prog = ev.QuotientProgram(cs.numerator(beta, gamma, y))
    evaluate = ev.evaluate_h_parts if quotient == "parts" else ev.evaluate_h_from_polys
    h = evaluate(prog, columns, dom, finish=True)[: n * dom.quotient_poly_degree]
    pieces = [np.ascontiguousarray(h[i * n:(i + 1) * n]) for i in range(dom.quotient_poly_degree)]
    for c in params.commit_batch(pieces):
        tr.write_ec_point(c)
    x = tr.squeeze_challenge()
    # 6. evaluations
    w = F.fr_from_limbs(dom.omega)
    rot_pt = lambda rot: x * pow(w, rot, R) % R
    at = lambda poly, pt: F.fr_from_limbs(h2.eval_polynomial(poly, F.fr_to_limbs(pt)))
    adv_evals = [at(adv_polys[c], rot_pt(rot)) for c, rot in cs.advice_queries]
    fix_evals = [at(keys.fixed_polys[c - na], rot_pt(rot)) for c, rot in cs.fixed_queries]
    for v in adv_evals + fix_evals:
        tr.write_scalar(v)
    random_eval = at(rand_poly, x)
    tr.write_scalar(random_eval)
    sigma_evals = [at(p, x) for p in keys.sigma_polys]
    for v in sigma_evals:
        tr.write_scalar(v)
    last_rot = -(bf + 1)
    z_evals = []
    for i, zp in enumerate(z_polys):
        e = [at(zp, x), at(zp, rot_pt(1))] + ([at(zp, rot_pt(last_rot))] if i + 1 < len(z_polys) else [])
        z_evals.append(e)
        for v in e:
            tr.write_scalar(v)
    lk_evals = []
    for m_poly, phi_poly in lk_polys:
        e = [at(phi_poly, x), at(phi_poly, rot_pt(1)), at(m_poly, x)]
        lk_evals.append(e)
        for v in e:
            tr.write_scalar(v)
    # 7. SHPLONK over every opening, in the order the verifier rebuilds them
    xn = pow(x, n, R)
    h_poly = pieces[-1]
    for p in reversed(pieces[:-1]):
        h_poly = h2.poly_op("axpy", p, h_poly, F.fr_to_limbs(xn))          # h(X) = sum_i x^(n i) h_i(X), Horner from the top piece
    queries = [mo.ProverQuery(rot_pt(rot), adv_polys[c]) for c, rot in cs.advice_queries]
    for i, zp in enumerate(z_polys):
        queries += [mo.ProverQuery(x, zp), mo.ProverQuery(rot_pt(1), zp)]
    for i, zp in reversed(list(enumerate(z_polys))[:-1]):
        queries.append(mo.ProverQuery(rot_pt(last_rot), zp))
    for m_poly, phi_poly in lk_polys:
        queries += [mo.ProverQuery(x, phi_poly), mo.ProverQuery(rot_pt(1), phi_poly), mo.ProverQuery(x, m_poly)]
    queries += [mo.ProverQuery(rot_pt(rot), keys.fixed_polys[c - na]) for c, rot in cs.fixed_queries]
    queries += [mo.ProverQuery(x, p) for p in keys.sigma_polys]
    queries += [mo.ProverQuery(x, h_poly), mo.ProverQuery(x, rand_poly)]
    mo.create_proof(params, queries, transcript=tr)
    if trace is not None:
        trace.update({"theta": theta, "beta": beta, "gamma": gamma, "y": y, "x": x, "advice": adv, "lookups": lk, "z": [_ints(z) for z in zs_w],
                      "n_instructions": len(prog.instrs), "n_queries": len(queries)})
    return tr.finalize()


# ---- verifier with the pairing replaced by the trapdoor of a test SRS ------------------------------------------------------------------
def _affine_wire(pt) -> np.ndarray:
    if pt is None:
        return np.zeros(8, np.uint64)
    return np.concatenate([F.fq_to_limbs(pt[0]), F.fq_to_limbs(pt[1])])


def _verifier_accumulate(keys: Keys, proof: bytes, instances=()):
    """VerifierSHPLONK + the PLONK identity check, restated (UPSTREAM plonk/verifier.rs, shplonk/verifier.rs), up to the final pairing:
    returns (acc, h2_pt, u) with acc = {point: scalar} ("G" = the generator) such that the verifier's left input is
    L = sum acc[pt] * pt + u * h2 and its check is e(L, [1]_2) == e(h2, [s]_2); None when the proof is malformed."""
    cs, params, dom = keys.cs, keys.params, keys.domain
    n, bf = params.n, cs.blinding_factors
    na = cs.num_advice
    tr = EvmTranscriptRead(proof)
    tr.common_scalar(keys.vk_repr)
    for col in instances:
        for v in col:
            tr.common_scalar(v)
    try:
        adv_c = [tr.read_ec_point() for _ in range(na)]
        tr.squeeze_challenge()                                        # theta
        m_c = [tr.read_ec_point() for _ in cs.lookups]
        beta, gamma = tr.squeeze_challenge(), tr.squeeze_challenge()
        z_c = [tr.read_ec_point() for _ in range(cs.num_z)]
        phi_c = [tr.read_ec_point() for _ in cs.lookups]
        rand_c = tr.read_ec_point()
        y = tr.squeeze_challenge()
        h_c = [tr.read_ec_point() for _ in range(dom.quotient_poly_degree)]
        x = tr.squeeze_challenge()
        adv_e = [tr.read_scalar() for _ in cs.advice_queries]
        fix_e = [tr.read_scalar() for _ in cs.fixed_queries]
        rand_e = tr.read_scalar()
        sig_e = [tr.read_scalar() for _ in cs.permutation_columns]
        z_e = [[tr.read_scalar() for _ in range(3 if i + 1 < cs.num_z else 2)] for i in range(cs.num_z)]
        lk_e = [[tr.read_scalar() for _ in range(3)] for _ in cs.lookups]
    except ValueError:
        return None
    w = F.fr_from_limbs(dom.omega)
    rot_pt = lambda rot: x * pow(w, rot, R) % R
    last_rot = -(bf + 1)
    u_row = n - bf - 1
    xn = pow(x, n, R)
    # l_0(x), l_last(x), l_blind(x) from the Lagrange basis at x
    lag = lambda row: (xn - 1) * pow(w, row, R) % R * pow(n * (x - pow(w, row, R)) % R, -1, R) % R
    l0_x, l_last_x = lag(0), lag(u_row)
    l_active_x = (1 - l_last_x - sum(lag(i) for i in range(u_row + 1, n))) % R
    L = cs.column_layout()
    table = {}
    for (c, rot), v in zip(cs.advice_queries, adv_e):
        table[(c, rot)] = v
    for (c, rot), v in zip(cs.fixed_queries, fix_e):
        table[(c, rot)] = v
    for i, c in enumerate(L["sigma"]):
        table[(c, 0)] = sig_e[i]
    for i, c in enumerate(L["z"]):
        table[(c, 0)], table[(c, 1)] = z_e[i][0], z_e[i][1]
        if i + 1 < cs.num_z:
            table[(c, last_rot)] = z_e[i][2]
    for (mc, pc), e in zip(L["lookup"], lk_e):
        table[(pc, 0)], table[(pc, 1)], table[(mc, 0)] = e
    table[(L["l0"], 0)], table[(L["l_last"], 0)], table[(L["l_active"], 0)], table[(L["x"], 0)] = l0_x, l_last_x, l_active_x, x
    try:
        numerator = expr_eval(cs.numerator(beta, gamma, y), lambda c, rot: table[(c, rot)])
    except KeyError:
        return None
    expected_h = numerator * pow(xn - 1, -1, R) % R
    # openings as (list of (scalar, point)) commitments, point, eval — same order as the prover's queries
    qs = [([(1, adv_c[c])], rot_pt(rot), v) for (c, rot), v in zip(cs.advice_queries, adv_e)]
    for i in range(cs.num_z):
        qs += [([(1, z_c[i])], x, z_e[i][0]), ([(1, z_c[i])], rot_pt(1), z_e[i][1])]
    for i in reversed(range(cs.num_z - 1)):
        qs.append(([(1, z_c[i])], rot_pt(last_rot), z_e[i][2]))
    for i in range(len(cs.lookups)):
        qs += [([(1, phi_c[i])], x, lk_e[i][0]), ([(1, phi_c[i])], rot_pt(1), lk_e[i][1]), ([(1, m_c[i])], x, lk_e[i][2])]
    fx = [_jac_to_xy(c) for c in keys.fixed_commitments]
    sg = [_jac_to_xy(c) for c in keys.sigma_commitments]
    qs += [([(1, fx[c - na])], rot_pt(rot), v) for (c, rot), v in zip(cs.fixed_queries, fix_e)]
    qs += [([(1, sg[i])], x, sig_e[i]) for i in range(len(sg))]
    qs += [([(pow(xn, i, R), h_c[i]) for i in range(len(h_c))], x, expected_h), ([(1, rand_c)], x, rand_e)]
    try:
        y2, v = tr.squeeze_challenge(), tr.squeeze_challenge()
        h1 = tr.read_ec_point()
        u = tr.squeeze_challenge()
        h2_pt = tr.read_ec_point()
    except ValueError:
        return None
    if tr.pos != len(proof):
        return None
    # rotation sets keyed by the commitment's identity (same grouping rule as the prover: first appearance order)
    by_commit, order = {}, []
    for comm, pt, val in qs:
        key = tuple((sc, p) for sc, p in comm)
        if key not in by_commit:
            by_commit[key] = (comm, [], [])
            order.append(key)
        if pt not in by_commit[key][1]:
            by_commit[key][1].append(pt)
            by_commit[key][2].append(val)
    sets, set_order = {}, []
    for key in order:
        comm, pts, vals = by_commit[key]
        sk = tuple(sorted(pts))
        if sk not in sets:
            sets[sk] = []
            set_order.append(sk)
        sets[sk].append((comm, dict(zip(pts, vals))))
    super_points = []
    for sk in set_order:
        for p in sk:
            if p not in super_points:
                super_points.append(p)
    zt = mo.evaluate_vanishing_polynomial(super_points, u)
    acc = {}                                                           # point -> scalar of the final MSM;  None key = generator

    def add(scalar, pt):
        acc[pt] = (acc.get(pt, 0) + scalar) % R

    z0_inv = None
    for i, sk in enumerate(set_order):
        zd = mo.evaluate_vanishing_polynomial([p for p in super_points if p not in sk], u)
        if z0_inv is None:
            z0_inv = pow(zd, -1, R)
        coef_i = pow(v, i, R) * zd % R * z0_inv % R
        for j, (comm, evals) in enumerate(sets[sk]):
            r_u = sum(c * pow(u, t, R) for t, c in enumerate(mo.lagrange_interpolate(list(sk), [evals[p] for p in sk]))) % R
            cj = coef_i * pow(y2, j, R) % R
            for sc, pt in comm:
                add(cj * sc, pt)
            add(-cj * r_u, "G")
    add(-zt * z0_inv, h1)
    return acc, h2_pt, u


def _msm_points(acc):
    """sum acc[pt] * pt as ONE MSM over the proof's and the key's commitments (normalised Jacobian wire; z = 0 for the identity)."""
    pts, scs = [], []
    for pt, sc in acc.items():
        if pt is None or sc % R == 0:
            continue
        pts.append(_affine_wire((1, 2) if pt == "G" else pt))
        scs.append(F.fr_to_limbs(sc % R))
    if not pts:
        return np.array([0] * 4 + list(F.fq_to_limbs(1)) + [0] * 4, np.uint64)
    bases = h2.Bases(np.stack(pts))
    res = h2.best_multiexp(np.stack(scs), bases)
    bases.release()
    return res


def verify_proof_with_trapdoor(keys: Keys, proof: bytes, s: int, instances=()) -> bool:
    """The restated verifier with the final pairing e(L, [1]_2) == e(h2, [s]_2) replaced by the group equation L - s * h2 == identity
    (the trapdoor s of a test SRS is known), computed as ONE MSM."""
    r = _verifier_accumulate(keys, proof, instances)
    if r is None:
        return False
    acc, h2_pt, u = r
    acc[h2_pt] = (acc.get(h2_pt, 0) + u - s) % R                      # + u * h2 - s * h2
    return not _msm_points(acc)[8:].any()                              # normalised identity has z = 0


def verify_proof_with_pairing(keys: Keys, proof: bytes, pairing_check, instances=()) -> bool:
    """The restated verifier with the REAL final check: pairing_check(L, h2) must decide e(L, [1]_2) == e(h2, [s]_2) for the SRS the
    keys were made with (L, h2 affine (x, y) python ints or None for the identity).  The pairing itself is not on the prover's path and
    is supplied by the caller (tests/pairing_bn254.py runs it on the reference's own SRS fixture)."""
    r = _verifier_accumulate(keys, proof, instances)
    if r is None:
        return False
    acc, h2_pt, u = r
    acc[h2_pt] = (acc.get(h2_pt, 0) + u) % R
    return bool(pairing_check(_jac_to_xy(_msm_points(acc)), h2_pt))


def _jac_to_xy(j):
    j = np.asarray(j, dtype=np.uint64).reshape(12)
    if not j[8:].any():
        return None
    from .transcript import fq_from_limbs
    return (fq_from_limbs(j[:4]), fq_from_limbs(j[4:8]))
