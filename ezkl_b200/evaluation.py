"""Host mirror of halo2's plonk/evaluation.rs: Expression -> straight-line program -> b200_quotient_eval (evaluate_h).

halo2's `Expression<F>` (Constant / Fixed / Advice / Instance query at a Rotation / Negated / Sum / Product / Scaled) is
lowered by its `GraphEvaluator` into calculations over value sources; this module does the same lowering into the
instruction format of include/ezkl_b200.h (b200_instr / b200_col_ref): common sub-expressions are shared, results live in
at most 32 slots (linear-scan allocation by last use), constants and column loads are referenced in place.
All queries index one flat list of extended-coset columns; rotations are in rows of the ORIGINAL domain (Rotation(r)),
the kernel scales them by 2^(ext_k - k).  Values are python ints mod r on the host side, wire limbs on the device.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as nat
from . import fields as F

OP_ADD, OP_SUB, OP_MUL, OP_NEG, OP_DOUBLE, OP_SQUARE, OP_MOV, OP_MULADD = range(8)
MAX_SLOTS = 256
NOSTORE = 1 << 31
_SLOT, _CONST, _LOAD, _PREV = 0, 1, 2, 3


class Expression:
    """Immutable expression node; build with Constant / Query and python operators (halo2's Expression<F>: Constant, Fixed /
    Advice / Instance query at a Rotation, Challenge (a Constant here), Negated, Sum, Product, Scaled)."""
    __slots__ = ("kind", "args")

    def __init__(self, kind, *args):
        self.kind, self.args = kind, args

    def __add__(self, o):
        return Expression("sum", self, _wrap(o))

    def __radd__(self, o):
        return Expression("sum", _wrap(o), self)

    def __sub__(self, o):
        return Expression("sub", self, _wrap(o))

    def __rsub__(self, o):
        return Expression("sub", _wrap(o), self)

    def __mul__(self, o):
        return Expression("product", self, _wrap(o))

    def __rmul__(self, o):
        return Expression("product", _wrap(o), self)

    def __neg__(self):
        return Expression("negated", self)


def Constant(v: int) -> Expression:
    return Expression("constant", v % F.FR_MODULUS)


def Query(column: int, rotation: int = 0) -> Expression:
    """Value of extended-coset column `column` at Rotation(rotation) (Fixed / Advice / Instance query)."""
    return Expression("query", int(column), int(rotation))


def _wrap(o):
    return o if isinstance(o, Expression) else Constant(int(o))


class QuotientProgram:
    """Compiled program: loads [(column, rotation)], constants [int], instructions [(op, dst_slot | NOSTORE, a, b, c)].

    Lowering (what halo2's GraphEvaluator::add_expression does, for the instruction format of include/ezkl_b200.h):
      * hash-consing — structurally equal sub-expressions become one node (memoised per object, so shared DAGs such as repeated
        squaring cost O(nodes), not O(tree));
      * a product whose only use is one operand of a sum becomes a fused multiply-add (GraphEvaluator's Horner steps are exactly these);
      * evaluation order by register need (the operand that needs more registers first), results in at most 256 slots allocated by
        last use; a result read only by the next instruction stays in the PREV register and is never stored."""

    def __init__(self, expr: Expression):
        self.loads, self.consts, self.instrs = [], [], []
        self._load_ix, self._const_ix = {}, {}
        # ---- 1. hash-consed DAG: node id -> (kind, payload / child ids)
        by_key, memo, nodes = {}, {}, []

        def intern(kind, payload):
            key = (kind,) + tuple(payload)
            if key not in by_key:
                by_key[key] = len(nodes)
                nodes.append((kind, tuple(payload)))
            return by_key[key]

        stack = [(expr, False)]
        while stack:                                       # iterative post-order: deep Horner chains do not hit the recursion limit
            e, ready = stack.pop()
            if id(e) in memo:
                continue
            if e.kind in ("constant", "query"):
                memo[id(e)] = intern(e.kind, e.args)
            elif ready:
                kids = tuple(memo[id(a)] for a in e.args)
                kind = e.kind
                if kind == "product" and kids[0] == kids[1]:
                    kind, kids = "square", (kids[0],)
                memo[id(e)] = intern(kind, kids)
            else:
                stack.append((e, True))
                for a in e.args:
                    if id(a) not in memo:
                        stack.append((a, False))
        root = memo[id(expr)]
        self._keep = expr                                  # ids in `memo` stay valid while the tree is alive
        leaf = lambda i: nodes[i][0] in ("constant", "query")
        if leaf(root):                                     # a bare leaf still needs one instruction to produce a row value
            root = intern("mov", (root,))
        # ---- 2. reference counts over the reachable DAG, then multiply-add fusion
        uses = {}
        seen, order_probe = set(), [root]
        while order_probe:
            i = order_probe.pop()
            if i in seen:
                continue
            seen.add(i)
            for c in (() if leaf(i) else nodes[i][1]):
                uses[c] = uses.get(c, 0) + 1
                order_probe.append(c)
        fused = {}                                         # sum node -> (x, y, addend) with x * y the absorbed product
        for i in seen:
            kind, kids = nodes[i]
            if kind == "sum":
                for pos in (0, 1):
                    p = kids[pos]
                    if nodes[p][0] == "product" and uses.get(p, 0) == 1:
                        fused[i] = (nodes[p][1][0], nodes[p][1][1], kids[1 - pos])
                        break
        operands_of = lambda i: fused[i] if i in fused else nodes[i][1]
        # ---- 3. register need (Sethi-Ullman on the DAG, shared nodes counted where first met) and evaluation order
        need = {}
        order = []
        work = [(root, False)]
        done = set()
        while work:
            i, ready = work.pop()
            if i in done or leaf(i):
                continue
            ops = [c for c in operands_of(i) if not leaf(c)]
            if ready:
                ns = sorted((need.get(c, 0) for c in ops), reverse=True)
                need[i] = max([n_ + j for j, n_ in enumerate(ns)] + [1])
                done.add(i)
                order.append(i)
            else:
                work.append((i, True))
                # children pushed so that the one with the LARGER need is popped (evaluated) first: estimate by subtree depth
                for c in sorted(ops, key=lambda c_: self._depth(nodes, operands_of, c_, leaf)):
                    if c not in done:
                        work.append((c, False))
        # ---- 4. emission with last-use slot allocation
        pos_of = {i: p for p, i in enumerate(order)}
        last_use, use_list = {}, {}
        for p, i in enumerate(order):
            for c in operands_of(i):
                if not leaf(c):
                    last_use[c] = p
                    use_list.setdefault(c, []).append(p)
        free, slot_of = list(range(MAX_SLOTS - 1, -1, -1)), {}

        def operand(c, p):
            kind, payload = nodes[c]
            if kind == "constant":
                if payload[0] not in self._const_ix:
                    self._const_ix[payload[0]] = len(self.consts)
                    self.consts.append(payload[0])
                return (_CONST << 30) | self._const_ix[payload[0]]
            if kind == "query":
                if payload not in self._load_ix:
                    self._load_ix[payload] = len(self.loads)
                    self.loads.append(payload)
                return (_LOAD << 30) | self._load_ix[payload]
            if pos_of[c] == p - 1:
                return _PREV << 30
            return (_SLOT << 30) | slot_of[c]

        opmap = {"sum": OP_ADD, "sub": OP_SUB, "product": OP_MUL, "negated": OP_NEG, "mov": OP_MOV, "square": OP_SQUARE}
        for p, i in enumerate(order):
            kind, _ = nodes[i]
            ops = operands_of(i)
            enc = [operand(c, p) for c in ops] + [0, 0]
            op = OP_MULADD if i in fused else opmap[kind]
            for c in set(ops):                             # operands whose last use is here free their slot before dst is chosen
                if c in slot_of and last_use.get(c) == p:
                    free.append(slot_of.pop(c))
            only_next = use_list.get(i) == [p + 1] or (i == root)
            if only_next:
                dst = NOSTORE
            else:
                if not free:
                    raise nat.B200Error("QuotientProgram: more than %d live intermediates; split the constraint system into partial sums" % MAX_SLOTS)
                slot_of[i] = free.pop()
                dst = slot_of[i]
            self.instrs.append((op, dst, enc[0], enc[1], enc[2]))

    @staticmethod
    def _depth(nodes, operands_of, i, leaf, _cache={}):
        # iterative depth with a per-call cache keyed on the node table identity
        key = (id(nodes), i)
        if key in _cache:
            return _cache[key]
        stack = [(i, False)]
        while stack:
            j, ready = stack.pop()
            kj = (id(nodes), j)
            if kj in _cache:
                continue
            if leaf(j):
                _cache[kj] = 0
                continue
            kids = operands_of(j)
            if ready:
                _cache[kj] = 1 + max(_cache[(id(nodes), c)] for c in kids)
            else:
                stack.append((j, True))
                for c in kids:
                    if (id(nodes), c) not in _cache:
                        stack.append((c, False))
        return _cache[key]

    @property
    def n_slots(self):
        return 1 + max([d & 0xFFFF for _, d, *_ in self.instrs if not d & NOSTORE] + [0])

    def arrays(self):
        loads = np.array(self.loads, dtype=np.int64).reshape(-1, 2).astype(np.int32)
        consts = np.stack([F.fr_to_limbs(c) for c in self.consts]) if self.consts else np.zeros((0, 4), np.uint64)
        prog = np.array([[(op | ((dst & 0xFFFF) << 8) | (dst & NOSTORE)), a, b, c] for op, dst, a, b, c in self.instrs], dtype=np.uint32).reshape(-1, 4)
        return np.ascontiguousarray(loads), np.ascontiguousarray(consts), np.ascontiguousarray(prog)

    def evaluate_ints(self, column_values, idx: int, n_rows: int, rot_scale: int) -> int:
        """Reference semantics on python ints (used by the tests to cross-check the compiler itself)."""
        r = F.FR_MODULUS
        slots = [0] * MAX_SLOTS
        prev = 0

        def src(s):
            kind, i = s >> 30, s & 0x3FFFFFFF
            if kind == _PREV:
                return prev
            if kind == _SLOT:
                return slots[i]
            if kind == _CONST:
                return self.consts[i]
            col, rot = self.loads[i]
            return column_values[col][(idx + rot * rot_scale) % n_rows]

        for op, dst, a, b, c in self.instrs:
            x = src(a)
            if op == OP_ADD:
                v = x + src(b)
            elif op == OP_SUB:
                v = x - src(b)
            elif op == OP_MUL:
                v = x * src(b)
            elif op == OP_MULADD:
                v = x * src(b) + src(c)
            elif op == OP_NEG:
                v = -x
            elif op == OP_DOUBLE:
                v = 2 * x
            elif op == OP_SQUARE:
                v = x * x
            else:
                v = x
            prev = v % r
            if not dst & NOSTORE:
                slots[dst] = prev
        return prev


def evaluate_h(program: QuotientProgram, columns, k: int, ext_k: int) -> np.ndarray:
    """Host-buffer path: columns = list of [2^ext_k, 4] wire arrays -> [2^ext_k, 4]."""
    nat.ensure_init()
    cols = [nat.as_u64(c, 4) for c in columns]
    N = 1 << ext_k
    assert all(c.shape[0] == N for c in cols)
    loads, consts, prog = program.arrays()
    out = np.zeros((N, 4), np.uint64)
    nat.check(nat.lib().b200_quotient_eval(nat.ptr_array(cols) if cols else None, C.c_size_t(len(cols)), C.c_uint32(k), C.c_uint32(ext_k),
                                           loads.ctypes.data_as(C.c_void_p), C.c_size_t(loads.shape[0]), nat.ptr(consts) if consts.size else None,
                                           C.c_size_t(consts.shape[0]), prog.ctypes.data_as(C.c_void_p), C.c_size_t(prog.shape[0]), nat.ptr(out)))
    return out


def evaluate_h_from_polys(program: QuotientProgram, polys, domain, finish: bool = False) -> np.ndarray:
    """b200_evaluate_h: columns given as the prover holds them — coefficient form (len < 2^ext_k: the library builds the coset) or already on
    the extended domain (len == 2^ext_k).  `domain` is a halo2.EvaluationDomain; finish=True also divides by the vanishing polynomial
    and returns the quotient's coefficients (all 2^ext_k of them)."""
    nat.ensure_init()
    cols = [nat.as_u64(c, 4) for c in polys]
    N = 1 << domain.extended_k
    lens = (C.c_size_t * max(1, len(cols)))(*[c.shape[0] for c in cols])
    loads, consts, prog = program.arrays()
    out = np.zeros((N, 4), np.uint64)
    t_ev = nat.ptr(domain.t_evaluations) if finish else None
    nat.check(nat.lib().b200_evaluate_h(nat.ptr_array(cols) if cols else None, lens, C.c_size_t(len(cols)), C.c_uint32(domain.k), C.c_uint32(domain.extended_k),
                                        nat.ptr(domain.extended_omega), nat.ptr(domain.g_coset), loads.ctypes.data_as(C.c_void_p), C.c_size_t(loads.shape[0]),
                                        nat.ptr(consts) if consts.size else None, C.c_size_t(consts.shape[0]), prog.ctypes.data_as(C.c_void_p), C.c_size_t(prog.shape[0]),
                                        t_ev, C.c_uint32(domain.t_evaluations.shape[0] if finish else 0), nat.ptr(domain.extended_omega_inv) if finish else None,
                                        nat.ptr(domain.extended_ifft_divisor) if finish else None, nat.ptr(out)))
    return out


def _parts_args(program: QuotientProgram, lengths, domain, finish: bool):
    """Arguments shared by b200_evaluate_h_parts and its device form, after the column pointers (include/ezkl_b200_parts.h)."""
    lens = (C.c_size_t * max(1, len(lengths)))(*lengths)
    loads, consts, prog = program.arrays()
    t = domain.t_evaluations
    keep = (loads, consts, prog)
    args = [lens, C.c_size_t(len(lengths)), C.c_uint32(domain.k), C.c_uint32(domain.extended_k), nat.ptr(domain.extended_omega), nat.ptr(domain.g_coset),
            loads.ctypes.data_as(C.c_void_p), C.c_size_t(loads.shape[0]), nat.ptr(consts) if consts.size else None, C.c_size_t(consts.shape[0]),
            prog.ctypes.data_as(C.c_void_p), C.c_size_t(prog.shape[0]), nat.ptr(t) if finish else None, C.c_uint32(t.shape[0] if finish else 0),
            nat.ptr(domain.extended_omega_inv) if finish else None, nat.ptr(domain.extended_ifft_divisor) if finish else None]
    return args, keep


def evaluate_h_parts(program: QuotientProgram, polys, domain, finish: bool = False) -> np.ndarray:
    """b200_evaluate_h_parts: what evaluate_h_from_polys computes, byte for byte, evaluated one coset part of the extended domain at a time,
    so that no column's full coset is ever on the device.  Columns are coefficient form (len <= n) or on the extended domain
    (len == 2^extended_k); finish=True returns the quotient's coefficients (all 2^extended_k of them)."""
    nat.ensure_init()
    cols = [nat.as_u64(c, 4) for c in polys]
    N = 1 << domain.extended_k
    args, _keep = _parts_args(program, [c.shape[0] for c in cols], domain, finish)
    out = np.zeros((N, 4), np.uint64)
    nat.check(nat.lib().b200_evaluate_h_parts(nat.ptr_array(cols) if cols else None, *args, nat.ptr(out)))
    return out


def evaluate_h_parts_device(program: QuotientProgram, columns, domain, finish: bool = False, out=None):
    """Device form of evaluate_h_parts: columns = list of torch int64 CUDA tensors [len, 4] (len <= n: coefficients, len == 2^extended_k:
    extended values, read in place); enqueued on torch's current stream.  Returns out [2^extended_k, 4]."""
    import torch
    from .device import _stream
    N = 1 << domain.extended_k
    for c in columns:
        assert c.is_cuda and c.dtype == torch.int64 and c.is_contiguous() and c.dim() == 2 and c.shape[1] == 4
    if out is None:
        out = torch.empty((N, 4), dtype=torch.int64, device="cuda")
    assert out.is_cuda and out.dtype == torch.int64 and out.is_contiguous() and out.shape == (N, 4)
    args, _keep = _parts_args(program, [c.shape[0] for c in columns], domain, finish)
    ptrs = (C.c_void_p * max(1, len(columns)))(*[c.data_ptr() for c in columns])
    nat.check(nat.lib().b200_evaluate_h_parts_dev(ptrs, *args, nat.dev(out.data_ptr()), _stream()))
    return out


def evaluate_h_device(program: QuotientProgram, columns, k: int, ext_k: int, out=None):
    """Device path: columns = list of torch int64 CUDA tensors [2^ext_k, 4]; enqueued on torch's current stream."""
    import torch
    from .device import _stream
    N = 1 << ext_k
    for c in columns:
        assert c.is_cuda and c.dtype == torch.int64 and c.is_contiguous() and c.shape == (N, 4)
    if out is None:
        out = torch.empty((N, 4), dtype=torch.int64, device="cuda")
    loads, consts, prog = program.arrays()
    ptrs = (C.c_void_p * max(1, len(columns)))(*[c.data_ptr() for c in columns])
    nat.check(nat.lib().b200_quotient_eval_dev(ptrs, C.c_size_t(len(columns)), C.c_uint32(k), C.c_uint32(ext_k), loads.ctypes.data_as(C.c_void_p),
                                               C.c_size_t(loads.shape[0]), nat.ptr(consts) if consts.size else None, C.c_size_t(consts.shape[0]),
                                               prog.ctypes.data_as(C.c_void_p), C.c_size_t(prog.shape[0]), nat.dev(out.data_ptr()), _stream()))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# Permutation grand product and mv-lookup grand sum (halo2 plonk/permutation/prover.rs, plonk/mv_lookup/prover.rs; stage 3
# of create_proof, SURVEY.md §3.1): row-wise numerator / denominator programs on the Lagrange domain (the same
# interpreter with k == ext_k), one batch inversion, one running product / sum.  All on the device.
DELTA = pow(7, 1 << 28, F.FR_MODULUS)          # Fr::DELTA = GENERATOR^(2^S): coset separator of the permutation argument


def _omega_powers_column(k: int) -> np.ndarray:
    """Lagrange-domain column of omega^i (the identity polynomial's values), built on the host once per k."""
    w = pow(F.FR_ROOT_OF_UNITY, 1 << (F.FR_S - k), F.FR_MODULUS)
    out, cur = [], 1
    for _ in range(1 << k):
        out.append(F.fr_to_limbs(cur))
        cur = cur * w % F.FR_MODULUS
    return np.stack(out)


def permutation_product(values, sigmas, k: int, beta: int, gamma: int, delta_start: int = 1, z0: int = 1, blinding_factors: int = 0, blinds=None):
    """z(X) in Lagrange form for ONE permutation chunk (halo2 plonk/permutation/prover.rs, the loop over column chunks):
        z[0] = z0 (the previous chunk's last_z; 1 for the first chunk),
        z[i+1] = z[i] * prod_j (v_j[i] + beta * delta_start * DELTA^j * omega^i + gamma) / (v_j[i] + beta * sigma_j[i] + gamma),
    the last `blinding_factors` rows overwritten with `blinds` (python ints; the prover draws them from its rng).
    values / sigmas: lists of [n,4] Lagrange columns (wire form); delta_start = DELTA^(index of the chunk's first column).
    Returns (z [n,4], last_z) with last_z = z[n - blinding_factors - 1], the seed of the next chunk."""
    from . import halo2 as h2
    m = len(values)
    assert m == len(sigmas) and m > 0
    r = F.FR_MODULUS
    n = 1 << k
    cols = list(values) + list(sigmas) + [_omega_powers_column(k)]
    X = Query(2 * m)
    num = den = None
    for j in range(m):
        d = delta_start * pow(DELTA, j, r) % r
        tn = Query(j) + X * Constant(beta * d % r) + Constant(gamma)
        td = Query(j) + Query(m + j) * Constant(beta) + Constant(gamma)
        num = tn if num is None else num * tn
        den = td if den is None else den * td
    numer = evaluate_h(QuotientProgram(num), cols, k, k)
    denom = h2.batch_invert(evaluate_h(QuotientProgram(den), cols, k, k))
    ratio = h2.poly_op("mul", numer, denom)
    z = h2.prefix_scan(ratio, F.fr_to_limbs(z0), True)
    if blinding_factors:
        assert blinds is not None and len(blinds) == blinding_factors
        for i, b in enumerate(blinds):
            z[n - blinding_factors + i] = F.fr_to_limbs(b)
    last_z = F.fr_from_limbs(z[n - blinding_factors - 1])
    return z, last_z


def permutation_products(columns, sigmas, k: int, beta: int, gamma: int, chunk_len: int, blinding_factors: int = 0, blinds=None):
    """All z_i(X) of a permutation argument: the columns are cut into chunks of chunk_len = cs.degree() - 2, every chunk's
    product starts at the previous chunk's last_z and its first column uses DELTA^(chunk start).  Returns the list of z columns."""
    zs, last_z = [], 1
    for ci, c0 in enumerate(range(0, len(columns), chunk_len)):
        bl = None if blinds is None else blinds[ci]
        z, last_z = permutation_product(columns[c0:c0 + chunk_len], sigmas[c0:c0 + chunk_len], k, beta, gamma, pow(DELTA, c0, F.FR_MODULUS), last_z, blinding_factors, bl)
        zs.append(z)
    return zs


def lookup_multiplicities(table, inputs, n_rows: int):
    """m(X) of an mv-lookup (stage 2): host-buffer call of b200_lookup_multiplicities; raises when an input is not in the table."""
    nat.ensure_init()
    t = nat.as_u64(table, 4)
    ins = [nat.as_u64(c, 4) for c in inputs]
    m = np.zeros_like(t)
    missing = C.c_uint64(0)
    nat.check(nat.lib().b200_lookup_multiplicities(nat.ptr(t), C.c_size_t(t.shape[0]), nat.ptr_array(ins), C.c_size_t(len(ins)), C.c_size_t(n_rows), nat.ptr(m), C.byref(missing)))
    if missing.value:
        raise nat.B200Error("lookup_multiplicities: %d input cells are not in the table" % missing.value)
    return m


# ---------------------------------------------------------------------------------------------------------------------
# Constraint-system terms in the order Evaluator::evaluate_h folds them (custom gates, permutation, lookups); each builder
# returns a list of Expressions over the flat coset-column list, `fold_y` chains them as value = value * y + term.
def fold_y(terms, y: int, start: Expression | None = None) -> Expression:
    value = start if start is not None else Constant(0)
    yc = Constant(y)
    for t in terms:
        value = value * yc + t
    return value


def base_op_gates(selectors: dict, a, b, out: int) -> list:
    """ezkl's BaseConfig custom gates for one block (/root/reference/src/circuit/ops/chip.rs:362-424, formulas
    /root/reference/src/circuit/ops/base.rs:28-66): `a`, `b` are the column indices of the two inputs' inner columns, `out` the
    output column; selectors maps an op name to its selector column.  Non-accumulating ops constrain every inner column,
    accumulating ops read the previous output at Rotation(-1) and constrain the row's single output cell."""
    A, B = [Query(c) for c in a], [Query(c) for c in b]
    terms = []
    for name, f in (("ADD", lambda x, y_: x + y_), ("SUB", lambda x, y_: x - y_), ("MULT", lambda x, y_: x * y_)):
        if name in selectors:
            sel = Query(selectors[name])
            # one output cell per inner column pair: out column queried at the same row (inner columns share the row in ezkl's layout;
            # here each pair writes the single output column of its own block)
            terms.append(sel * (Query(out) - f(A[0], B[0])))
    dot = None
    for x, y_ in zip(A, B):
        dot = x * y_ if dot is None else dot + x * y_
    ssum = None
    for y_ in B:
        ssum = y_ if ssum is None else ssum + y_
    prod = None
    for y_ in B:
        prod = y_ if prod is None else prod * y_
    prev = Query(out, -1)
    for name, res in (("DOTINIT", dot), ("DOT", prev + dot), ("SUMINIT", ssum), ("SUM", prev + ssum), ("CUMPRODINIT", prod), ("CUMPROD", prev * prod)):
        if name in selectors:
            terms.append(Query(selectors[name]) * (Query(out) - res))
    return terms


def permutation_terms(columns, sigmas, zs, l0: int, l_last: int, l_active: int, x_col: int, beta: int, gamma: int, chunk_len: int, blinding_factors: int) -> list:
    """The permutation argument's terms (UPSTREAM plonk/evaluation.rs, "Permutations"): columns / sigmas / zs are column indices
    (values, sigma cosets, grand products), x_col the coset of the identity polynomial X, rotations of z at +1 and -(blinding+1)."""
    r = F.FR_MODULUS
    last_rot = -(blinding_factors + 1)
    L0, LL, LA, X = Query(l0), Query(l_last), Query(l_active), Query(x_col)
    terms = [(Constant(1) - Query(zs[0])) * L0, (Query(zs[-1]) * Query(zs[-1]) - Query(zs[-1])) * LL]
    for i in range(1, len(zs)):
        terms.append((Query(zs[i]) - Query(zs[i - 1], last_rot)) * L0)
    for ci, z in enumerate(zs):
        cols = columns[ci * chunk_len:(ci + 1) * chunk_len]
        sig = sigmas[ci * chunk_len:(ci + 1) * chunk_len]
        left, right = Query(z, 1), Query(z)
        for j, (c, s_) in enumerate(zip(cols, sig)):
            left = left * (Query(c) + Query(s_) * Constant(beta) + Constant(gamma))
            right = right * (Query(c) + X * Constant(beta * pow(DELTA, ci * chunk_len + j, r) % r) + Constant(gamma))
        terms.append((left - right) * LA)
    return terms


def mv_lookup_terms(inputs, table: Expression, m: int, phi: int, l0: int, l_last: int, l_active: int, beta: int) -> list:
    """One mv-lookup's terms (zkonduit fork, UPSTREAM plonk/evaluation.rs "Lookups"): inputs = list of (theta-compressed) input
    Expressions f_i, table = compressed table Expression t.  With phi_i = f_i + beta and tau = t + beta:
        l0 * Phi,   l_last * Phi,   l_active * ( tau * prod(phi_i) * (Phi(wX) - Phi(X))  -  (tau * sum_i prod_{j != i} phi_j  -  m * prod(phi_i)) ).
    (The CPU evaluator writes the second bracket with per-row inversions, prod(phi) * (tau * sum 1/phi_i - m); the two agree wherever
    no phi_i vanishes.)"""
    phis = [f + Constant(beta) for f in inputs]
    tau = table + Constant(beta)
    prod = phis[0]
    for p_ in phis[1:]:
        prod = prod * p_
    partial = None
    for i in range(len(phis)):
        term = None
        for j, p_ in enumerate(phis):
            if j != i:
                term = p_ if term is None else term * p_
        term = term if term is not None else Constant(1)
        partial = term if partial is None else partial + term
    lhs = tau * prod * (Query(phi, 1) - Query(phi))
    rhs = tau * partial - Query(m) * prod
    return [Query(l0) * Query(phi), Query(l_last) * Query(phi), (lhs - rhs) * Query(l_active)]


def lookup_grand_sum(inputs, table, multiplicities, k: int, beta: int) -> np.ndarray:
    """phi(X) in Lagrange form for a logUp / mv-lookup argument:  phi[0] = 0,
        phi[i+1] = phi[i] + sum_j 1 / (f_j[i] + beta) - m[i] / (t[i] + beta).
    inputs: list of compressed input-expression columns f_j; table: compressed table column t; multiplicities: m."""
    from . import halo2 as h2
    nin = len(inputs)
    cols = list(inputs) + [table]
    one = F.fr_to_limbs(1)
    dens = [h2.batch_invert(evaluate_h(QuotientProgram(Query(j) + Constant(beta)), cols, k, k)) for j in range(nin + 1)]
    acc = dens[0]
    for j in range(1, nin):
        acc = h2.poly_op("add", acc, dens[j])
    acc = h2.poly_op("sub", acc, h2.poly_op("mul", multiplicities, dens[nin]))
    return h2.prefix_scan(acc, np.zeros(4, np.uint64), False)
