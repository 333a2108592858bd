"""Host-side mirror of the halo2 interfaces on the prover hot path, executing on the B200 through the C ABI.

Same names, argument meaning and error behaviour as the reference's dependency (UPSTREAM halo2_proofs 0.3.0 @
zkonduit/halo2#01c88842, not vendored; ezkl call sites cited per function), so the parity tests read like the reference's
own: best_multiexp / best_fft / eval_polynomial / kate_division (arithmetic.rs), EvaluationDomain (poly/domain.rs),
ParamsKZG (poly/kzg/commitment.rs; /root/reference/src/pfsys/srs.rs:14-47).

All arrays are numpy uint64 in the wire format (Fr [n,4], G1Affine [n,8]).  No CPU fallback: every function raises
B200Error if the CUDA library or device is unavailable.
"""
from __future__ import annotations

import ctypes as C
import struct

import numpy as np

from . import _native as nat
from . import fields as F


def _fr(a) -> np.ndarray:
    return nat.as_u64(a, 4)


# ------------------------------------------------------------------------------------------------------------
# SRS bases
class Bases:
    """Device-resident, window-precomputed base vector (ParamsKZG.g or .g_lagrange)."""

    def __init__(self, points, window_bits: int = 0):
        nat.ensure_init()
        pts = nat.as_u64(points, 8)
        self.n = pts.shape[0]
        h = C.c_uint64(0)
        nat.check(nat.lib().b200_bases_register(nat.ptr(pts), C.c_size_t(self.n), C.c_int(window_bits), C.byref(h)))
        self.handle = h.value

    @classmethod
    def from_device(cls, d_ptr: int, n: int, window_bits: int = 0):
        nat.ensure_init()
        self = cls.__new__(cls)
        self.n = n
        h = C.c_uint64(0)
        nat.check(nat.lib().b200_bases_register_dev(nat.dev(d_ptr), C.c_size_t(n), C.c_int(window_bits), C.byref(h)))
        self.handle = h.value
        return self

    def info(self):
        n, c, w = C.c_size_t(0), C.c_int(0), C.c_int(0)
        nat.check(nat.lib().b200_bases_info(C.c_uint64(self.handle), C.byref(n), C.byref(c), C.byref(w)))
        return {"n": n.value, "window_bits": c.value, "windows": w.value}

    def release(self):
        if self.handle:
            nat.check(nat.lib().b200_bases_release(C.c_uint64(self.handle)))
            self.handle = 0


# ------------------------------------------------------------------------------------------------------------
# arithmetic.rs
def best_multiexp(coeffs, bases: Bases) -> np.ndarray:
    """sum_i coeffs[i] * bases[i] -> G1 Jacobian wire (uint64[12], normalised z = 1).  Panics upstream if
    coeffs.len() != bases.len(); here len(coeffs) <= len(bases) is accepted (ParamsKZG::commit slices bases[..size])."""
    sc = _fr(coeffs)
    if sc.shape[0] > bases.n:
        raise nat.B200Error("best_multiexp: %d coefficients but %d bases" % (sc.shape[0], bases.n))
    out = np.zeros(12, np.uint64)
    nat.check(nat.lib().b200_msm(C.c_uint64(bases.handle), nat.ptr(sc), C.c_size_t(sc.shape[0]), nat.ptr(out)))
    return out


def best_multiexp_batch(columns, bases: Bases) -> np.ndarray:
    """One MSM per column over shared bases (the per-column commit loops of create_proof) -> [batch,12]."""
    cols = [_fr(c) for c in columns]
    if not cols:
        return np.zeros((0, 12), np.uint64)
    n = cols[0].shape[0]
    assert all(c.shape[0] == n for c in cols)
    out = np.zeros((len(cols), 12), np.uint64)
    nat.check(nat.lib().b200_msm_batch(C.c_uint64(bases.handle), nat.ptr_array(cols), C.c_size_t(n), C.c_size_t(len(cols)), nat.ptr(out)))
    return out


def best_fft(a, omega, log_n: int) -> np.ndarray:
    """In halo2 this mutates `a`; here the transformed copy is returned.  a.len() must be 2^log_n (upstream asserts)."""
    a = _fr(a).copy()
    if a.shape[0] != 1 << log_n:
        raise nat.B200Error("best_fft: len %d != 2^%d" % (a.shape[0], log_n))
    nat.ensure_init()
    nat.check(nat.lib().b200_fft(nat.ptr(a), C.c_uint32(log_n), nat.ptr(_fr(omega))))
    return a


def eval_polynomial(poly, point) -> np.ndarray:
    poly = _fr(poly)
    out = np.zeros(4, np.uint64)
    nat.ensure_init()
    nat.check(nat.lib().b200_poly_eval(nat.ptr(poly), C.c_size_t(poly.shape[0]), nat.ptr(_fr(point)), nat.ptr(out)))
    return out


def eval_polynomial_batch(polys, points) -> np.ndarray:
    ps = [_fr(p) for p in polys]
    xs = _fr(points)
    assert xs.shape[0] == len(ps)
    out = np.zeros((len(ps), 4), np.uint64)
    if not ps:
        return out
    nat.ensure_init()
    nat.check(nat.lib().b200_poly_eval_batch(nat.ptr_array(ps), C.c_size_t(ps[0].shape[0]), nat.ptr(xs), C.c_size_t(len(ps)), nat.ptr(out)))
    return out


def kate_division(a, b) -> np.ndarray:
    a = _fr(a)
    if a.shape[0] < 1:
        raise nat.B200Error("kate_division: empty polynomial")
    q = np.zeros((a.shape[0] - 1, 4), np.uint64)
    nat.ensure_init()
    nat.check(nat.lib().b200_kate_division(nat.ptr(a), C.c_size_t(a.shape[0]), nat.ptr(_fr(b)), nat.ptr(q)))
    return q


def batch_invert(a) -> np.ndarray:
    a = _fr(a).copy()
    nat.ensure_init()
    nat.check(nat.lib().b200_batch_invert(nat.ptr(a), C.c_size_t(a.shape[0])))
    return a


def prefix_scan(a, init, product: bool) -> np.ndarray:
    a = _fr(a)
    out = np.empty_like(a)
    nat.ensure_init()
    nat.check(nat.lib().b200_prefix_scan(C.c_int(1 if product else 0), nat.ptr(a), C.c_size_t(a.shape[0]), nat.ptr(_fr(init)), nat.ptr(out)))
    return out


_OPS = {"add": 0, "sub": 1, "mul": 2, "scale": 3, "axpy": 4}


def poly_op(op: str, a, b=None, s=None) -> np.ndarray:
    """Polynomial +, -, * (element-wise), * scalar, and a + s*b."""
    a = _fr(a)
    out = np.empty_like(a)
    nat.ensure_init()
    bp = nat.ptr(_fr(b)) if b is not None else None
    sp = nat.ptr(_fr(s)) if s is not None else None
    nat.check(nat.lib().b200_poly_op(C.c_int(_OPS[op]), nat.ptr(a), bp, sp, nat.ptr(out), C.c_size_t(a.shape[0])))
    return out


def poly_lincomb(polys, scalars) -> np.ndarray:
    """sum_j scalars[j] * polys[j] in one pass (the multiopen / SHPLONK combinations q(X) = sum y^j p_j(X))."""
    ps = [_fr(p) for p in polys]
    sc = _fr(scalars)
    assert sc.shape[0] == len(ps) and len(ps) > 0
    out = np.zeros_like(ps[0])
    nat.ensure_init()
    nat.check(nat.lib().b200_poly_lincomb(nat.ptr_array(ps), nat.ptr(sc), C.c_size_t(len(ps)), C.c_size_t(ps[0].shape[0]), nat.ptr(out)))
    return out


# ------------------------------------------------------------------------------------------------------------
# poly/domain.rs
class EvaluationDomain:
    """EvaluationDomain::new(j, k) (in-tree use: /root/reference/src/circuit/modules/polycommit.rs:52)."""

    def __init__(self, j: int, k: int):
        nat.ensure_init()
        self.k = k
        self.n = 1 << k
        self.quotient_poly_degree = j - 1
        ext_k = k
        while (1 << ext_k) < self.n * self.quotient_poly_degree:
            ext_k += 1
        if ext_k > F.FR_S:
            raise nat.B200Error("EvaluationDomain: extended_k %d exceeds the field's 2-adicity %d" % (ext_k, F.FR_S))
        self.extended_k = ext_k
        r = F.FR_MODULUS
        ext_omega = pow(F.FR_ROOT_OF_UNITY, 1 << (F.FR_S - ext_k), r)
        omega = pow(ext_omega, 1 << (ext_k - k), r)
        self._omega, self._ext_omega = omega, ext_omega
        self.omega = F.fr_to_limbs(omega)
        self.omega_inv = F.fr_to_limbs(F.fr_inv(omega))
        self.extended_omega = F.fr_to_limbs(ext_omega)
        self.extended_omega_inv = F.fr_to_limbs(F.fr_inv(ext_omega))
        self.g_coset = F.fr_to_limbs(F.FR_ZETA)
        self.g_coset_inv = F.fr_to_limbs(F.FR_ZETA * F.FR_ZETA % r)
        self.ifft_divisor = F.fr_to_limbs(F.fr_inv(1 << k))
        self.extended_ifft_divisor = F.fr_to_limbs(F.fr_inv(1 << ext_k))
        d = 1 << (ext_k - k)
        t = [(pow(F.FR_ZETA * pow(ext_omega, i, r) % r, self.n, r) - 1) % r for i in range(d)]
        self.t_evaluations = np.stack([F.fr_to_limbs(F.fr_inv(v)) for v in t])   # stored inverted, as upstream

    def extended_len(self) -> int:
        return 1 << self.extended_k

    def lagrange_to_coeff(self, a) -> np.ndarray:
        a = _fr(a).copy()
        assert a.shape[0] == self.n
        nat.check(nat.lib().b200_ifft(nat.ptr(a), C.c_uint32(self.k), nat.ptr(self.omega_inv), nat.ptr(self.ifft_divisor)))
        return a

    def lagrange_to_coeff_batch(self, cols):
        cols = [_fr(c).copy() for c in cols]
        if cols:
            nat.check(nat.lib().b200_ifft_batch(nat.ptr_array(cols), C.c_size_t(len(cols)), C.c_uint32(self.k), nat.ptr(self.omega_inv), nat.ptr(self.ifft_divisor)))
        return cols

    def coeff_to_lagrange(self, a) -> np.ndarray:
        return best_fft(a, self.omega, self.k)

    def coeff_to_extended(self, a) -> np.ndarray:
        a = _fr(a)
        assert a.shape[0] == self.n
        out = np.zeros((self.extended_len(), 4), np.uint64)
        nat.check(nat.lib().b200_coeff_to_extended(nat.ptr(a), C.c_size_t(a.shape[0]), C.c_uint32(self.extended_k), nat.ptr(self.extended_omega),
                                                    nat.ptr(self.g_coset), nat.ptr(out)))
        return out

    def coeff_to_extended_batch(self, cols):
        cols = [_fr(c) for c in cols]
        outs = [np.zeros((self.extended_len(), 4), np.uint64) for _ in cols]
        if cols:
            nat.check(nat.lib().b200_coeff_to_extended_batch(nat.ptr_array(cols), C.c_size_t(len(cols)), C.c_size_t(self.n), C.c_uint32(self.extended_k),
                                                              nat.ptr(self.extended_omega), nat.ptr(self.g_coset), nat.ptr_array(outs)))
        return outs

    def coeff_to_extended_part(self, a, part: int) -> np.ndarray:
        """Part `part` of coeff_to_extended(a): its values at zeta * extended_omega^part * omega^t, t < n, i.e. coeff_to_extended(a)[part::d]
        with d = 2^(extended_k - k).  a has at most n coefficients (include/ezkl_b200_parts.h)."""
        return self.coeff_to_extended_part_batch([a], part)[0]

    def coeff_to_extended_part_batch(self, cols, part: int):
        cols = [_fr(c) for c in cols]
        outs = [np.zeros((self.n, 4), np.uint64) for _ in cols]
        if cols:
            n_coeffs = cols[0].shape[0]
            if any(c.shape[0] != n_coeffs for c in cols) or n_coeffs > self.n:
                raise nat.B200Error("coeff_to_extended_part: polynomials need one length <= n = %d" % self.n)
            nat.check(nat.lib().b200_coeff_to_extended_part_batch(nat.ptr_array(cols), C.c_size_t(len(cols)), C.c_size_t(n_coeffs), C.c_uint32(self.k),
                                                                   C.c_uint32(self.extended_k), C.c_uint32(part), nat.ptr(self.extended_omega),
                                                                   nat.ptr(self.g_coset), nat.ptr_array(outs)))
        return outs

    def extended_to_coeff(self, a) -> np.ndarray:
        """Returns n * quotient_poly_degree coefficients (upstream truncates the same way)."""
        a = _fr(a).copy()
        assert a.shape[0] == self.extended_len()
        nat.check(nat.lib().b200_extended_to_coeff(nat.ptr(a), C.c_uint32(self.extended_k), nat.ptr(self.extended_omega_inv),
                                                    nat.ptr(self.extended_ifft_divisor), nat.ptr(self.g_coset)))
        return a[: self.n * self.quotient_poly_degree]

    def divide_by_vanishing_poly(self, a) -> np.ndarray:
        a = _fr(a).copy()
        assert a.shape[0] == self.extended_len()
        nat.check(nat.lib().b200_poly_scale_cycle(nat.ptr(a), C.c_size_t(a.shape[0]), nat.ptr(self.t_evaluations), C.c_uint32(self.t_evaluations.shape[0])))
        return a

    def keygen_l_polys(self, blinding_factors: int):
        """l0, l_last, l_active_row on the extended coset, as halo2 keygen_pk builds them (UPSTREAM plonk/keygen.rs; entered
        from /root/reference/src/pfsys/mod.rs:396): l0 = L_0, l_last = L_{n - blinding_factors - 1},
        l_active_row = 1 - (l_last + l_blind) with l_blind = sum of the Lagrange polynomials of the last blinding rows."""
        l0, l_last, l_blind = self.coeff_to_extended_batch(self._l_basis_coeffs(blinding_factors))
        ones = np.tile(F.fr_to_limbs(1), (self.extended_len(), 1))
        l_active = poly_op("sub", ones, poly_op("add", l_last, l_blind))
        return l0, l_last, l_active

    def keygen_l_coeffs(self, blinding_factors: int):
        """l0, l_last, l_active_row of keygen_l_polys in coefficient form (n coefficients each); their cosets are exactly keygen_l_polys'
        (l_active_row = 1 - (l_last + l_blind) holds coefficient-wise, the constant 1 being the coefficient vector [1, 0, ...])."""
        l0, l_last, l_blind = self._l_basis_coeffs(blinding_factors)
        unit = np.zeros((self.n, 4), np.uint64)
        unit[0] = F.fr_to_limbs(1)
        return l0, l_last, poly_op("sub", unit, poly_op("add", l_last, l_blind))

    def _l_basis_coeffs(self, blinding_factors: int):
        """Coefficients of L_0, L_{n - blinding_factors - 1} and the sum of the last blinding rows' Lagrange polynomials."""
        n = self.n
        one = F.fr_to_limbs(1)
        rows = np.zeros((3, n, 4), np.uint64)
        rows[0, 0] = one
        rows[1, n - blinding_factors - 1] = one
        rows[2, n - blinding_factors:] = one
        return self.lagrange_to_coeff_batch([rows[0], rows[1], rows[2]])

    def rotate_omega(self, value: int, rotation: int) -> int:
        r = F.FR_MODULUS
        return value * pow(self._omega, rotation % self.n, r) % r


def g_to_lagrange(g, k: int) -> np.ndarray:
    """halo2 poly/kzg/commitment.rs g_to_lagrange: best_fft over the group with omega^-1, then * n^-1, then normalise.
    g: [2^k, 8] affine points -> the Lagrange-basis commitment key [2^k, 8]."""
    g = nat.as_u64(g, 8)
    n = 1 << k
    assert g.shape[0] == n
    r = F.FR_MODULUS
    omega = pow(F.FR_ROOT_OF_UNITY, 1 << (F.FR_S - k), r)
    out = np.zeros_like(g)
    nat.ensure_init()
    nat.check(nat.lib().b200_g1_fft(nat.ptr(g), C.c_uint32(k), nat.ptr(F.fr_to_limbs(F.fr_inv(omega))), nat.ptr(F.fr_to_limbs(F.fr_inv(n))), nat.ptr(out)))
    return out


# ------------------------------------------------------------------------------------------------------------
# poly/kzg/commitment.rs
class ParamsKZG:
    """ParamsKZG<Bn256>: k, n, g, g_lagrange (G2 part kept as opaque bytes; it never reaches the prover's MSMs).

    File layout = ParamsKZG::write (SURVEY.md Appendix B): u32 LE k | g[n] | g_lagrange[n] | g2 | s_g2.
    Loaded by the reference through src/pfsys/srs.rs:30-47 (load_srs_prover)."""

    def __init__(self, k: int, g: np.ndarray, g_lagrange: np.ndarray, tail: bytes = b""):
        self.k, self.n = k, 1 << k
        self.g, self.g_lagrange, self._tail = nat.as_u64(g, 8), nat.as_u64(g_lagrange, 8), tail
        assert self.g.shape[0] == self.n and self.g_lagrange.shape[0] == self.n
        self._bases = {}

    @classmethod
    def read(cls, path: str) -> "ParamsKZG":
        d = open(path, "rb").read()
        (k,) = struct.unpack("<I", d[:4])
        n = 1 << k
        if len(d) != 4 + 128 * n + 256:
            raise nat.B200Error("ParamsKZG::read: %d bytes, expected %d for k=%d" % (len(d), 4 + 128 * n + 256, k))
        g = np.frombuffer(d, dtype="<u8", count=8 * n, offset=4).reshape(n, 8).copy()
        gl = np.frombuffer(d, dtype="<u8", count=8 * n, offset=4 + 64 * n).reshape(n, 8).copy()
        return cls(k, g, gl, d[4 + 128 * n:])

    @classmethod
    def setup(cls, k: int, s: int) -> "ParamsKZG":
        """ParamsKZG::new(k) with a caller-supplied trapdoor (the reference's gen_srs uses OsRng; test / bench SRS only).
        The G2 half is not produced: it never reaches the prover's MSMs."""
        from . import device as dev
        g, gl = dev.setup_srs(k, s)
        return cls(k, dev.to_host(g), dev.to_host(gl), b"")

    def downsize(self, new_k: int):
        """ParamsKZG::downsize(k) as ezkl's load_params_prover uses it (/root/reference/src/execute.rs:1745-1748): keep the first
        2^k monomial-basis points and rebuild the Lagrange-basis key with the group FFT."""
        if new_k > self.k:
            raise nat.B200Error("downsize: new k %d > current k %d" % (new_k, self.k))
        if new_k == self.k:
            return
        n = 1 << new_k
        for b in self._bases.values():
            b.release()
        self._bases = {}
        self.k, self.n = new_k, n
        self.g = np.ascontiguousarray(self.g[:n])
        self.g_lagrange = g_to_lagrange(self.g, new_k)

    def write(self, path: str):
        with open(path, "wb") as f:
            f.write(struct.pack("<I", self.k) + self.g.tobytes() + self.g_lagrange.tobytes() + self._tail)

    def _get(self, which: str) -> Bases:
        if which not in self._bases:
            self._bases[which] = Bases(self.g if which == "g" else self.g_lagrange)
        return self._bases[which]

    def commit(self, poly, _blind=None) -> np.ndarray:
        """MSM of coefficient-form poly against g[..len] (the blind is ignored for KZG, as upstream)."""
        return best_multiexp(poly, self._get("g"))

    def commit_lagrange(self, poly, _blind=None) -> np.ndarray:
        """MSM of Lagrange-form poly against g_lagrange (src/circuit/modules/polycommit.rs:71)."""
        poly = _fr(poly)
        if poly.shape[0] != self.n:
            raise nat.B200Error("commit_lagrange: poly has %d evaluations, params n = %d" % (poly.shape[0], self.n))
        return best_multiexp(poly, self._get("g_lagrange"))

    def commit_lagrange_batch(self, polys) -> np.ndarray:
        return best_multiexp_batch(polys, self._get("g_lagrange"))

    def commit_batch(self, polys) -> np.ndarray:
        return best_multiexp_batch(polys, self._get("g"))


# ------------------------------------------------------------------------------------------------------------
# plonk/keygen.rs + plonk.rs ProvingKey (RawBytes layout, SURVEY.md Appendix B)
class ProvingKey:
    """ProvingKey<G1Affine> as `ProvingKey::write(.., SerdeFormat::RawBytes)` lays it out (what src/pfsys/mod.rs:615-636 loads):
    vk bytes | l0 | l_last | l_active_row | fixed_values | fixed_polys | fixed_cosets | permutations | polys | cosets.
    The constraint system is not in the file (upstream re-derives it from the circuit), so the two counts the layout depends on
    are arguments.  `keygen_pk_polys` recomputes every derived vector on the device from fixed_values / permutations."""

    def __init__(self):
        self.k = 0
        self.vk_bytes = b""
        self.l0 = self.l_last = self.l_active_row = None
        self.fixed_values, self.fixed_polys, self.fixed_cosets = [], [], []
        self.permutations, self.permutation_polys, self.permutation_cosets = [], [], []

    @staticmethod
    def _poly(d, off):
        (ln,) = struct.unpack(">I", d[off:off + 4])
        off += 4
        return np.frombuffer(d, dtype="<u8", count=4 * ln, offset=off).reshape(ln, 4).copy(), off + 32 * ln

    @classmethod
    def _slice(cls, d, off):
        (cnt,) = struct.unpack(">I", d[off:off + 4])
        off += 4 + 4 * cnt                       # parallel-poly-read length table
        out = []
        for _ in range(cnt):
            p, off = cls._poly(d, off)
            out.append(p)
        return out, off

    @classmethod
    def read(cls, path: str, num_permutation_columns: int, num_selectors: int) -> "ProvingKey":
        d = open(path, "rb").read()
        pk = cls()
        ver, k = d[0], d[1]
        if ver != 3:
            raise nat.B200Error("ProvingKey::read: unsupported key version %d" % ver)
        pk.k = k
        (nf,) = struct.unpack("<I", d[3:7])
        off = 7 + 64 * nf + 64 * num_permutation_columns + num_selectors * ((1 << k) // 8)
        pk.vk_bytes = d[:off]
        try:
            pk.l0, off = cls._poly(d, off)
            pk.l_last, off = cls._poly(d, off)
            pk.l_active_row, off = cls._poly(d, off)
            pk.fixed_values, off = cls._slice(d, off)
            pk.fixed_polys, off = cls._slice(d, off)
            pk.fixed_cosets, off = cls._slice(d, off)
            pk.permutations, off = cls._slice(d, off)
            pk.permutation_polys, off = cls._slice(d, off)
            pk.permutation_cosets, off = cls._slice(d, off)
        except (ValueError, struct.error) as e:
            raise nat.B200Error("ProvingKey::read: malformed key or wrong column counts (%s)" % e)
        if off != len(d):
            raise nat.B200Error("ProvingKey::read: %d trailing bytes (wrong column counts?)" % (len(d) - off))
        return pk

    def keygen_pk_polys(self, j: int, blinding_factors: int):
        """Recompute on the device what keygen_pk derives (create_keys, /root/reference/src/pfsys/mod.rs:376-400):
        fixed_polys / cosets, permutation polys / cosets, l0 / l_last / l_active_row.  Returns a dict of lists."""
        dom = EvaluationDomain(j, self.k)
        fp = dom.lagrange_to_coeff_batch(self.fixed_values)
        pp = dom.lagrange_to_coeff_batch(self.permutations)
        l0, l_last, l_active = dom.keygen_l_polys(blinding_factors)
        return {"fixed_polys": fp, "fixed_cosets": dom.coeff_to_extended_batch(fp), "permutation_polys": pp,
                "permutation_cosets": dom.coeff_to_extended_batch(pp), "l0": l0, "l_last": l_last, "l_active_row": l_active}
