"""Device-resident front end: the same operations as halo2.py, on torch CUDA tensors, with no host round trips.

Tensors are torch.int64 views of the wire format (bit-identical to uint64): Fr columns [n, 4] (or [batch, n, 4]),
G1Affine [n, 8], XYZZ partial sums [batch, 16].  Every call is enqueued on torch's current stream (so torch.cuda.Event
timing and stream ordering see the kernels) and does not synchronise.  torch is plumbing here — allocation, streams,
torch.distributed — the arithmetic is all in libezkl_b200.so.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _native as nat
from . import fields as F


def _stream():
    """torch's current stream as a cudaStream_t.  The legacy default stream has handle 0, which the C ABI reads as "use the
    library's own stream"; pass CUDA's explicit cudaStreamLegacy handle (0x1) instead so ordering and event timing hold."""
    h = torch.cuda.current_stream().cuda_stream
    return C.c_void_p(h if h else 1)


def _chk(t: torch.Tensor, last: int):
    assert t.is_cuda and t.dtype == torch.int64 and t.is_contiguous() and t.shape[-1] == last, (t.dtype, t.shape, t.device)


def _host_fr(x) -> np.ndarray:
    return nat.as_u64(x, 4)


def generate_bases(n: int, seed: int = 0xE2C1B200) -> torch.Tensor:
    nat.ensure_init()
    out = torch.empty((n, 8), dtype=torch.int64, device="cuda")
    nat.check(nat.lib().b200_g1_generate_dev(C.c_uint64(seed), C.c_size_t(n), nat.dev(out.data_ptr()), _stream()))
    return out


def fixed_base_mul(scalars: torch.Tensor, base=None) -> torch.Tensor:
    """scalars [n,4] (Montgomery wire) -> [n,8] affine points [scalar_i] * base (default: the G1 generator (1, 2))."""
    _chk(scalars, 4)
    n = scalars.numel() // 4
    if base is None:
        base = np.concatenate([F.fq_to_limbs(1), F.fq_to_limbs(2)])
    base = nat.as_u64(base, 8)
    out = torch.empty((n, 8), dtype=torch.int64, device="cuda")
    nat.check(nat.lib().b200_g1_fixed_base_mul_dev(nat.dev(scalars.data_ptr()), C.c_size_t(n), nat.ptr(base), nat.dev(out.data_ptr()), _stream()))
    return out


def constant_column(value_int: int, n: int) -> torch.Tensor:
    t = torch.empty((n, 4), dtype=torch.int64, device="cuda")
    t[:] = torch.from_numpy(F.fr_to_limbs(value_int).view(np.int64)).cuda()
    return t


def setup_srs(k: int, s: int):
    """ParamsKZG::new / setup with a caller-chosen trapdoor s (gen_srs, /root/reference/src/pfsys/srs.rs:14-16), all on the device:
    g[i] = [s^i] G,  g_lagrange[i] = [L_i(s)] G with L_i(s) = omega^i (s^n - 1) / (n (s - omega^i)).  Returns (g, g_lagrange) [n,8]."""
    r = F.FR_MODULUS
    n = 1 << k
    omega = pow(F.FR_ROOT_OF_UNITY, 1 << (F.FR_S - k), r)
    one = F.fr_to_limbs(1)
    s_pows = prefix_scan(constant_column(s, n), one, True)                      # s^i
    w_pows = prefix_scan(constant_column(omega, n), one, True)                  # omega^i
    den = poly_op("sub", constant_column(s, n), w_pows)                         # s - omega^i  (s must not be an n-th root of unity)
    batch_invert(den)
    lag = poly_op("mul", w_pows, den)
    poly_op("scale", lag, s=F.fr_to_limbs((pow(s, n, r) - 1) * F.fr_inv(n) % r), out=lag)
    return fixed_base_mul(s_pows), fixed_base_mul(lag)


def random_scalars(n: int, batch: int | None = None, seed: int = 0, small_bits: int | None = None) -> torch.Tensor:
    """Uniform scalars < 2^252 (or < 2^small_bits) in Montgomery wire form, generated on the device with torch's RNG."""
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    shape = (n, 4) if batch is None else (batch, n, 4)
    t = torch.randint(-(1 << 63), (1 << 63) - 1, shape, dtype=torch.int64, device="cuda", generator=g)
    if small_bits is not None:
        assert small_bits <= 62
        t[..., 1:] = 0
        t[..., 0] &= (1 << small_bits) - 1
        # canonical small integers -> Montgomery form: multiply by R^2 via the library (x * R^2 * R^-1 = x R)
        r2 = F.fr_to_limbs(pow(2, 256, F.FR_MODULUS))     # to_limbs(R) = R*R mod r in limbs = R^2 representation
        flat = t.view(-1, 4)
        poly_op("scale", flat, s=r2, out=flat)
        return t
    t[..., 3] &= 0x0FFFFFFFFFFFFFFF
    return t


class DeviceBases:
    def __init__(self, d_points: torch.Tensor, window_bits: int = 0):
        nat.ensure_init()
        _chk(d_points, 8)
        self.n = d_points.shape[0]
        torch.cuda.current_stream().synchronize()
        h = C.c_uint64(0)
        nat.check(nat.lib().b200_bases_register_dev(nat.dev(d_points.data_ptr()), C.c_size_t(self.n), C.c_int(window_bits), C.byref(h)))
        self.handle = h.value

    def release(self):
        if self.handle:
            nat.check(nat.lib().b200_bases_release(C.c_uint64(self.handle)))
            self.handle = 0


def msm_batch(bases: DeviceBases, scalars: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
    """scalars [batch, n, 4] (or [n, 4]) -> un-normalised XYZZ partial sums [batch, 16] on the device."""
    if scalars.dim() == 2:
        scalars = scalars.unsqueeze(0)
    _chk(scalars, 4)
    batch, n = scalars.shape[0], scalars.shape[1]
    if out is None:
        out = torch.empty((batch, 16), dtype=torch.int64, device="cuda")
    nat.check(nat.lib().b200_msm_batch_dev(C.c_uint64(bases.handle), nat.dev(scalars.data_ptr()), C.c_size_t(n), C.c_size_t(n), C.c_size_t(batch),
                                           nat.dev(out.data_ptr()), _stream()))
    return out


def g1_sum(points: torch.Tensor) -> torch.Tensor:
    """points [groups, count, 16] -> [groups, 16]."""
    _chk(points, 16)
    groups, count = points.shape[0], points.shape[1]
    out = torch.empty((groups, 16), dtype=torch.int64, device="cuda")
    nat.check(nat.lib().b200_g1_sum_dev(nat.dev(points.data_ptr()), C.c_size_t(groups), C.c_size_t(count), nat.dev(out.data_ptr()), _stream()))
    return out


def normalize(points_xyzz: torch.Tensor) -> np.ndarray:
    """Device XYZZ [m,16] -> host normalised Jacobian wire [m,12] (synchronises)."""
    h = points_xyzz.cpu().numpy().view(np.uint64).reshape(-1, 16)
    out = np.zeros((h.shape[0], 12), np.uint64)
    nat.check(nat.lib().b200_g1_normalize(nat.ptr(np.ascontiguousarray(h)), C.c_size_t(h.shape[0]), nat.ptr(out)))
    return out


def ntt(src: torch.Tensor, log_n: int, omega, *, n_in: int | None = None, pre=None, post=None, out: torch.Tensor | None = None,
        tmp: torch.Tensor | None = None) -> torch.Tensor:
    """src [batch, n_in, 4] -> out [batch, 2^log_n, 4]; pre/post = None | [c] | [c0,c1,c2] host constants (wire form)."""
    if src.dim() == 2:
        src = src.unsqueeze(0)
    _chk(src, 4)
    batch, n_src = src.shape[0], src.shape[1]
    N = 1 << log_n
    n_in = n_src if n_in is None else n_in
    if out is None:
        out = torch.empty((batch, N, 4), dtype=torch.int64, device="cuda")
    if tmp is None:
        tmp = torch.empty((batch, N, 4), dtype=torch.int64, device="cuda")
    pre_a = np.ascontiguousarray(np.stack([_host_fr(c) for c in pre])) if pre is not None else None
    post_a = np.ascontiguousarray(np.stack([_host_fr(c) for c in post])) if post is not None else None
    nat.check(nat.lib().b200_ntt_dev(nat.dev(src.data_ptr()), C.c_size_t(n_src), C.c_size_t(n_in), nat.dev(tmp.data_ptr()), nat.dev(out.data_ptr()), C.c_size_t(N),
                                     C.c_uint32(log_n), nat.ptr(_host_fr(omega)), C.c_int(0 if pre is None else len(pre)), nat.ptr(pre_a) if pre is not None else None,
                                     C.c_int(0 if post is None else len(post)), nat.ptr(post_a) if post is not None else None, C.c_size_t(batch), _stream()))
    return out


def coeff_to_extended_part(src: torch.Tensor, domain, part: int, *, out: torch.Tensor | None = None, tmp: torch.Tensor | None = None) -> torch.Tensor:
    """src [batch, n_coeffs, 4] (n_coeffs <= n) -> out [batch, n, 4]: part `part` of every polynomial's extended coset,
    coeff_to_extended(p)[part::d] (b200_coeff_to_extended_part_dev).  domain: a halo2.EvaluationDomain."""
    if src.dim() == 2:
        src = src.unsqueeze(0)
    _chk(src, 4)
    batch, n_src = src.shape[0], src.shape[1]
    n = 1 << domain.k
    if out is None:
        out = torch.empty((batch, n, 4), dtype=torch.int64, device="cuda")
    if tmp is None:
        tmp = torch.empty((batch, n, 4), dtype=torch.int64, device="cuda")
    _chk(out, 4)
    _chk(tmp, 4)
    assert out.numel() >= batch * n * 4 and tmp.numel() >= batch * n * 4
    nat.check(nat.lib().b200_coeff_to_extended_part_dev(nat.dev(src.data_ptr()), C.c_size_t(n_src), C.c_size_t(n_src), nat.dev(tmp.data_ptr()),
                                                        nat.dev(out.data_ptr()), C.c_size_t(n), C.c_uint32(domain.k), C.c_uint32(domain.extended_k),
                                                        C.c_uint32(part), nat.ptr(domain.extended_omega), nat.ptr(domain.g_coset), C.c_size_t(batch), _stream()))
    return out


_OPS = {"add": 0, "sub": 1, "mul": 2, "scale": 3, "axpy": 4}


def poly_op(op: str, a: torch.Tensor, b: torch.Tensor | None = None, s=None, out: torch.Tensor | None = None) -> torch.Tensor:
    _chk(a, 4)
    if out is None:
        out = torch.empty_like(a)
    n = a.numel() // 4
    sp = nat.ptr(_host_fr(s)) if s is not None else None
    nat.check(nat.lib().b200_poly_op_dev(C.c_int(_OPS[op]), nat.dev(a.data_ptr()), nat.dev(b.data_ptr()) if b is not None else None, sp,
                                         nat.dev(out.data_ptr()), C.c_size_t(n), _stream()))
    return out


def lincomb(polys, scalars, out: torch.Tensor | None = None) -> torch.Tensor:
    """sum_j scalars[j] * polys[j]; polys = list of [n,4] CUDA tensors (or a [count,n,4] tensor), scalars host [count,4]."""
    plist = [polys[i] for i in range(len(polys))]
    for p_ in plist:
        _chk(p_, 4)
    n = plist[0].numel() // 4
    sc = nat.as_u64(scalars, 4)
    assert sc.shape[0] == len(plist)
    if out is None:
        out = torch.empty_like(plist[0])
    ptrs = (C.c_void_p * len(plist))(*[p_.data_ptr() for p_ in plist])
    nat.check(nat.lib().b200_poly_lincomb_dev(ptrs, nat.ptr(sc), C.c_size_t(len(plist)), C.c_size_t(n), nat.dev(out.data_ptr()), _stream()))
    return out


def scale_cycle(a: torch.Tensor, consts) -> torch.Tensor:
    _chk(a, 4)
    cs = nat.as_u64(consts, 4)
    nat.check(nat.lib().b200_poly_scale_cycle_dev(nat.dev(a.data_ptr()), C.c_size_t(a.numel() // 4), nat.ptr(cs), C.c_uint32(cs.shape[0]), _stream()))
    return a


def eval_batch(polys: torch.Tensor, xs) -> torch.Tensor:
    """polys [batch, n, 4], xs host [batch, 4] -> device [batch, 4]."""
    _chk(polys, 4)
    batch, n = polys.shape[0], polys.shape[1]
    xs = nat.as_u64(xs, 4)
    out = torch.empty((batch, 4), dtype=torch.int64, device="cuda")
    nat.check(nat.lib().b200_poly_eval_batch_dev(nat.dev(polys.data_ptr()), C.c_size_t(n), C.c_size_t(n), nat.ptr(xs), C.c_size_t(batch), nat.dev(out.data_ptr()), _stream()))
    return out


def batch_invert(a: torch.Tensor) -> torch.Tensor:
    _chk(a, 4)
    nat.check(nat.lib().b200_batch_invert_dev(nat.dev(a.data_ptr()), C.c_size_t(a.numel() // 4), _stream()))
    return a


def prefix_scan(a: torch.Tensor, init, product: bool, out: torch.Tensor | None = None) -> torch.Tensor:
    _chk(a, 4)
    if out is None:
        out = torch.empty_like(a)
    nat.check(nat.lib().b200_prefix_scan_dev(C.c_int(1 if product else 0), nat.dev(a.data_ptr()), C.c_size_t(a.numel() // 4), nat.ptr(_host_fr(init)),
                                             nat.dev(out.data_ptr()), _stream()))
    return out


def prefix_scan_batch(a: torch.Tensor, inits, product: bool, out: torch.Tensor | None = None) -> torch.Tensor:
    """a [batch, n, 4]: one exclusive running product / sum per column in one call; inits host [batch, 4]."""
    _chk(a, 4)
    batch, n = a.shape[0], a.shape[1]
    if out is None:
        out = torch.empty_like(a)
    iv = nat.as_u64(inits, 4)
    assert iv.shape[0] == batch
    nat.check(nat.lib().b200_prefix_scan_batch_dev(C.c_int(1 if product else 0), nat.dev(a.data_ptr()), C.c_size_t(n), C.c_size_t(n), C.c_size_t(batch), nat.ptr(iv),
                                                   nat.dev(out.data_ptr()), C.c_size_t(n), _stream()))
    return out


def kate_division(a: torch.Tensor, b, out: torch.Tensor | None = None) -> torch.Tensor:
    _chk(a, 4)
    n = a.numel() // 4
    if out is None:
        out = torch.empty((n - 1, 4), dtype=torch.int64, device="cuda")
    nat.check(nat.lib().b200_kate_division_dev(nat.dev(a.data_ptr()), C.c_size_t(n), nat.ptr(_host_fr(b)), nat.dev(out.data_ptr()), _stream()))
    return out


def to_host(t: torch.Tensor) -> np.ndarray:
    return t.cpu().numpy().view(np.uint64)


def from_host(a: np.ndarray) -> torch.Tensor:
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).cuda()
