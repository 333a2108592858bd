"""Shared helpers for the parity tests: wire-format <-> python int conversion, fixture loading."""
import os
import struct

import numpy as np

from oracle import pyref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def limbs_to_int(a) -> int:
    a = np.asarray(a, dtype=np.uint64).reshape(-1)
    return sum(int(a[i]) << (64 * i) for i in range(a.size))


def int_to_limbs(x: int, n: int = 4) -> np.ndarray:
    return np.array([(x >> (64 * i)) & 0xFFFFFFFFFFFFFFFF for i in range(n)], dtype=np.uint64)


def fr_wire(x: int) -> np.ndarray:
    return int_to_limbs(pyref.to_mont(x % pyref.R, pyref.R))


def fr_unwire(a) -> int:
    return pyref.from_mont(limbs_to_int(a), pyref.R)


def fq_wire(x: int) -> np.ndarray:
    return int_to_limbs(pyref.to_mont(x % pyref.P, pyref.P))


def fr_array(xs) -> np.ndarray:
    return np.stack([fr_wire(x) for x in xs]) if len(xs) else np.zeros((0, 4), np.uint64)


def fr_list(a) -> list:
    return [fr_unwire(r) for r in np.asarray(a).reshape(-1, 4)]


def g1_wire(pt) -> np.ndarray:
    if pt is None:
        return np.zeros(8, np.uint64)
    return np.concatenate([fq_wire(pt[0]), fq_wire(pt[1])])


def g1_unwire(a):
    a = np.asarray(a, np.uint64).reshape(8)
    x, y = pyref.from_mont(limbs_to_int(a[:4]), pyref.P), pyref.from_mont(limbs_to_int(a[4:]), pyref.P)
    return None if (x == 0 and y == 0) else (x, y)


def load_srs_fixture():
    """tests/golden/kzg_k6.srs -> (k, g[n,8], g_lagrange[n,8]) as uint64 wire arrays (ParamsKZG::read layout)."""
    d = open(os.path.join(GOLDEN, "kzg_k6.srs"), "rb").read()
    k = struct.unpack("<I", d[:4])[0]
    n = 1 << k
    g = np.frombuffer(d, dtype="<u8", count=8 * n, offset=4).reshape(n, 8).copy()
    gl = np.frombuffer(d, dtype="<u8", count=8 * n, offset=4 + 64 * n).reshape(n, 8).copy()
    return k, g, gl


def load_pk_fixture():
    return dict(np.load(os.path.join(GOLDEN, "pk_k6_subset.npz")))


def write_reference_pk(path):
    """Rebuilds the reference's k = 6 pk.key (ProvingKey::write, RawBytes) at `path` from tests/golden: the verifying-key bytes,
    l0 / l_last / l_active_row and the Lagrange values of the 38 fixed and 32 permutation columns are stored; their coefficient
    and extended-coset forms are derived with the CPU oracle.  The result must hash to the sha256 the manifest recorded for pk.key."""
    import hashlib
    import json
    from oracle import oracle as orc
    k, ext_k, n_fixed = 6, 9, 38
    values = np.load(os.path.join(GOLDEN, "pk_k6_values.npy"))
    polys = [orc.lagrange_to_coeff(v, k) for v in values]
    cosets = [orc.coeff_to_extended(p, ext_k) for p in polys]
    sub = load_pk_fixture()

    def poly(a):
        return struct.pack(">I", a.shape[0]) + np.ascontiguousarray(a, dtype="<u8").tobytes()

    def slice_(arrs):
        return struct.pack(">I", len(arrs)) + struct.pack(">%dI" % len(arrs), *[a.shape[0] for a in arrs]) + b"".join(poly(a) for a in arrs)

    parts = [open(os.path.join(GOLDEN, "pk_k6_vk.bin"), "rb").read(), poly(sub["l0"]), poly(sub["l_last"]), poly(sub["l_active_row"])]
    for lo, hi in ((0, n_fixed), (n_fixed, len(values))):
        parts += [slice_(list(values[lo:hi])), slice_(polys[lo:hi]), slice_(cosets[lo:hi])]
    data = b"".join(parts)
    expected = json.load(open(os.path.join(GOLDEN, "manifest.json")))["pk.key"]
    assert len(data) == expected["bytes"] and hashlib.sha256(data).hexdigest() == expected["sha256"], "rebuilt pk.key differs from the reference's"
    with open(path, "wb") as f:
        f.write(data)
