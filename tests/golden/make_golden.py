#!/usr/bin/env python
"""Regenerates tests/golden/* from the reference's own checked-in fixtures.

Needs a checkout of zkonduit/ezkl; the tests read only what this writes:
    python tests/golden/make_golden.py <ezkl checkout>/tests/assets

Inputs (reference fixtures, SURVEY.md Appendix B):
  kzg         ParamsKZG::write output for k=6 (what src/pfsys/srs.rs:40-47 reads)
  pk.key      ProvingKey::write (RawBytes), read by src/pfsys/mod.rs:615
  proof.json  a proof of the k=6 fixture circuit made by the Rust prover

Outputs:
  tests/golden/kzg_k6.srs           the 8452-byte SRS data fixture, verbatim (data, not source)
  tests/golden/pk_k6_subset.npz     a few columns of the proving key:
      fixed_values/fixed_polys/fixed_cosets[c]  c in FIXED_COLS, perm_{values,polys,cosets}[0],
      l0, l_last, l_active_row   -- all as uint64[.,4] little-endian Montgomery limbs (the wire form)
  tests/golden/pk_k6_vk.bin         the verifying-key bytes that open pk.key, verbatim
  tests/golden/pk_k6_values.npy     every fixed column's values, then every permutation column's, uint64[38 + 32, 64, 4];
      with the above, enough to rebuild pk.key byte for byte (tests/helpers.py write_reference_pk; the polys and
      cosets in it are derived from these values)
  tests/golden/reference_proof_k6.bin  the proof bytes of proof.json
  tests/golden/manifest.json        sizes + sha256 of the outputs and of pk.key, and the relations verified while generating

Known-answer content these fixtures give the hot path:
  * 64 MSM known answers:  g_lagrange[j] = n^-1 * sum_i omega^(-ij) * g[i]     (pins MSM, omega, G1 add)
  * NTT known answers:     fixed_values[c] = NTT_omega(fixed_polys[c])          (pins best_fft conventions)
  * coset-NTT answers:     fixed_cosets[c][j] = fixed_polys[c](zeta * omega_9^j) (pins coeff_to_extended)
"""
import hashlib
import json
import os
import struct
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from oracle import pyref as ref  # noqa: E402

FIXED_COLS = [0, 1, 5, 37]


def parse_srs(d: bytes):
    k = struct.unpack("<I", d[:4])[0]
    n = 1 << k
    off = 4
    g = [d[off + 64 * i: off + 64 * (i + 1)] for i in range(n)]
    off += 64 * n
    gl = [d[off + 64 * i: off + 64 * (i + 1)] for i in range(n)]
    off += 64 * n
    assert len(d) - off == 256
    return k, g, gl


def read_poly(d, off):
    (ln,) = struct.unpack(">I", d[off:off + 4])
    off += 4
    return d[off:off + 32 * ln], off + 32 * ln


def read_slice(d, off):
    (cnt,) = struct.unpack(">I", d[off:off + 4])
    off += 4
    lens = struct.unpack(">%dI" % cnt, d[off:off + 4 * cnt])
    off += 4 * cnt
    out = []
    for i in range(cnt):
        p, off = read_poly(d, off)
        assert len(p) == 32 * lens[i]
        out.append(p)
    return out, off


def parse_pk(d: bytes):
    ver, k, _cs = d[0], d[1], d[2]
    assert ver == 3
    n = 1 << k
    (nf,) = struct.unpack("<I", d[3:7])
    off = 7 + 64 * nf
    nperm = 32
    off += 64 * nperm
    nsel = 80
    off += nsel * (n // 8)
    vk = d[:off]
    l0, off = read_poly(d, off)
    l_last, off = read_poly(d, off)
    l_active, off = read_poly(d, off)
    fixed_values, off = read_slice(d, off)
    fixed_polys, off = read_slice(d, off)
    fixed_cosets, off = read_slice(d, off)
    perms, off = read_slice(d, off)
    perm_polys, off = read_slice(d, off)
    perm_cosets, off = read_slice(d, off)
    assert off == len(d), (off, len(d))
    return dict(k=k, vk=vk, l0=l0, l_last=l_last, l_active_row=l_active, fixed_values=fixed_values,
                fixed_polys=fixed_polys, fixed_cosets=fixed_cosets, perms=perms, perm_polys=perm_polys,
                perm_cosets=perm_cosets)


def limbs(b: bytes):
    return np.frombuffer(b, dtype="<u8").reshape(-1, 4).copy()


def frs(b: bytes):
    return [ref.fr_from_wire(b[i:i + 32]) for i in range(0, len(b), 32)]


def save_npz_if_changed(path, arrays):
    """np.savez stamps the time into the archive: keep the committed file when its arrays are already these."""
    if os.path.exists(path):
        old = np.load(path)
        if set(old.files) == set(arrays) and all(np.array_equal(old[name], a) for name, a in arrays.items()):
            return
    np.savez_compressed(path, **arrays)


def main(assets):
    checks = []
    srs = open(os.path.join(assets, "kzg"), "rb").read()
    k, g, gl = parse_srs(srs)
    n = 1 << k
    gp = [ref.g1_from_wire(x) for x in g]
    glp = [ref.g1_from_wire(x) for x in gl]
    assert gp[0] == (1, 2)
    assert all(ref.g1_is_on_curve(p) for p in gp + glp)
    checks.append("kzg: g[0]==(1,2); all 128 points on curve")
    w_inv = pow(ref.omega_for(k), -1, ref.R)
    n_inv = pow(n, -1, ref.R)
    for j in range(n):
        sc = [pow(w_inv, i * j, ref.R) * n_inv % ref.R for i in range(n)]
        assert ref.msm_naive(sc, gp) == glp[j], j
    checks.append("kzg: g_lagrange[j] == n^-1 sum_i omega^-ij g[i] for all 64 j")
    with open(os.path.join(HERE, "kzg_k6.srs"), "wb") as f:
        f.write(srs)

    pk_bytes = open(os.path.join(assets, "pk.key"), "rb").read()
    pk = parse_pk(pk_bytes)
    assert pk["k"] == 6
    ext_k = 9
    out = {}
    for c in FIXED_COLS:
        vals, polys, cos = frs(pk["fixed_values"][c]), frs(pk["fixed_polys"][c]), frs(pk["fixed_cosets"][c])
        assert ref.best_fft(polys, ref.omega_for(6), 6) == vals
        assert ref.lagrange_to_coeff(vals, 6) == polys
        assert ref.coeff_to_extended(polys, 6, ext_k) == cos
        out["fixed_values_%d" % c] = limbs(pk["fixed_values"][c])
        out["fixed_polys_%d" % c] = limbs(pk["fixed_polys"][c])
        out["fixed_cosets_%d" % c] = limbs(pk["fixed_cosets"][c])
    checks.append("pk: fixed_values == best_fft(fixed_polys), fixed_cosets == coeff_to_extended(fixed_polys) "
                  "for cols %s (all rows)" % FIXED_COLS)
    vals, polys, cos = frs(pk["perms"][0]), frs(pk["perm_polys"][0]), frs(pk["perm_cosets"][0])
    assert ref.best_fft(polys, ref.omega_for(6), 6) == vals
    assert ref.coeff_to_extended(polys, 6, ext_k) == cos
    checks.append("pk: permutation col 0 values/polys/cosets consistent")
    out["perm_values_0"], out["perm_polys_0"], out["perm_cosets_0"] = (
        limbs(pk["perms"][0]), limbs(pk["perm_polys"][0]), limbs(pk["perm_cosets"][0]))
    # l0 = L_0 on the extended coset; l_last = L_{n-6}; l_active_row = 1 - l_last - sum blinding rows
    l0c = ref.lagrange_to_coeff([1] + [0] * (n - 1), 6)
    assert ref.coeff_to_extended(l0c, 6, ext_k) == frs(pk["l0"])
    llc = ref.lagrange_to_coeff([1 if i == n - 6 else 0 for i in range(n)], 6)
    assert ref.coeff_to_extended(llc, 6, ext_k) == frs(pk["l_last"])
    checks.append("pk: l0 == coset-extended L_0, l_last == coset-extended L_{n-6}")
    out["l0"], out["l_last"], out["l_active_row"] = limbs(pk["l0"]), limbs(pk["l_last"]), limbs(pk["l_active_row"])
    save_npz_if_changed(os.path.join(HERE, "pk_k6_subset.npz"), out)
    with open(os.path.join(HERE, "pk_k6_vk.bin"), "wb") as f:
        f.write(pk["vk"])
    np.save(os.path.join(HERE, "pk_k6_values.npy"), np.stack([limbs(v) for v in pk["fixed_values"] + pk["perms"]]))

    proof = bytes(json.load(open(os.path.join(assets, "proof.json")))["proof"])
    assert len(proof) == 114 * 64 + 231 * 32 + 2 * 64
    checks.append("proof: 114 commitments, 231 evaluations, 2 SHPLONK points")
    with open(os.path.join(HERE, "reference_proof_k6.bin"), "wb") as f:
        f.write(proof)

    man = {"source": "zkonduit/ezkl tests/assets/{kzg,pk.key,proof.json}", "k": 6, "ext_k": ext_k, "checks": checks}
    for fn in ("kzg_k6.srs", "pk_k6_subset.npz", "pk_k6_vk.bin", "pk_k6_values.npy", "reference_proof_k6.bin"):
        b = open(os.path.join(HERE, fn), "rb").read()
        man[fn] = {"bytes": len(b), "sha256": hashlib.sha256(b).hexdigest()}
    man["pk.key"] = {"bytes": len(pk_bytes), "sha256": hashlib.sha256(pk_bytes).hexdigest()}
    json.dump(man, open(os.path.join(HERE, "manifest.json"), "w"), indent=1)
    print("\n".join(checks))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit("usage: python tests/golden/make_golden.py <ezkl checkout>/tests/assets")
    main(sys.argv[1])
