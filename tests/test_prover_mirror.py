"""create_proof mirror (ezkl_b200/prover.py) + EvmTranscript (ezkl_b200/transcript.py): Keccak known answers, the rng, the proof
encoding against the reference's own fixture, and a full prove -> verify round trip on the ezkl-shaped constraint system."""
import hashlib
import os
import random

import numpy as np
import pytest

from ezkl_b200 import evaluation as ev
from ezkl_b200 import fields as F
from ezkl_b200 import prover as pv
from ezkl_b200 import transcript as ts
from oracle import pyref
from tests import test_constraint_system as tcs

R = pyref.R


def test_keccak256_known_answers_and_permutation_against_sha3():
    assert ts.keccak256(b"").hex() == "c5d2460186f7233c927e7db2dcc703c0e500b653ca82273b7bfad8045d85a470"
    assert ts.keccak256(b"abc").hex() == "4e03657aea45a94fc7d47ba826c8d667c0d1e6e33a64a036ec44f58fa12d6c45"
    # the permutation and the absorb loop are shared with SHA3-256 (only the domain byte differs): check multi-block inputs there
    rng = random.Random(1)
    for ln in (0, 1, 135, 136, 137, 272, 1000):
        data = bytes(rng.randrange(256) for _ in range(ln))
        msg = bytearray(data) + b"\x06"
        while len(msg) % 136:
            msg.append(0)
        msg[-1] |= 0x80
        a = [[0] * 5 for _ in range(5)]
        for off in range(0, len(msg), 136):
            for i in range(17):
                a[i % 5][i // 5] ^= int.from_bytes(msg[off + 8 * i: off + 8 * i + 8], "little")
            a = ts._keccak_f(a)
        assert b"".join(a[i % 5][i // 5].to_bytes(8, "little") for i in range(4)) == hashlib.sha3_256(data).digest(), ln


def test_chacha12_rng_known_answer():
    """ChaCha12 block 0 for the all-zero key / nonce (the stream `StdRng::from_seed([0; 32])` starts with under det-prove,
    /root/reference/src/pfsys/mod.rs:437): first bytes 9b f4 9a 6a 07 55 f9 53 (ChaCha test vectors, TC1, 12 rounds)."""
    rng = pv.ChaCha12Rng(bytes(32))
    first = b"".join(rng.next_u32().to_bytes(4, "little") for _ in range(4))
    assert first.hex() == "9bf49a6a0755f953811fce125f2683d5"
    a = pv.ChaCha12Rng(bytes(32))
    lo, hi = a.next_u32(), a.next_u32()
    b = pv.ChaCha12Rng(bytes(32))
    assert b.next_u64() == lo | (hi << 32)
    assert 0 <= pv.random_fr(pv.ChaCha12Rng(bytes(32))) < R


def test_transcript_rules():
    t = ts.EvmTranscriptWrite()
    t.common_scalar(5)
    assert bytes(t.buf) == (5).to_bytes(32, "big")
    c1 = t.squeeze_challenge()
    assert c1 == int.from_bytes(ts.keccak256((5).to_bytes(32, "big") + b"\x01"), "big") % R     # 32-byte buffer: the 0x01 rule applies to a lone scalar too
    c2 = t.squeeze_challenge()                                                                       # nothing absorbed in between: hash(prev || 0x01)
    assert c2 == int.from_bytes(ts.keccak256(ts.keccak256((5).to_bytes(32, "big") + b"\x01") + b"\x01"), "big") % R
    g = np.concatenate([F.fq_to_limbs(1), F.fq_to_limbs(2)])
    t.write_ec_point(g)
    assert t.finalize() == (1).to_bytes(32, "big") + (2).to_bytes(32, "big") and len(t.buf) == 96
    assert ts.point_bytes(np.zeros(8, np.uint64)) == bytes(64)
    rd = ts.EvmTranscriptRead(t.finalize())
    rd.common_scalar(5)
    rd.squeeze_challenge(), rd.squeeze_challenge()
    assert rd.read_ec_point() == (1, 2)
    with pytest.raises(ValueError):
        ts.EvmTranscriptRead((1).to_bytes(32, "big") + (3).to_bytes(32, "big")).read_ec_point()     # not on the curve


def test_reference_proof_fixture_parses_with_the_read_transcript():
    """The reference's own proof fixture (tests/assets/proof.json, made by the Rust prover; its proof bytes are
    tests/golden/reference_proof_k6.bin): 114 commitments, 231 evaluations, 2 SHPLONK points — every point must pass the on-curve
    check of EvmTranscriptRead, every scalar must be canonical."""
    proof = open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_proof_k6.bin"), "rb").read()
    rd = ts.EvmTranscriptRead(proof)
    assert len(proof) == 114 * 64 + 231 * 32 + 2 * 64
    pts = [rd.read_ec_point() for _ in range(114)]
    scs = [rd.read_scalar() for _ in range(231)]
    pts += [rd.read_ec_point() for _ in range(2)]
    assert rd.pos == len(proof) and all(p is not None for p in pts) and len(scs) == 231


def build_system(rng, k):
    """The ezkl-shaped system of tests/test_constraint_system.py packed as a ConstraintSystem + fixed / sigma columns + advice."""
    col, u = tcs.build_witness(rng, k)
    n = 1 << k
    # flat columns: advice 0..4 (a0, a1, b0, b1, out), fixed 5..11 (five selectors, table, lookup selector)
    gates = ev.base_op_gates(tcs.SEL, [tcs.A0, tcs.A1], [tcs.B0, tcs.B1], tcs.OUT)
    lookup_in = ev.Query(tcs.SEL_L) * ev.Query(tcs.A1) + (ev.Constant(1) - ev.Query(tcs.SEL_L)) * ev.Constant(col[tcs.TABLE][0])
    cs = pv.ConstraintSystem(5, 7, gates, [tcs.A0, tcs.A1, tcs.B0, tcs.B1, tcs.OUT], [([lookup_in], ev.Query(tcs.TABLE))], blinding_factors=tcs.BLIND)
    fixed = [pv._wire(col[c]) for c in range(5, 12)]
    sigmas = [pv._wire(col[c]) for c in tcs.SIG]
    advice = [col[c] for c in range(5)]
    return cs, fixed, sigmas, advice


def test_constraint_system_shape():
    cs, fixed, sigmas, advice = build_system(random.Random(7), 6)
    assert cs.degree == 5 and cs.chunk_len == 3 and cs.num_z == 2
    assert (tcs.OUT, -1) in cs.advice_queries and (tcs.A0, 0) in cs.advice_queries
    L = cs.column_layout()
    assert L["sigma"] == tcs.SIG and L["z"] == tcs.Z and L["lookup"] == [(tcs.M, tcs.PHI)] and L["x"] == tcs.XCOL and L["count"] == tcs.NCOLS


def test_prove_and_verify_round_trip_on_the_cpu_backend(monkeypatch):
    """The create_proof mirror end to end WITHOUT a GPU: transcript, rng, blinding, commit phases, multiplicities, chained grand products,
    grand sum, quotient, evaluations and SHPLONK run as host logic, every polynomial-sized primitive redirected to the CPU oracle
    (tests/cpu_backend.patch_backend).  The proof verifies against the restated verifier at the trapdoor, is deterministic, and every
    rejection case of the GPU test rejects here too."""
    from tests import cpu_backend as cb
    cb.patch_backend(monkeypatch)
    rng = random.Random(123)
    k = 6
    s = rng.randrange(2, R)
    params = cb.FullTrapdoorParams(k, s)
    cs, fixed, sigmas, advice = build_system(rng, k)
    keys = pv.Keys(params, cs, fixed, sigmas, vk_repr=0x77)
    trace = {}
    proof = pv.create_proof(keys, advice, rng=pv.ChaCha12Rng(bytes(32)), trace=trace)
    n_pts = 5 + 1 + 2 + 1 + 1 + keys.domain.quotient_poly_degree
    n_sc = len(cs.advice_queries) + len(cs.fixed_queries) + 1 + 5 + (3 + 2) + 3
    assert len(proof) == 64 * (n_pts + 2) + 32 * n_sc
    assert pv.verify_proof_with_trapdoor(keys, proof, s)
    assert pv.create_proof(keys, advice, rng=pv.ChaCha12Rng(bytes(32))) == proof                 # deterministic (det-prove rng)
    assert pv.create_proof(keys, advice, rng=pv.ChaCha12Rng(bytes([1] * 32))) != proof           # the blinding comes from the rng
    bad = bytearray(proof)
    bad[64 * n_pts + 31] ^= 1
    assert not pv.verify_proof_with_trapdoor(keys, bytes(bad), s)                               # a flipped evaluation
    bad = bytearray(proof)
    bad[40] ^= 1
    assert not pv.verify_proof_with_trapdoor(keys, bytes(bad), s)                               # a flipped commitment coordinate
    assert not pv.verify_proof_with_trapdoor(keys, proof, (s + 1) % R)                          # the wrong trapdoor
    assert not pv.verify_proof_with_trapdoor(keys, proof[:-32], s)                              # a truncated proof
    advice_bad = [list(c) for c in advice]
    advice_bad[tcs.OUT][3] = (advice_bad[tcs.OUT][3] + 1) % R
    assert not pv.verify_proof_with_trapdoor(keys, pv.create_proof(keys, advice_bad, rng=pv.ChaCha12Rng(bytes(32))), s)    # an unsatisfied gate


GOLDEN_PROOF = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mirror_proof_k6.bin")


def golden_case():
    """The fixed case behind tests/golden/mirror_proof_k6.bin: trapdoor, ezkl-shaped system and witness from one seeded generator, the
    det-prove rng (ChaCha12, zero seed)."""
    rng = random.Random(20260923)
    k = 6
    s = rng.randrange(2, R)
    cs, fixed, sigmas, advice = build_system(rng, k)
    return k, s, cs, fixed, sigmas, advice


def test_cpu_backend_proof_equals_the_golden_bytes(monkeypatch):
    """The proof the mirror emits with every primitive on the CPU oracle is the committed golden (regenerate with
    `python tests/test_prover_mirror.py --regenerate` only when the mirror's transcript / rng order changes on purpose)."""
    from tests import cpu_backend as cb
    cb.patch_backend(monkeypatch)
    k, s, cs, fixed, sigmas, advice = golden_case()
    keys = pv.Keys(cb.FullTrapdoorParams(k, s), cs, fixed, sigmas, vk_repr=0x5EED)
    proof = pv.create_proof(keys, advice, rng=pv.ChaCha12Rng(bytes(32)))
    assert pv.verify_proof_with_trapdoor(keys, proof, s)
    assert proof == open(GOLDEN_PROOF, "rb").read()


@pytest.mark.gpu
def test_device_proof_bytes_equal_the_cpu_oracle_proof_bytes():
    """Same SRS trapdoor, circuit, witness and transcript seed: the proof produced through the CUDA library (real SRS, MSM commitments,
    device NTTs / evaluate_h / scans) is BYTE-IDENTICAL to the one produced with every primitive on the CPU oracle (the golden file).
    This is the north star's bit-identical-proof claim with the CPU port standing in for the Rust prover."""
    from ezkl_b200 import _native as nat
    from ezkl_b200 import halo2 as h2
    nat.init(-1)
    k, s, cs, fixed, sigmas, advice = golden_case()
    keys = pv.Keys(h2.ParamsKZG.setup(k, s), cs, fixed, sigmas, vk_repr=0x5EED)
    proof = pv.create_proof(keys, advice, rng=pv.ChaCha12Rng(bytes(32)))
    assert proof == open(GOLDEN_PROOF, "rb").read()


@pytest.mark.gpu
def test_prove_and_verify_round_trip_with_trapdoor_srs():
    from ezkl_b200 import _native as nat
    from ezkl_b200 import halo2 as h2
    nat.init(-1)
    rng = random.Random(99)
    k = 7
    s = rng.randrange(2, R)
    params = h2.ParamsKZG.setup(k, s)
    cs, fixed, sigmas, advice = build_system(rng, k)
    keys = pv.Keys(params, cs, fixed, sigmas, vk_repr=0x1234)
    trace = {}
    proof = pv.create_proof(keys, advice, rng=pv.ChaCha12Rng(bytes(32)), trace=trace)
    # layout: 5 advice + 1 m + 2 z + 1 phi + 1 random + 4 quotient pieces commitments, evaluations, 2 SHPLONK points
    n_pts = 5 + 1 + 2 + 1 + 1 + keys.domain.quotient_poly_degree
    n_sc = len(cs.advice_queries) + len(cs.fixed_queries) + 1 + 5 + (3 + 2) + 3
    assert len(proof) == 64 * (n_pts + 2) + 32 * n_sc
    assert pv.verify_proof_with_trapdoor(keys, proof, s)
    # deterministic: same rng seed, same bytes
    assert pv.create_proof(keys, advice, rng=pv.ChaCha12Rng(bytes(32))) == proof
    # any flipped evaluation, a wrong trapdoor or a truncated proof must fail
    bad = bytearray(proof)
    bad[64 * n_pts + 31] ^= 1
    assert not pv.verify_proof_with_trapdoor(keys, bytes(bad), s)
    assert not pv.verify_proof_with_trapdoor(keys, proof, (s + 1) % R)
    assert not pv.verify_proof_with_trapdoor(keys, proof[:-32], s)
    # an unsatisfied witness: the prover refuses (lookup) or the verifier rejects (gate)
    advice_bad = [list(c) for c in advice]
    advice_bad[tcs.OUT][3] = (advice_bad[tcs.OUT][3] + 1) % R
    proof_bad = pv.create_proof(keys, advice_bad, rng=pv.ChaCha12Rng(bytes(32)))
    assert not pv.verify_proof_with_trapdoor(keys, proof_bad, s)


if __name__ == "__main__":          # python tests/test_prover_mirror.py --regenerate : rewrite the golden proof with the CPU backend
    import sys
    if "--regenerate" in sys.argv:
        from _pytest.monkeypatch import MonkeyPatch
        from tests import cpu_backend as cb
        mp = MonkeyPatch()
        cb.patch_backend(mp)
        k, s, cs, fixed, sigmas, advice = golden_case()
        keys = pv.Keys(cb.FullTrapdoorParams(k, s), cs, fixed, sigmas, vk_repr=0x5EED)
        data = pv.create_proof(keys, advice, rng=pv.ChaCha12Rng(bytes(32)))
        assert pv.verify_proof_with_trapdoor(keys, data, s)
        open(GOLDEN_PROOF, "wb").write(data)
        mp.undo()
        print("wrote %s (%d bytes, sha256 %s)" % (GOLDEN_PROOF, len(data), hashlib.sha256(data).hexdigest()))
