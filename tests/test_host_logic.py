"""CPU-side checks of the product: C-ABI surface, loud failure without a device, and the host-compiled (portable-path)
field / group-law / digit-recoding code that the CUDA kernels share with the host, against the oracle."""
import ctypes as C
import os
import random
import re

import numpy as np
import pytest

from ezkl_b200 import _native as nat
from ezkl_b200 import fields as F
from oracle import oracle as orc
from oracle import pyref
from tests import helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_cabi_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "ezkl_b200.h")).read()
    names = re.findall(r"^\s*(?:int|void|uint64_t|const char\*)\s+(b200_\w+)\s*\(", hdr, flags=re.M)
    assert len(names) >= 40
    lib = nat.lib()
    for nm in names:
        assert hasattr(lib, nm), "libezkl_b200.so does not export %s" % nm


def test_no_cpu_fallback_without_device():
    """Without a usable CUDA device the product must fail loudly (never compute on the CPU)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    lib = nat.lib()
    assert lib.b200_init(C.c_int(-1)) != 0
    assert b"no CUDA device" in lib.b200_last_error()
    a = np.zeros((4, 4), np.uint64)
    w = np.zeros(4, np.uint64)
    assert lib.b200_fft(nat.ptr(a), C.c_uint32(2), nat.ptr(w)) == -3
    out = np.zeros(12, np.uint64)
    assert lib.b200_msm(C.c_uint64(1), nat.ptr(a), C.c_size_t(4), nat.ptr(out)) == -3
    with pytest.raises(nat.B200Error):
        nat.init(-1)


def test_product_does_not_import_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "ezkl_b200")):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".h", ".hpp")):
                src = open(os.path.join(dirpath, fn)).read()
                assert "oracle" not in src.replace("# oracle-free", ""), "%s mentions the oracle" % fn


def test_host_constants_match_oracle():
    assert F.FR_MODULUS == pyref.R and F.FQ_MODULUS == pyref.P
    assert F.FR_ROOT_OF_UNITY == pyref.FR_ROOT_OF_UNITY and F.FR_ZETA == pyref.FR_ZETA
    assert np.array_equal(F.fr_to_limbs(1), orc.fr_one())
    assert F.fr_from_limbs(orc.omega(17)) == pyref.omega_for(17)


def test_portable_field_ops_vs_oracle():
    L = nat.lib()
    rng = random.Random(5)
    for fid, (field, mod) in enumerate((("fr", pyref.R), ("fq", pyref.P))):
        xs = [rng.randrange(mod) for _ in range(300)] + [0, 1, mod - 1]
        ys = [rng.randrange(mod) for _ in range(300)] + [mod - 1, 0, mod - 1]
        a = np.stack([H.int_to_limbs(pyref.to_mont(x, mod)) for x in xs])
        b = np.stack([H.int_to_limbs(pyref.to_mont(y, mod)) for y in ys])
        for opi, op in enumerate(("add", "sub", "mul")):
            out = np.zeros_like(a)
            assert nat.dbg_lib().b200_debug_host_field_op(fid, opi, nat.ptr(a), nat.ptr(b), nat.ptr(out), C.c_size_t(len(xs))) == 0
            assert np.array_equal(out, orc.field_op(field, op, a, b)), (field, op)
        out = np.zeros_like(a)
        nat.dbg_lib().b200_debug_host_field_op(fid, 3, nat.ptr(a), nat.ptr(b), nat.ptr(out), C.c_size_t(len(xs)))
        assert np.array_equal(out, orc.fr_inv(a) if field == "fr" else orc.fq_inv(a))


def test_group_law_vs_oracle_including_degenerate_inputs():
    L = nat.lib()
    rng = random.Random(6)
    bases = orc.gen_bases(64, seed=9, threads=2)
    A, B = bases[:32].copy(), bases[32:].copy()
    A[0] = 0          # identity + P
    B[1] = 0          # P + identity
    A[2] = B[2]       # P + P through the mixed-add doubling branch
    n = C.c_size_t(32)
    out = np.zeros_like(A)
    nat.dbg_lib().b200_debug_host_g1_op(0, nat.ptr(A), nat.ptr(B), nat.ptr(out), n)
    assert np.array_equal(out, orc.g1_add_affine(A, B))
    nat.dbg_lib().b200_debug_host_g1_op(1, nat.ptr(A), nat.ptr(B), nat.ptr(out), n)
    assert np.array_equal(out, orc.g1_add_affine(A, A))
    K = B.copy()
    ks = [rng.randrange(1 << 20) for _ in range(32)]
    ks[3], ks[4] = 0, 1
    ks[5:16] = [2, 3, 4, 0xFFFFF, 0x55555, 0xAAAAA, 0xFFFFFFFF, 0x80000000, 0x40000000, 12, 0x30003]      # every 2-bit window digit, top windows, max
    for i, k in enumerate(ks):
        K[i, 0] = k
    nat.dbg_lib().b200_debug_host_g1_op(2, nat.ptr(A), nat.ptr(K), nat.ptr(out), n)
    assert np.array_equal(out, orc.g1_scalar_mul(A, H.fr_array(ks)))
    nat.dbg_lib().b200_debug_host_g1_op(3, nat.ptr(A), nat.ptr(B), nat.ptr(out), n)
    assert np.array_equal(out, orc.g1_add_affine(A, orc.g1_add_affine(B, B)))
    out[:] = 1
    nat.dbg_lib().b200_debug_host_g1_op(4, nat.ptr(A), nat.ptr(B), nat.ptr(out), n)
    assert not out.any()      # P + (-P) = identity = (0,0)


@pytest.mark.parametrize("c", [4, 7, 8, 13, 15, 16, 17, 20, 22, 24])
def test_signed_window_recoding(c):
    L = nat.lib()
    rng = random.Random(c)
    xs = [rng.randrange(pyref.R) for _ in range(200)] + [0, 1, pyref.R - 1, 1 << 253, (1 << c) - 1, 1 << (c - 1), (1 << (c - 1)) + 1]
    can = np.stack([H.int_to_limbs(x) for x in xs])
    W = (255 + c - 1) // c
    out = np.zeros((len(xs), W), np.int32)
    nat.dbg_lib().b200_debug_digits_host(nat.ptr(can), C.c_size_t(len(xs)), C.c_int(c), out.ctypes.data_as(C.c_void_p))
    for i, x in enumerate(xs):
        assert sum(int(out[i, w]) << (c * w) for w in range(W)) == x
        assert all(-(1 << (c - 1)) <= int(d) <= (1 << (c - 1)) for d in out[i])


def test_proving_key_reader_on_reference_fixture(tmp_path):
    """ProvingKey::read mirror against the reference's own tests/assets/pk.key, rebuilt byte for byte from tests/golden."""
    path = str(tmp_path / "pk.key")
    H.write_reference_pk(path)
    from ezkl_b200 import halo2 as h2
    pk = h2.ProvingKey.read(path, num_permutation_columns=32, num_selectors=80)
    g = H.load_pk_fixture()
    assert pk.k == 6 and len(pk.fixed_values) == 38 and len(pk.permutations) == 32
    assert pk.l0.shape == (512, 4) and pk.fixed_cosets[0].shape == (512, 4) and pk.fixed_polys[0].shape == (64, 4)
    for c in (0, 1, 5, 37):
        assert np.array_equal(pk.fixed_values[c], g["fixed_values_%d" % c])
        assert np.array_equal(pk.fixed_polys[c], g["fixed_polys_%d" % c])
        assert np.array_equal(pk.fixed_cosets[c], g["fixed_cosets_%d" % c])
    assert np.array_equal(pk.permutation_cosets[0], g["perm_cosets_0"]) and np.array_equal(pk.l_active_row, g["l_active_row"])
    with pytest.raises(nat.B200Error):
        h2.ProvingKey.read(path, num_permutation_columns=31, num_selectors=80)      # wrong layout is detected, not mis-parsed


def test_bench_reference_arm_prints_contract_json():
    """`bench.py --impl reference` (the CPU port arm the driver runs first) prints one JSON line with the contract's keys."""
    import json
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--k", "8", "--steps", "1", "--warmup", "0", "--cpu-budget", "1"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
                "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["higher_is_better"] is False and line["cpu_baseline"]["kind"] == "port"
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and "workload" in line["config"]


def test_bench_output_digits_are_exact():
    """bench.py --dump-outputs writes wire limbs as float32 16-bit digits: every bit must come back."""
    import sys
    sys.path.insert(0, ROOT)
    import bench
    a = np.random.default_rng(3).integers(0, 1 << 63, size=(50, 4), dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    a[0], a[1] = 0, np.uint64(0xFFFFFFFFFFFFFFFF)
    d = bench.wire_digits(a)
    assert d.dtype == np.float32 and d.shape == (50, 16) and d.max() <= 0xFFFF
    back = np.ascontiguousarray(d.astype(np.uint16)).view(np.uint64)
    assert np.array_equal(back, a)


@pytest.mark.gpu
def test_bench_dump_outputs_are_reproducible(tmp_path):
    """Two bench runs with different --steps dump the same outputs (seeded inputs, every step recomputes them); the line reports
    the steps that were asked for, and the dump has the trace's shapes, in float32 / float64, under 64 MB."""
    import json
    import subprocess
    import sys
    sys.path.insert(0, ROOT)
    import bench
    dumps = {}
    for steps in (2, 1):
        d = tmp_path / ("steps%d" % steps)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--k", "9", "--steps", str(steps), "--warmup", "0", "--no-cpu-baseline",
                            "--dump-outputs", str(d)], capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
        dumps[steps] = {f: np.load(d / f) for f in sorted(os.listdir(d))}
    tr = bench.TRACES[bench.CONFIG_FOR_K[9]]
    n_commits = sum(c for kind, c in bench.trace_ops(tr) if kind.startswith("msm"))
    got = dumps[1]
    assert got["commitments.npy"].shape == (n_commits, 48) and got["evaluations.npy"].shape == (tr["evals"], 16)
    assert got["quotient.npy"].shape == (tr["quotient_pieces"] << 9, 16)
    assert all(a.dtype in (np.float32, np.float64) for a in got.values()) and sum(a.nbytes for a in got.values()) <= 64 << 20
    assert dumps[2].keys() == got.keys() and all(np.array_equal(dumps[2][f], got[f]) for f in got)


def test_fp64_pipe_multiplier_vs_bigint():
    """fd.cuh host build: the 5 x 52-bit-limb Montgomery multiplication whose limb products are split with round-toward-zero
    FMAs must return a * b * 2^-260 mod N (< 2N, limbs normalised) for both fields, including the extremes of the container."""
    D = nat.dbg_lib()
    rng = random.Random(3)
    for fid, N in ((0, pyref.R), (1, pyref.P)):
        xs = [rng.getrandbits(256) for _ in range(500)] + [0, 1, N - 1, (1 << 256) - 1, N, 2 * N - 1]
        ys = [rng.getrandbits(256) for _ in range(500)] + [N - 1, (1 << 256) - 1, N - 1, (1 << 256) - 1, N, 2 * N - 1]
        a = np.stack([H.int_to_limbs(x) for x in xs])
        b = np.stack([H.int_to_limbs(y) for y in ys])
        out = np.zeros_like(a)
        assert D.b200_debug_host_fd_mul(C.c_int(fid), nat.ptr(a), nat.ptr(b), nat.ptr(out), C.c_size_t(len(xs))) == 0
        rinv = pow(1 << 260, -1, N)
        for i, (x, y) in enumerate(zip(xs, ys)):
            v = H.limbs_to_int(out[i])
            assert v % N == x * y * rinv % N and v < 2 * N, (fid, i)


def test_batched_affine_accumulation_bodies_on_host():
    """tools/experiments/msm_affine.cuh (the batched-affine accumulation EXPERIMENT, not in the product library) run on the CPU: every chunk's tree of batched-affine additions (hierarchical Montgomery trick) must equal
    the plain sum of its points — incl. repeated points (doubling), P + (-P), identity entries, negated entries, length-1 chunks."""
    L = nat.lib()
    rng = random.Random(8)
    npts = 300
    table = orc.gen_bases(npts, seed=77, threads=2)
    table[5] = 0                                            # an identity table entry
    ents, starts, lens = [], [], []
    shapes = [1, 2, 3, 4, 5, 7, 8, 16, 31, 33, 64, 100, 1, 2] + [rng.randrange(1, 40) for _ in range(80)]
    for ln in shapes:
        starts.append(len(ents))
        lens.append(ln)
        for _ in range(ln):
            ents.append(rng.randrange(npts) | (0x80000000 if rng.random() < 0.3 else 0))
    # crafted chunks: P + P, P + (-P), identity + P, P + P + P + P
    for special in ([7, 7], [9, 9 | 0x80000000], [5, 11], [13, 13, 13, 13], [5, 5], [20, 20 | 0x80000000, 21]):
        starts.append(len(ents))
        lens.append(len(special))
        ents.extend(special)
    ents = np.array(ents, dtype=np.uint32)
    starts = np.array(starts, dtype=np.uint32)
    lens = np.array(lens, dtype=np.uint32)
    out = np.zeros((len(lens), 8), np.uint64)
    assert nat.dbg_lib().b200_debug_host_affine_chunks(nat.ptr(table), ents.ctypes.data_as(C.c_void_p), C.c_size_t(len(ents)), starts.ctypes.data_as(C.c_void_p),
                                           lens.ctypes.data_as(C.c_void_p), C.c_size_t(len(lens)), nat.ptr(out)) == 0
    for c in range(len(lens)):
        acc = None
        for e in ents[starts[c]:starts[c] + lens[c]]:
            p = H.g1_unwire(table[int(e) & 0x7FFFFFFF])
            if int(e) >> 31:
                p = pyref.g1_neg(p)
            acc = pyref.g1_add(acc, p)
        assert H.g1_unwire(out[c]) == acc, (c, int(lens[c]))


def test_generated_field_arithmetic_is_verified_and_current(tmp_path):
    """fp_gen.py executes every emitted PTX instruction list (multiply, add, sub, two-product multiply, squaring) in its own
    interpreter against bigints; the committed fp_ptx.cuh must be exactly what the generator emits today."""
    import importlib.util
    gen_path = os.path.join(ROOT, "ezkl_b200", "csrc", "fp_gen.py")
    spec = importlib.util.spec_from_file_location("fp_gen", gen_path)
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    for name, mod in gen.FIELDS.items():
        counts = gen.check(name, mod, trials=300)
        assert counts[0] == 312 and counts[3] < 2 * counts[0] and counts[4] < counts[0]
    committed = open(os.path.join(ROOT, "ezkl_b200", "csrc", "fp_ptx.cuh")).read()
    for name, mod in gen.FIELDS.items():
        for fn, ins, n_in in (("mul", gen.gen_mul(mod), 2), ("mul2", gen.gen_mul2(mod), 4), ("sqr", gen.gen_sqr(mod), 1)):
            assert gen.emit_fn("%s_%s_ptx" % (name, fn), ins, n_in) in committed, "%s_%s_ptx is stale: run fp_gen.py" % (name, fn)


def test_keygen_host_logic_reproduces_reference_proving_key_bytes_on_the_cpu_backend(monkeypatch):
    """create_keys' derived vectors (src/pfsys/mod.rs:376-400) through the SAME host code the GPU test drives (ProvingKey.keygen_pk_polys,
    EvaluationDomain.keygen_l_polys: which rows l_last / the blinding rows sit on, how l_active_row is formed, which columns are
    transformed how), with the transforms redirected to the CPU oracle: byte for byte the reference pk.key's polys, extended cosets, l0,
    l_last and l_active_row (tests/golden/pk_k6_subset.npz)."""
    from ezkl_b200 import halo2 as h2
    from tests import cpu_backend as cb
    cb.patch_backend(monkeypatch)
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
    assert np.array_equal(out["l0"], pk["l0"]) and np.array_equal(out["l_last"], pk["l_last"]) and np.array_equal(out["l_active_row"], pk["l_active_row"])


def test_bench_trace_shape_matches_the_reference_fixture_proof():
    """bench.py's default op trace is shaped like the reference's own fixture proof (tests/assets/proof.json, SURVEY.md Appendix B/D4):
    114 commitments + 2 SHPLONK points, 231 evaluations; config dicts of the two bench arms are the same object shape."""
    import sys
    sys.path.insert(0, ROOT)
    import bench
    tr = bench.TRACES["conv2d_mnist"]
    ops = bench.trace_ops(tr)
    msm_cols = [c for kind, c in ops if kind.startswith("msm")]
    assert sum(msm_cols) == 114 + 2 and msm_cols[-1] == 2
    assert dict(ops)["eval"] == 231
    assert bench.n_coset_columns(tr) == tr["advice"] + tr["instance"] + tr["perm_z"] + 2 * tr["lookups"] == 107
    pairs, ntt_elts = bench.count_units(ops, 1 << 17, tr)
    assert pairs == 116 << 17 and ntt_elts == (107 << 17) + (108 << 20)
    cfg = bench.make_config(17, "conv2d_mnist")
    assert cfg["k"] == 17 and cfg["msm_pairs_per_step"] == pairs and "workload" in cfg
