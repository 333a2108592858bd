"""Guard ordering of the C ABI: before b200_init, every entry point declared in include/ezkl_b200.h must fail (or succeed) the
way it always has, without touching CUDA first.  One subprocess loads libezkl_b200.so, never calls b200_init, and calls each
entry twice: once with small real host buffers for every pointer argument and once with NULL for every pointer argument.
Safe on a machine with a GPU: no entry reaches CUDA before its guard."""
import json
import os
import re
import subprocess
import sys

from ezkl_b200 import _native as nat

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# entries that start or stop the library, and the four that call CUDA without a guard
SKIP = {"b200_init", "b200_init_multi", "b200_shutdown", "b200_dev_free", "b200_host_alloc", "b200_host_free", "b200_profile_read"}

NOT_INIT = (-3, "not initialised")
# name -> ((result, last-error substring) with real buffers, (result, last-error substring) with NULL pointers)
EXPECTED = {
    "b200_version": ((200, None), (200, None)),
    "b200_device_count": ((0, None), (0, None)),
    "b200_launch_count": ((0, None), (0, None)),
    "b200_last_error": (("str", None), ("str", None)),
    "b200_profile_enable": ((0, None), (0, None)),
    "b200_bases_info": ((-1, "unknown handle"), (-1, "unknown handle")),
    "b200_g1_normalize": ((0, None), (-1, "null pointer")),
    "b200_fft": (NOT_INIT, (-1, "null pointer")),
    "b200_fft_batch": (NOT_INIT, (-1, "null pointer")),
    "b200_ifft": (NOT_INIT, (-1, "null pointer")),
    "b200_ifft_batch": (NOT_INIT, (-1, "null pointer")),
    "b200_coeff_to_extended": (NOT_INIT, (-1, "null pointer")),
    "b200_coeff_to_extended_batch": (NOT_INIT, (-1, "null pointer")),
    "b200_extended_to_coeff": (NOT_INIT, (-1, "null pointer")),
}
for _name in ("b200_bases_register", "b200_bases_register_dev", "b200_bases_release", "b200_msm", "b200_msm_batch", "b200_msm_batch_dev",
              "b200_msm_sharded_dev", "b200_g1_sum_dev", "b200_g1_fft", "b200_g1_fft_dev", "b200_g1_fixed_base_mul_dev", "b200_g1_generate_dev",
              "b200_ntt_dev", "b200_ntt_sharded_dev", "b200_poly_op", "b200_poly_op_dev", "b200_poly_lincomb", "b200_poly_lincomb_dev",
              "b200_poly_scale_cycle", "b200_poly_scale_cycle_dev", "b200_poly_eval", "b200_poly_eval_batch", "b200_poly_eval_batch_dev",
              "b200_batch_invert", "b200_batch_invert_dev", "b200_prefix_scan", "b200_prefix_scan_dev", "b200_prefix_scan_batch_dev",
              "b200_kate_division", "b200_kate_division_dev", "b200_lookup_multiplicities", "b200_lookup_multiplicities_dev",
              "b200_quotient_eval", "b200_quotient_eval_dev", "b200_evaluate_h", "b200_dev_alloc", "b200_dev_alloc_on", "b200_dev_upload",
              "b200_dev_upload_async", "b200_dev_download", "b200_sync", "b200_sync_all"):
    EXPECTED[_name] = (NOT_INIT, NOT_INIT)

_PROBE = r"""
import ctypes as C, json, re, sys
lib_path, hdr_path = sys.argv[1], sys.argv[2]
skip = set(sys.argv[3].split(","))
lib = C.CDLL(lib_path)
lib.b200_last_error.restype = C.c_char_p
hdr = re.sub(r"/\*.*?\*/", "", open(hdr_path).read(), flags=re.S)
INTS = {"int": C.c_int, "size_t": C.c_size_t, "uint32_t": C.c_uint32, "uint64_t": C.c_uint64}
RESTYPES = {"int": C.c_int, "uint64_t": C.c_uint64, "const char*": C.c_char_p}
keep = []                                    # every buffer stays alive until the process ends

def buffer(nbytes=4096):
    b = C.create_string_buffer(nbytes)
    keep.append(b)
    return C.cast(b, C.c_void_p)

def pointer_array():
    arr = (C.c_void_p * 8)(*[buffer() for _ in range(8)])
    keep.append(arr)
    return C.cast(arr, C.c_void_p)

def args_for(params, null):
    argtypes, args = [], []
    for p in params:
        stars = p.count("*")
        if stars:
            argtypes.append(C.c_void_p)
            args.append(None if null else (pointer_array() if stars >= 2 else buffer()))
        else:
            t = INTS[p.replace("const ", "").split()[0]]
            argtypes.append(t)
            args.append(4)
    return argtypes, args

out = {}
for ret, name, params in re.findall(r"^(int|uint64_t|const char\*)\s+(b200_\w+)\s*\(([^)]*)\);", hdr, flags=re.M | re.S):
    if name in skip:
        continue
    params = [q.strip() for q in params.split(",") if q.strip() and q.strip() != "void"]
    fn = getattr(lib, name)
    fn.restype = RESTYPES[ret]
    res = []
    for null in (False, True):
        fn.argtypes, args = args_for(params, null)
        lib.b200_profile_enable(0)                           # leaves the thread's last error as it is
        r = fn(*args)
        if isinstance(r, bytes):
            r = "str"
        res.append([r, lib.b200_last_error().decode()])
    out[name] = res
print(json.dumps(out))
"""


def test_every_entry_point_checks_its_guard_before_cuda():
    r = subprocess.run([sys.executable, "-c", _PROBE, nat.LIB_PATH, os.path.join(ROOT, "include", "ezkl_b200.h"), ",".join(sorted(SKIP))],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    got = json.loads(r.stdout.strip().splitlines()[-1])
    assert set(got) == set(EXPECTED), "declared entries changed: %s" % sorted(set(got) ^ set(EXPECTED))
    for name, want in EXPECTED.items():
        for (rc, err), (want_rc, want_err), how in zip(got[name], want, ("real buffers", "NULL pointers")):
            assert rc == want_rc, "%s with %s returned %r, expected %r (%s)" % (name, how, rc, want_rc, err)
            if want_err is not None:
                assert want_err in err, "%s with %s: last error %r lacks %r" % (name, how, err, want_err)
