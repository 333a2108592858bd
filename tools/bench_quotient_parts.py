#!/usr/bin/env python
"""evaluate_h over the whole extended domain (b200_evaluate_h) against evaluate_h one coset part at a time (b200_evaluate_h_parts), in the
host-pointer and the device-pointer form, finishing to the quotient's coefficients as a proof does.

Systems: bench.py's quotient group (32 coefficient columns and the carried partial sum h as an extended column) and tools/bench_quotient.py's
ezkl-sized system (132 coefficient columns, 436 instructions), random inputs from fixed seeds.  Before anything is timed, the two paths'
outputs on the timed inputs are compared byte for byte.  Each (system, k, form) records the device memory of one call of each path (free
memory before and after the call, in a calling thread that exits afterwards so the library's scratch is released; the box may be shared, so
other processes' allocations move these figures too) and the times of `--reps` calls, the two paths alternating.  Where the full path does
not fit on the device (k = 22 with 132 columns, k = 23) it is recorded as such and only the parts path runs.

    python tools/bench_quotient_parts.py --out profiles/r03_quotient_parts.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from ezkl_b200 import _native as nat  # noqa: E402
from ezkl_b200 import device as dev  # noqa: E402
from ezkl_b200 import evaluation as ev  # noqa: E402
from ezkl_b200 import fields as F  # noqa: E402
from ezkl_b200 import halo2 as h2  # noqa: E402

GIB = float(1 << 30)


def group_system():
    """bench.py's gate_program(32): 32 coset columns and the partial sum h (column 32)."""
    value = ev.Query(32)
    y = ev.Constant(0x1234567890ABCDEF1234567890ABCDEF)
    for t in range(32):
        a, b, c = ev.Query(t), ev.Query((t + 1) % 32, 1), ev.Query((t + 2) % 32, -1)
        value = value * y + (a * b + c * a - b)
    return ev.QuotientProgram(value), 32, 1


def ezkl_system(blocks=8):
    """tools/bench_quotient.py's system: BaseConfig blocks, a permutation in chunks of 3, one mv-lookup per two blocks, folded with y."""
    col = [0]

    def new(cnt):
        r = list(range(col[0], col[0] + cnt))
        col[0] += cnt
        return r

    terms, perm_cols, blks = [], [], []
    for _ in range(blocks):
        adv, sel = new(5), new(5)
        blks.append((adv, sel))
        terms += ev.base_op_gates(dict(zip(["ADD", "MULT", "DOTINIT", "DOT", "SUM"], sel)), adv[0:2], adv[2:4], adv[4])
        perm_cols += [adv[0], adv[2], adv[4]]
    sig = new(len(perm_cols))
    zs = new((len(perm_cols) + 2) // 3)
    l0, l_last, l_active, xcol = new(4)
    terms += ev.permutation_terms(perm_cols, sig, zs, l0, l_last, l_active, xcol, 11, 13, 3, 5)
    for b in range(0, blocks, 2):
        table, sel_l, m, phi = new(4)
        f = ev.Query(sel_l) * ev.Query(blks[b][0][1]) + (ev.Constant(1) - ev.Query(sel_l)) * ev.Constant(7)
        terms += ev.mv_lookup_terms([f], ev.Query(table), m, phi, l0, l_last, l_active, 17)
    return ev.QuotientProgram(ev.fold_y(terms, 99)), col[0], 0


def in_thread(fn):
    """Runs fn in a calling thread that exits afterwards (its library scratch is released) -> (result, device bytes the call held at its end)."""
    box = {}

    def body():
        torch.cuda.set_device(0)
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        free0 = torch.cuda.mem_get_info()[0]
        try:
            box["out"] = fn()
            torch.cuda.synchronize()
            box["used"] = free0 - torch.cuda.mem_get_info()[0]
        except (nat.B200Error, torch.cuda.OutOfMemoryError) as e:
            box["err"] = str(e).splitlines()[0][:300]
    th = threading.Thread(target=body)
    th.start()
    th.join()
    torch.cuda.empty_cache()
    return box


def full_dev(prog, coeffs, ext_cols, dom):
    """The whole-domain path on device buffers: batched coset NTTs, b200_quotient_eval_dev, the vanishing factor, the extended iNTT."""
    k, ext_k = dom.k, dom.extended_k
    N = 1 << ext_k
    z = F.FR_ZETA
    one, zeta, zeta2 = F.fr_to_limbs(1), F.fr_to_limbs(z), F.fr_to_limbs(z * z % F.FR_MODULUS)
    dv = F.fr_from_limbs(dom.extended_ifft_divisor)
    post = [F.fr_to_limbs(dv), F.fr_to_limbs(dv * z * z % F.FR_MODULUS), F.fr_to_limbs(dv * z % F.FR_MODULUS)]
    nc = coeffs.shape[0]
    cos = torch.empty((nc, N, 4), dtype=torch.int64, device="cuda")
    sub = 8
    tmp = torch.empty((sub, N, 4), dtype=torch.int64, device="cuda")
    for b0 in range(0, nc, sub):
        b = min(sub, nc - b0)
        dev.ntt(coeffs[b0:b0 + b], ext_k, dom.extended_omega, n_in=1 << k, pre=[one, zeta, zeta2], out=cos[b0:b0 + b], tmp=tmp[:b])
    out = ev.evaluate_h_device(prog, [cos[i] for i in range(nc)] + list(ext_cols), k, ext_k)
    dev.scale_cycle(out, dom.t_evaluations)
    res = dev.ntt(out, ext_k, dom.extended_omega_inv, post=post, tmp=tmp[:1])[0]
    del cos, tmp
    return res


def run_case(name, prog, ncoeff, next_, k, forms, reps, full_ok):
    dom = h2.EvaluationDomain(9, k)
    ext_k = dom.extended_k
    n, N = 1 << k, 1 << ext_k
    coeffs = dev.random_scalars(n, batch=ncoeff, seed=1000 + k)
    ext_cols = [dev.random_scalars(N, seed=2000 + k + i) for i in range(next_)]
    torch.cuda.synchronize()
    rec = {"system": name, "k": k, "ext_k": ext_k, "columns": ncoeff + next_, "coefficient_columns": ncoeff, "extended_columns": next_,
           "instructions": len(prog.instrs), "forms": {}}
    for form in forms:
        r = {}
        if form == "host":
            hc = dev.to_host(coeffs).reshape(ncoeff, n, 4)
            cols = [hc[i] for i in range(ncoeff)] + [dev.to_host(c).reshape(N, 4) for c in ext_cols]
            call_full = lambda: ev.evaluate_h_from_polys(prog, cols, dom, finish=True)
            call_parts = lambda: ev.evaluate_h_parts(prog, cols, dom, finish=True)
            same = lambda a, b: bool(np.array_equal(a, b))
        else:
            cols = [coeffs[i] for i in range(ncoeff)] + ext_cols
            call_full = lambda: full_dev(prog, coeffs, ext_cols, dom)
            call_parts = lambda: ev.evaluate_h_parts_device(prog, cols, dom, finish=True)
            same = lambda a, b: bool(torch.equal(a, b))
        parts = in_thread(call_parts)
        if "err" in parts:
            r["parts_error"] = parts["err"]
            rec["forms"][form] = r
            print(name, k, form, "parts failed:", parts["err"], flush=True)
            continue
        r["parts_device_bytes"] = parts["used"]
        full = in_thread(call_full) if full_ok else {"err": "not attempted: the full cosets exceed the device"}
        if "err" in full:
            r["full_error"] = full["err"]
        else:
            r["full_device_bytes"] = full["used"]
            r["byte_identical"] = same(full["out"], parts["out"])
            assert r["byte_identical"], "%s k=%d %s: parts output differs from the full path" % (name, k, form)
        del full, parts
        # timing: both paths in one calling thread, alternating, after one warm-up call each
        paths = [("parts", call_parts)] + ([("full", call_full)] if "full_error" not in r else [])
        times = {p: [] for p, _ in paths}

        def timed():
            torch.cuda.set_device(0)
            for _, fn in paths:
                fn()
            torch.cuda.synchronize()
            for _ in range(reps):
                for p, fn in paths:
                    t0 = time.perf_counter()
                    fn()
                    torch.cuda.synchronize()
                    times[p].append((time.perf_counter() - t0) * 1e3)
        th = threading.Thread(target=timed)
        th.start()
        th.join()
        torch.cuda.empty_cache()
        for p in times:
            r[p + "_ms"] = [round(t, 3) for t in times[p]]
            r[p + "_ms_median"] = round(statistics.median(times[p]), 3) if times[p] else None
        if times.get("full") and times["parts"]:
            r["parts_over_full"] = round(r["parts_ms_median"] / r["full_ms_median"], 3)
        rec["forms"][form] = r
        print(name, k, form, {kk: v for kk, v in r.items() if not kk.endswith("_ms")}, flush=True)
    del coeffs, ext_cols
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ks", default="17,20,22", help="k values with full vs parts")
    ap.add_argument("--big-k", type=int, default=23, help="k of the parts-only run of the 132-column system (0 = skip)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    nat.init(0)
    torch.cuda.set_device(0)
    ctx = {"device": torch.cuda.get_device_name(0), "free_bytes_at_start": torch.cuda.mem_get_info()[0], "total_bytes": torch.cuda.mem_get_info()[1]}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=60)
        ctx["nvidia_smi"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        ctx["nvidia_smi"] = "unavailable: %s" % e
    print(ctx, flush=True)
    results = []
    systems = [("bench_group_33", group_system()), ("ezkl_132", ezkl_system())]
    for k in [int(x) for x in a.ks.split(",") if x]:
        for name, (prog, nc, ne) in systems:
            N = 1 << (k + 3)
            fits = (nc + ne) * N * 32 + 4 * N * 32 < 0.8 * ctx["free_bytes_at_start"]
            results.append(run_case(name, prog, nc, ne, k, ("host", "dev"), a.reps, fits))
    if a.big_k:
        prog, nc, ne = ezkl_system()
        results.append(run_case("ezkl_132", prog, nc, ne, a.big_k, ("dev",), a.reps, False))
    doc = {"tool": "tools/bench_quotient_parts.py", "context": ctx, "reps": a.reps,
           "note": "finish=True (quotient coefficients); times are host-clock milliseconds per call ending in a device synchronise; device bytes = "
                   "free memory before minus after one call in a fresh calling thread (inputs excluded, outputs and scratch included; the box is shared)",
           "results": results}
    s = json.dumps(doc, indent=1)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
