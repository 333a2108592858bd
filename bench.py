#!/usr/bin/env python
"""bench.py — prove-trace replay of the Halo2/KZG prover hot path on B200 (BASELINE.json metric: prove time (s) at k;
MSM G1 pairs/s and NTT Fr elts/s vs the HBM roofline).

A "step" is ONE proof's worth of hot-path work (SURVEY.md §3.1 stages 1-9 minus synthesize / transcript, which stay on the
CPU in Rust — see DESIGN.md): the MSMs, (i)NTTs, coset NTTs, the quotient-numerator evaluation (evaluate_h, a synthetic
gate program touching every coset column at three rotations) and the column-polynomial passes one `create_proof` issues
for a circuit of the shape named in `config.workload`, on synthetic seeded columns.
  * parity gate: BEFORE anything is timed, the exact timed inputs (the first batched MSM, the first batched iNTT, the first
                coset-NTT group, its evaluate_h group and the evaluation batch) are compared byte for byte with the CPU oracle;
                a mismatch aborts the run without printing a line (`parity_checked` in the line lists what was compared).
  * `value`   : seconds per proof with all columns resident in HBM (device entry points), CUDA-event timed.  Schedule: one
                high-priority stream in trace order, plus the iNTT / coset NTT of the witness-only columns (no transcript
                challenge feeds them) on a low-priority side stream issued by a second host thread, joined before evaluate_h;
                steps never overlap each other (`schedule` in the line; --no-overlap = everything on one stream).
  * `e2e`     : the same trace through the C ABI starting from pinned HOST buffers: each witness-derived column is uploaded
                once, later stages use the device-pointer entry points (the resident-column shim of INTEGRATION.md §2b),
                commitments are normalised on the host and evaluations read back; H2D/D2H and the host tail are timed.
  * `e2e_host_pointer`: the same trace through the HOST-POINTER entry points only (b200_msm_batch, b200_ifft_batch,
                b200_coeff_to_extended_batch, b200_quotient_eval, ...) on pageable numpy buffers: what the minimal Rust drop-in
                of INTEGRATION.md §2a binds; every operand crosses PCIe on every call.
  * `cold_start`: what one `ezkl prove` process pays before its first commit: SRS file read, both base registrations
                (upload + window-table build) and the NTT plans.
  * `roofline`: the dominant kernel (MSM bucket accumulation) against the measured HBM peak, timed with CUDA events
                inside the library on the launching stream.
  * `cpu_baseline` / `--impl reference`: the CPU restatement of halo2's Rayon algorithms (oracle/, "port") running the WHOLE
                trace for real on the box's host cores (a persistent thread pool, every op instance executed, nothing extrapolated).
--dump-outputs DIR: after the timed steps, DIR/<name>.npy holds what the last timed step computed (see dump_outputs); the inputs
are seeded, so two builds run with the same arguments can be compared output for output.
--simulate-rank-of N: ONE GPU executes rank 0's share of an N-way run (same deal, same kernels, exchanges skipped) so that a rank's
per-step kernel list can be profiled without N GPUs; the line is marked SIMULATED and is not a bench value.
N > 1 (torchrun): independent columns are dealt round-robin to ranks (strong scaling, no data-path collective inside an
op; one small all-gather of the commitments per step), timed as max over ranks; rank 0 then also times the same trace with ONE
process driving all N devices through the library's own multi-device host-pointer path (`in_process`).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# Circuit-shaped op traces (counts per proof).  Shape parameters come from the reference's own k=6 fixture proof
# (114 commitments + 2 SHPLONK points, 231 evaluations, 38 fixed / 32 permutation columns, extended domain 8n:
# SURVEY.md Appendix B/D4) held fixed while k grows; see DESIGN.md §measurement.
TRACES = {
    "conv2d_mnist": dict(advice=60, lookups=20, perm_cols=32, perm_z=6, instance=1, quotient_pieces=7, fixed=38, evals=231, ext_bits=3,
                         shplonk_sets=4),
    "accum_einsum_matmul": dict(advice=12, lookups=2, perm_cols=8, perm_z=2, instance=1, quotient_pieces=5, fixed=6, evals=60, ext_bits=3,
                                shplonk_sets=3),
}
CONFIG_FOR_K = {17: "conv2d_mnist", 20: "accum_einsum_matmul", 22: "conv2d_mnist", 9: "accum_einsum_matmul"}


def trace_ops(tr):
    """Expands a trace into op groups: (kind, count) in create_proof order."""
    A, L, Z, I, Q = tr["advice"], tr["lookups"], tr["perm_z"], tr["instance"], tr["quotient_pieces"]
    ncoset = A + I + Z + 2 * L                      # columns that go coeff -> extended coset for the quotient
    return [
        ("msm_lagrange", A),                        # stage 1: advice commitments
        ("msm_lagrange", L),                        # stage 2: lookup multiplicities m(X)
        ("batch_invert", tr["perm_cols"] + L),      # stage 3: denominators of z(X) and phi(X)
        ("prefix_product", Z),
        ("prefix_sum", L),
        ("msm_lagrange", Z + L),                    #          commitments to z's and phi's
        ("msm_coeff", 1),                           # stage 4: vanishing random polynomial
        ("intt", ncoset),                           # stage 5: Lagrange -> coefficients
        ("quotient", 1),                            # stages 6-7: ncoset coset NTTs -> evaluate_h -> divide by vanishing -> extended iNTT
        ("msm_coeff", Q),
        ("eval", tr["evals"]),                      # stage 8
        ("lincomb", tr["shplonk_sets"]),            # stage 9: SHPLONK linear combinations (npolys polynomials over the rotation sets)
        ("kate_division", tr["shplonk_sets"]),
        ("msm_coeff", 2),
    ]


def make_config(k, tname):
    """`config` of the JSON line — identical for the GPU arm and the reference arm (the driver compares them)."""
    tr = TRACES[tname]
    pairs, ntt_elts = count_units(trace_ops(tr), 1 << k, tr)
    return {"workload": "prove-trace replay, %s-shaped circuit at k=%d (MSM, NTT, evaluate_h with a synthetic gate program and poly stages of create_proof; "
                        "synthesize and transcript stay on the CPU and are not replayed)" % (tname, k),
            "k": k, "trace": tr, "msm_pairs_per_step": pairs, "ntt_elts_per_step": ntt_elts}


def n_coset_columns(tr):
    return tr["advice"] + tr["instance"] + tr["perm_z"] + 2 * tr["lookups"]


def count_units(ops, n, tr):
    pairs = sum(c for k, c in ops if k.startswith("msm")) * n
    ntt_elts = sum(c * n for k, c in ops if k == "intt") + (n_coset_columns(tr) + 1) * (n << tr["ext_bits"])
    return pairs, ntt_elts


QUOTIENT_GROUP = 32          # coset columns evaluated per evaluate_h call (partial sums carried in h)
GATE_Y = 0x1234567890ABCDEF1234567890ABCDEF


def gate_program(m):
    """Synthetic gate set over m coset columns + the running sum h (column m): for every column t one degree-2 term reading
    three columns at rotations 0 / +1 / -1, folded with y exactly like evaluate_h folds gates:  h <- h*y + (a*b + c*a - b)."""
    from ezkl_b200 import evaluation as ev
    value = ev.Query(m)
    y = ev.Constant(GATE_Y)
    for t in range(m):
        a, b, c = ev.Query(t), ev.Query((t + 1) % m, 1), ev.Query((t + 2) % m, -1)
        value = value * y + (a * b + c * a - b)
    return ev.QuotientProgram(value)


DUMP_QUOTIENT_ROWS = 1 << 19      # 32 MB of quotient digits; with the rest, a dump stays under 64 MB at every k


def wire_digits(a):
    """uint64 wire limbs [..., L] -> float32 [..., 4L]: the same bits as little-endian 16-bit digits, exact in float32, so a
    difference of one in any limb survives a float comparison."""
    a = np.ascontiguousarray(a).view(np.uint64)
    return a.view("<u2").reshape(a.shape[:-1] + (4 * a.shape[-1],)).astype(np.float32)


def dump_outputs(out_dir, commits_xyzz, evals, h):
    """Writes one step's results in the library's wire format (Montgomery limbs) through wire_digits: the commitments (normalised
    Jacobian), the evaluations, and the quotient's coefficients (all of them, or a seeded sample of DUMP_QUOTIENT_ROWS rows, whose
    row numbers go to quotient_rows.npy)."""
    import torch
    from ezkl_b200 import device as dev
    os.makedirs(out_dir, exist_ok=True)
    rows = h.shape[0]
    pick = np.arange(rows) if rows <= DUMP_QUOTIENT_ROWS else np.sort(np.random.default_rng(0xD0).choice(rows, DUMP_QUOTIENT_ROWS, replace=False))
    out = {"commitments": wire_digits(dev.normalize(commits_xyzz)),
           "evaluations": wire_digits(dev.to_host(torch.cat(evals))),
           "quotient": wire_digits(dev.to_host(h[torch.from_numpy(pick).to(h.device)])),
           "quotient_rows": pick.astype(np.float64)}
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons while the timed regions run: ONE long-lived `nvidia-smi -lms 100` process (started
    before the warm-up so its start-up cost is outside the timed region); rows are stamped on arrival and only those that fall
    inside a marked region are summarised."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, device):
        super().__init__(daemon=True)
        self.device, self.rows, self.regions, self.proc = device, [], [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                parts = [x.strip() for x in line.strip().split(",")]
                if len(parts) >= 8:
                    self.rows.append((time.time(), parts))
        except Exception:
            pass

    def mark(self, t0, t1):
        self.regions.append((t0, t1))

    def summary(self):
        time.sleep(0.15)
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=3)
        inside = [r for (ts, r) in self.rows if any(t0 <= ts <= t1 + 0.1 for t0, t1 in self.regions)] or [r for _, r in self.rows]
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(float(r[1]) for r in inside)
        reasons = set()
        for r in inside:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(inside[0][2]), "power_w_max": max(float(r[3]) for r in inside),
                "reasons": sorted(reasons), "samples": len(inside)}


# ---------------------------------------------------------------------------------------------------------------
# GPU arm
def run_b200(args):
    import torch
    import torch.distributed as dist
    from ezkl_b200 import _native as nat
    from ezkl_b200 import device as dev
    from ezkl_b200 import fields as F
    from ezkl_b200 import halo2 as h2
    from ezkl_b200 import parallel as par

    rank, world, local = par.init_distributed("nccl" if args.gpus > 1 else None)
    assert world == args.gpus, "launch with torchrun --nproc-per-node %d" % args.gpus
    sim = args.simulate_rank_of > 1            # profiling aid: this ONE GPU plays rank 0 of an N-way run (same deal, same kernels, exchanges skipped)
    if sim:
        assert world == 1, "--simulate-rank-of runs on one GPU"
        world = args.simulate_rank_of
    torch.cuda.set_device(local)
    nat.init(local)
    # all work of the trace is enqueued on one high-priority stream (the side stream of the two-stream schedule has the lowest priority,
    # so its transforms only take what the main chain leaves idle); CUDA events below are recorded on this stream
    prio_main, prio_side = [int(x) for x in os.environ.get("BENCH_STREAM_PRIORITIES", "-1,0").split(",")]      # tuning knob (A/B runs)
    torch.cuda.set_stream(torch.cuda.Stream(priority=prio_main))
    k = args.k
    n = 1 << k
    tname = args.trace or CONFIG_FOR_K.get(k, "conv2d_mnist")
    tr = TRACES[tname]
    ops = trace_ops(tr)
    ext_k = k + tr["ext_bits"]
    dom = h2.EvaluationDomain((1 << tr["ext_bits"]) + 1, k)
    assert dom.extended_k == ext_k

    # ---- cold start (what one `ezkl prove` process pays before its first commit): SRS file -> host -> device -> window tables,
    #      then the NTT plans.  The synthetic SRS is generated on the device and written to disk first (untimed).
    import tempfile
    srs_path = os.path.join(tempfile.gettempdir(), "b200_bench_srs_k%d_r%d.bin" % (k, rank))
    _pts = torch.stack([dev.generate_bases(n, seed=0xE2C1B200), dev.generate_bases(n, seed=0xE2C1B201)])
    dev.to_host(_pts).tofile(srs_path)
    del _pts
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    srs_host = np.fromfile(srs_path, dtype=np.uint64).reshape(2, n, 8)
    t1 = time.perf_counter()
    g_lag = h2.Bases(srs_host[0])            # b200_bases_register: upload + table build, synchronous
    g_coef = h2.Bases(srs_host[1])
    t2 = time.perf_counter()
    _probe = dev.random_scalars(n, batch=1, seed=5)
    dev.ntt(_probe, k, dom.omega_inv, post=[dom.ifft_divisor])
    _e = dev.ntt(_probe, ext_k, dom.extended_omega, n_in=n, pre=[F.fr_to_limbs(1), F.fr_to_limbs(F.FR_ZETA), F.fr_to_limbs(F.FR_ZETA * F.FR_ZETA % F.FR_MODULUS)])
    dev.ntt(_e, ext_k, dom.extended_omega_inv)
    torch.cuda.synchronize()
    t3 = time.perf_counter()
    del _probe, _e
    os.unlink(srs_path)
    _info = g_lag.info()
    cold = {"windows": _info["windows"], "srs_read_s": round(t1 - t0, 4), "bases_register_s": round(t2 - t1, 4), "ntt_plans_s": round(t3 - t2, 4), "total_s": round(t3 - t0, 4),
            "what": "np.fromfile of the 2 x n x 64 B SRS vectors; b200_bases_register x 2 (H2D + window-table build, c=%d W=%d); first iNTT(k), coset NTT(ext_k), "
                    "extended iNTT(ext_k) incl. their twiddle tables" % (_info["window_bits"], _info["windows"])}

    # ---- synthetic inputs (seeded), resident on the device and mirrored in pinned host memory for the e2e leg
    ncols = max(c for _, c in ops if True)
    ncols = min(ncols, 64)                                      # column pool; ops cycle through it
    cols = dev.random_scalars(n, batch=ncols, seed=1234 + rank)
    tmp_n = torch.empty((ncols, n, 4), dtype=torch.int64, device="cuda")
    out_n = torch.empty((ncols, n, 4), dtype=torch.int64, device="cuda")
    xs = dev.to_host(dev.random_scalars(ncols, seed=99))
    one = F.fr_to_limbs(1)
    ones_b = np.ascontiguousarray(np.tile(one, (64, 1)))
    zeta, zeta2 = F.fr_to_limbs(F.FR_ZETA), F.fr_to_limbs(F.FR_ZETA * F.FR_ZETA % F.FR_MODULUS)
    d = F.fr_from_limbs(dom.extended_ifft_divisor)
    post_ext = [F.fr_to_limbs(d), F.fr_to_limbs(d * F.FR_ZETA * F.FR_ZETA % F.FR_MODULUS), F.fr_to_limbs(d * F.FR_ZETA % F.FR_MODULUS)]
    host_cols = torch.empty((ncols, n, 4), dtype=torch.int64).pin_memory()
    host_cols.copy_(cols.cpu())
    host_evals = torch.empty((max(ncols, 256), 4), dtype=torch.int64).pin_memory()

    def mine(count, base):
        """op instances of one group owned by this rank (round-robin over a running global index)."""
        return [i for i in range(count) if par.column_owner(base + i, world) == rank]

    from ezkl_b200 import evaluation as ev
    ncoset = n_coset_columns(tr)
    log_g = world.bit_length() - 1
    assert world == 1 << log_g and world <= (1 << tr["ext_bits"]), "quotient stage: world must be a power of two <= 2^ext_bits"
    N_ext = 1 << ext_k
    slab = N_ext // world
    group = QUOTIENT_GROUP if ext_k <= 23 else 16
    programs = {}
    d_ext = 1 << tr["ext_bits"]
    tinv_local = np.ascontiguousarray(np.stack([dom.t_evaluations[(rank + world * t) % d_ext] for t in range(max(1, d_ext // world))]))

    coll = {"on": False, "events": []}

    def timed_collective(fn):
        """Runs a torch.distributed call; while the profiling pass is on, brackets it with CUDA events on the current stream."""
        if not coll["on"]:
            return fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = fn()
        e1.record()
        coll["events"].append((e0, e1))
        return r

    # ---- two-stream schedule -------------------------------------------------------------------------------------------------
    # The iNTT and coset NTT of a witness-only column (advice, instance) depend on no transcript challenge, so a prover may run them any
    # time after witness generation.  The MSM phases spend ~11 ms of a k = 17 step in latency-bound kernels (digit recoding, bucket
    # reduction: few warps, the multiply pipe mostly idle), so those transforms are enqueued from a second host thread on a low-priority
    # side stream and fill the idle pipe; the quotient stage waits for them.  Nothing of step i+1 starts before step i has finished
    # (the side stream waits for an event recorded at the start of the step; the step ends by joining the side stream).
    n_early = tr["advice"] + tr["instance"]                      # coset columns [0, n_early) are witness-only
    q_groups = []
    for g0 in range(0, ncoset, group):
        gcols = list(range(g0, min(ncoset, g0 + group)))
        my = [j for j in gcols if par.column_owner(j, world) == rank]
        q_groups.append((gcols, my, len([j for j in my if j < n_early])))
    my_ext_bytes = sum(len(my) for _, my, _ in q_groups) * N_ext * 32
    overlap = (not args.no_overlap) and my_ext_bytes <= (24 << 30)
    ov = {"bufs": None}
    if overlap:
        import concurrent.futures
        ov["pool"] = concurrent.futures.ThreadPoolExecutor(1)
        ov["stream"] = torch.cuda.Stream(priority=prio_side)    # default: lowest priority; the main work runs on a high-priority stream
        ov["start"], ov["done"] = torch.cuda.Event(), torch.cuda.Event()
        ov["bufs"] = [torch.empty((len(my), N_ext, 4), dtype=torch.int64, device="cuda") for _, my, _ in q_groups]
        ne_max = max([ne for _, _, ne in q_groups] + [1])
        ov["tmp"] = torch.empty((ne_max, N_ext, 4), dtype=torch.int64, device="cuda")
        ov["side_out"] = torch.empty((ncols, n, 4), dtype=torch.int64, device="cuda")
        ov["side_tmp"] = torch.empty((ncols, n, 4), dtype=torch.int64, device="cuda")

    EARLY_CHUNK = 8          # columns per side-stream call when the columns are still arriving over PCIe (e2e leg)

    def early_transforms(cols_, n_intt_early, ready):
        """Side thread: iNTT of this rank's witness-only columns, then their coset NTTs straight into the quotient stage's buffers.
        ready(slot) -> the CUDA event after which pool slot `slot` holds its column (e2e leg: the witness is still being uploaded, so the
        work is cut into EARLY_CHUNK-column calls that start as soon as their columns have landed), or None when everything is resident."""
        torch.cuda.set_device(local)
        with torch.cuda.stream(ov["stream"]):
            ov["stream"].wait_event(ov["start"])
            step_cols = EARLY_CHUNK if ready is not None else ncols
            done = 0
            while done < n_intt_early:
                b = min(n_intt_early - done, step_cols, ncols - done % ncols)
                lo = done % ncols
                if ready is not None:
                    ov["stream"].wait_event(ready(lo + b - 1))
                dev.ntt(cols_[lo:lo + b], k, dom.omega_inv, post=[dom.ifft_divisor], out=ov["side_out"][lo:lo + b], tmp=ov["side_tmp"][lo:lo + b])
                done += b
            for gi, (gcols, my, ne) in enumerate(q_groups):
                for a0 in range(0, ne, step_cols if ready is not None else max(ne, 1)):
                    sub = my[a0:min(ne, a0 + (step_cols if ready is not None else ne))]
                    if ready is not None:
                        ov["stream"].wait_event(ready(max(j % ncols for j in sub)))
                    src = torch.stack([cols_[j % ncols] for j in sub])
                    dev.ntt(src, ext_k, dom.extended_omega, n_in=n, pre=[one, zeta, zeta2], out=ov["bufs"][gi][a0:a0 + len(sub)], tmp=ov["tmp"][:len(sub)])
            ov["done"].record(ov["stream"])

    def quotient_stage(get_col, put_h, early=False):
        """Stages 6-7.  Coset NTTs are dealt by column; evaluate_h runs row-cyclic (row idx on rank idx mod world): since
        world divides 2^ext_bits every Rotation(r) = r * 2^ext_bits rows stays on its rank, so the only exchange is one
        all-to-all per column group; h slabs are all-gathered once for the single extended iNTT on rank 0.  With early=True the
        witness-only columns of every group were already transformed on the side stream (early_transforms)."""
        h = torch.zeros((slab, 4), dtype=torch.int64, device="cuda")
        if early:
            torch.cuda.current_stream().wait_event(ov["done"])
        for gi, (gcols, my, ne) in enumerate(q_groups):
            if early:
                ext_my = ov["bufs"][gi]
                if len(my) > ne:
                    src = torch.stack([get_col(j) for j in my[ne:]])
                    dev.ntt(src, ext_k, dom.extended_omega, n_in=n, pre=[one, zeta, zeta2], out=ext_my[ne:])
            elif my:
                src = torch.stack([get_col(j) for j in my])
                ext_my = dev.ntt(src, ext_k, dom.extended_omega, n_in=n, pre=[one, zeta, zeta2])
            else:
                ext_my = torch.empty((0, N_ext, 4), dtype=torch.int64, device="cuda")
            if world > 1:
                packed = ext_my.view(len(my), slab, world, 4).permute(2, 0, 1, 3).contiguous()      # ONE strided copy: [destination rank][column][row][limb]
                send = [packed[s_] for s_ in range(world)]
                counts = [len([j for j in gcols if par.column_owner(j, world) == q]) for q in range(world)]
                recv = [torch.empty((counts[q], slab, 4), dtype=torch.int64, device="cuda") for q in range(world)]
                if sim:     # no peers: the packing copies above are kept, the received slabs are stand-ins cut from this rank's own columns
                    pool_ = torch.cat(send) if my else torch.zeros((1, slab, 4), dtype=torch.int64, device="cuda")
                    recv = [pool_[torch.arange(counts[q], device="cuda") % pool_.shape[0]] if counts[q] else recv[q] for q in range(world)]
                else:
                    timed_collective(lambda: dist.all_to_all(recv, send))
                by_col = {}
                for q in range(world):
                    for i_, j in enumerate([j for j in gcols if par.column_owner(j, world) == q]):
                        by_col[j] = recv[q][i_]
                slabs = [by_col[j] for j in gcols]
            else:
                slabs = [ext_my[i_] for i_ in range(len(my))]
            m = len(gcols)
            if m not in programs:
                programs[m] = gate_program(m)
            h = ev.evaluate_h_device(programs[m], slabs + [h], k, ext_k - log_g)
        dev.scale_cycle(h, tinv_local)
        if world > 1:
            parts = [torch.empty_like(h) for _ in range(world)]
            if sim:
                parts = [h] * world
            else:
                timed_collective(lambda: dist.all_gather(parts, h))
            full = torch.stack(parts, dim=1).reshape(1, N_ext, 4).contiguous()      # idx = t*world + rank
        else:
            full = h.view(1, N_ext, 4)
        if rank == 0:
            coeff = dev.ntt(full, ext_k, dom.extended_omega_inv, post=post_ext)
            if put_h is not None:
                put_h(coeff[0, : tr["quotient_pieces"] * n])

    commits = []
    commit_counts = [0] * world
    _g = 0
    for _kind, _count in ops:
        if _kind.startswith("msm"):
            for _i in range(_count):
                commit_counts[par.column_owner(_g + _i, world)] += 1
        _g += _count

    evals = []
    quotient = {}
    npolys_total = tr["advice"] + tr["fixed"] + tr["perm_cols"] + tr["perm_z"] + 2 * tr["lookups"] + 1 + tr["quotient_pieces"]
    lin_scalars = np.ascontiguousarray(np.tile(xs, (npolys_total // ncols + 1, 1))[:npolys_total])

    def step_device(pool=None, ready=None, serial=False, main_wait=None):
        """One proof's trace with device-resident columns (pool defaults to the resident synthetic columns).  serial=True runs the
        whole trace on one stream in trace order (the per-kernel-class profiling pass needs non-overlapping kernels)."""
        cols_ = cols if pool is None else pool
        commits.clear()
        evals.clear()
        two = overlap and not serial
        fut = None
        n_intt_early = 0
        if two:
            g_ = 0
            for kind_, count_ in ops:
                if kind_ == "intt":
                    n_intt_early = len([i for i in mine(count_, g_) if i < n_early])
                g_ += count_
            ov["start"].record(torch.cuda.current_stream())
            fut = ov["pool"].submit(early_transforms, cols_, n_intt_early, ready)
        if main_wait is not None:          # e2e leg: the commit chain needs the first batch of columns; the side stream (released above) does not
            torch.cuda.current_stream().wait_event(main_wait)
        gidx = 0
        for kind, count in ops:
            m = len(mine(count, gidx)) if kind != "quotient" else 1     # the quotient stage is cooperative: every rank takes part
            if kind == "intt":
                m -= n_intt_early                                         # those run on the side stream
            gidx += count
            done = 0
            while done < m:
                b = min(m - done, ncols)
                v = cols_[:b]
                if kind == "msm_lagrange":
                    commits.append(dev.msm_batch(g_lag, v))
                elif kind == "msm_coeff":
                    commits.append(dev.msm_batch(g_coef, v))
                elif kind == "batch_invert":
                    out_n[:b].copy_(v)
                    dev.batch_invert(out_n[:b])
                elif kind == "prefix_product":
                    for i in range(b):
                        dev.prefix_scan(v[i], one, True, out=out_n[i])
                elif kind == "prefix_sum":          # the lookups' grand sums are independent of each other: one batched call
                    dev.prefix_scan_batch(v, ones_b[:b], False, out=out_n[:b])
                elif kind == "intt":
                    dev.ntt(v, k, dom.omega_inv, post=[dom.ifft_divisor], out=out_n[:b], tmp=tmp_n[:b])
                elif kind == "quotient":
                    if fut is not None:
                        fut.result()                  # the side thread has ENQUEUED everything (its done event is recorded); no device sync
                        fut = None
                    quotient_stage(lambda j: cols_[j % ncols], lambda h: quotient.update(h=h), early=two)
                elif kind == "eval":
                    evals.append(dev.eval_batch(v, xs[:b]))
                elif kind == "lincomb":
                    per_set = max(1, npolys_total // tr["shplonk_sets"])
                    for i in range(b):
                        dev.lincomb([cols_[j % ncols] for j in range(per_set)], lin_scalars[:per_set], out=out_n[i])
                elif kind == "kate_division":
                    for i in range(b):
                        dev.kate_division(v[i], xs[i], out=out_n[i][: n - 1])
                done += b
        pts = torch.cat(commits) if commits else torch.zeros((0, 16), dtype=torch.int64, device="cuda")
        if world > 1 and not sim:
            timed_collective(lambda: par.allgather_columns(pts, commit_counts))      # per-rank counts follow from the deal: no size exchange, no host sync
        return pts

    L = nat.lib()
    import ctypes as C
    n_inputs = tr["advice"] + tr["instance"] + tr["lookups"] + 1      # witness-derived columns that exist only on the host before a proof
    e2e_pool = torch.empty((max(ncols, n_inputs), n, 4), dtype=torch.int64, device="cuda")
    for _s in range(0, e2e_pool.shape[0], ncols):      # valid uniform scalars everywhere: slots a rank does not upload into must not be zeros
        e2e_pool[_s:_s + ncols].copy_(cols[: min(ncols, e2e_pool.shape[0] - _s)])
    upload_stream = torch.cuda.Stream()
    upload_first = torch.cuda.Event()
    upload_done = torch.cuda.Event()
    upload_chunk_ev = [torch.cuda.Event() for _ in range(e2e_pool.shape[0] // 8 + 2)]

    def step_host():
        """End to end through the C ABI from HOST buffers: every witness-derived column crosses PCIe once (b200_dev_upload from
        pinned memory into a device-resident column), all later stages use the device-pointer entry points, and the step's
        results come back to the host: commitments (XYZZ -> b200_g1_normalize on the host) and the evaluations."""
        my_inputs = [i for i in range(n_inputs) if par.column_owner(i, world) == rank] if world > 1 else list(range(n_inputs))
        h2d = d2h = 0
        # uploads are enqueued on a side stream in column order; the compute stream waits only for the columns the trace reads
        # (the first `ncols` slots), so the tail of the witness upload overlaps the first commit batch
        with torch.cuda.stream(upload_stream):
            for slot, i in enumerate(my_inputs):
                nat.check(L.b200_dev_upload_async(nat.dev(e2e_pool[slot].data_ptr()), C.c_void_p(host_cols[i % ncols].data_ptr()), C.c_size_t(n * 32),
                                                  C.c_void_p(upload_stream.cuda_stream)))
                h2d += n * 32
                if (slot + 1) % EARLY_CHUNK == 0 or slot == len(my_inputs) - 1:
                    upload_chunk_ev[slot // EARLY_CHUNK].record(upload_stream)
                if slot == min(ncols, len(my_inputs)) - 1:
                    upload_first.record(upload_stream)
            upload_done.record(upload_stream)
        n_up = len(my_inputs)
        # slot -> the event after which it is on the device (slots past the uploaded ones are resident stand-ins: the last event covers them)
        ready = (lambda slot: upload_chunk_ev[min(slot, n_up - 1) // EARLY_CHUNK]) if n_up else None
        pts = step_device(e2e_pool, ready=ready, main_wait=upload_first)
        torch.cuda.current_stream().wait_event(upload_done)
        jac = dev.normalize(pts)                                  # D2H of the XYZZ partials + host normalisation
        d2h += pts.numel() * 8
        for e in evals:
            host_evals[: e.shape[0]].copy_(e)
            d2h += e.numel() * 8
        torch.cuda.synchronize()
        return h2d, d2h, jac

    # ---- parity gate: the exact timed inputs against the CPU oracle, before anything is timed ---------------------------------
    def parity_gate():
        from oracle import oracle as orc
        th = max(1, orc.host_threads() // world)
        checked = []

        def same(got, exp, what):
            if not np.array_equal(np.asarray(got), np.asarray(exp)):
                raise SystemExit("bench.py: PARITY GATE FAILED on rank %d: %s differs from the CPU oracle — no number is reported" % (rank, what))

        # (1) the first commit batch of the trace: b columns x 2^k against g_lagrange, the registered window
        b = min(len(mine(tr["advice"], 0)), ncols)
        jac = dev.normalize(dev.msm_batch(g_lag, cols[:b]))
        hc = dev.to_host(cols[:max(b, 1)])
        for i in range(b):
            same(jac[i, :8], orc.msm(hc[i], srs_host[0], th), "MSM column %d of the %d x 2^%d batch" % (i, b, k))
        checked.append("msm_batch %d x 2^%d (c=%d)" % (b, k, _info["window_bits"]))
        # (2) the iNTT batch
        bi = min(len(mine(ncoset, 0)), ncols, 8)
        co = dev.to_host(dev.ntt(cols[:bi], k, dom.omega_inv, post=[dom.ifft_divisor]))
        for i in range(bi):
            same(co[i], orc.lagrange_to_coeff(hc[i] if i < hc.shape[0] else dev.to_host(cols[i]), k, th), "iNTT column %d" % i)
        checked.append("intt_batch %d x 2^%d" % (bi, k))
        # (3) the first coset-NTT group of the quotient stage and (4) its evaluate_h group, on this rank's rows
        gcols = list(range(0, min(ncoset, group)))
        my = [j for j in gcols if par.column_owner(j, world) == rank]
        src = torch.stack([cols[j % ncols] for j in my])
        ext_my = dev.ntt(src, ext_k, dom.extended_omega, n_in=n, pre=[one, zeta, zeta2])
        ext_h = dev.to_host(ext_my)
        for i_, j in enumerate(my):
            same(ext_h[i_], orc.coeff_to_extended(dev.to_host(cols[j % ncols]), ext_k, th), "coset NTT of column %d (2^%d -> 2^%d)" % (j, k, ext_k))
        checked.append("coset_ntt_batch %d x 2^%d" % (len(my), ext_k))
        if world == 1:
            m = len(gcols)
            prog = programs.setdefault(m, gate_program(m))
            h0 = dev.random_scalars(N_ext, seed=4242)
            got = dev.to_host(ev.evaluate_h_device(prog, [ext_my[i_] for i_ in range(m)] + [h0], k, ext_k))
            loads, consts, pr = prog.arrays()
            exp = orc.quotient_eval([ext_h[i_] for i_ in range(m)] + [dev.to_host(h0)], k, ext_k, loads, consts, pr, th)
            same(got, exp, "evaluate_h group (%d columns + running sum, 2^%d rows, %d instructions)" % (m, ext_k, pr.shape[0]))
            checked.append("quotient_eval %d columns x 2^%d" % (m + 1, ext_k))
        # (5) the evaluation batch
        be = min(ncols, 16)
        evs = dev.to_host(dev.eval_batch(cols[:be], xs[:be]))
        hce = dev.to_host(cols[:be])
        for i in range(be):
            same(evs[i], orc.eval_polynomial(hce[i], xs[i]), "evaluation %d" % i)
        checked.append("eval_batch %d x 2^%d" % (be, k))
        torch.cuda.synchronize()
        return checked

    # ---- the same trace through the HOST-POINTER entry points only, on pageable numpy buffers (INTEGRATION.md §2a) -------------
    hp = {}

    def step_host_pointer():
        if not hp:
            hp["cols"] = [np.array(host_cols[i].numpy().view(np.uint64), copy=True) for i in range(ncols)]       # pageable copies
            hp["xs"] = np.array(xs, copy=True)
        pc, xh = hp["cols"], hp["xs"]
        pick = lambda cnt: [pc[i % ncols] for i in range(cnt)]
        h2d = d2h = 0
        results = []
        for kind, count in ops:
            if kind == "msm_lagrange" or kind == "msm_coeff":
                results.append(h2.best_multiexp_batch(pick(count), g_lag if kind == "msm_lagrange" else g_coef))
                h2d += count * n * 32; d2h += count * 128
            elif kind == "batch_invert":
                for c_ in pick(count):
                    h2.batch_invert(c_)
                h2d += count * n * 32; d2h += count * n * 32
            elif kind in ("prefix_product", "prefix_sum"):
                for c_ in pick(count):
                    h2.prefix_scan(c_, one, kind == "prefix_product")
                h2d += count * n * 32; d2h += count * n * 32
            elif kind == "intt":
                hp["coeffs"] = dom.lagrange_to_coeff_batch(pick(count))
                h2d += count * n * 32; d2h += count * n * 32
            elif kind == "quotient":
                coeffs = hp["coeffs"]
                hq = np.zeros((N_ext, 4), np.uint64)
                for g0 in range(0, ncoset, group):
                    m = min(group, ncoset - g0)
                    last = g0 + group >= ncoset
                    prog = programs.setdefault(m, gate_program(m))
                    # b200_evaluate_h: coefficient columns in (n each), the running sum as an extended column; the last group also divides by
                    # the vanishing polynomial and returns the quotient's coefficients
                    hq = ev.evaluate_h_from_polys(prog, [coeffs[(g0 + j) % len(coeffs)] for j in range(m)] + [hq], dom, finish=last)
                    h2d += m * n * 32 + N_ext * 32; d2h += N_ext * 32
                hp["h"] = hq[: tr["quotient_pieces"] * n]
            elif kind == "eval":
                done = 0
                while done < count:
                    b = min(count - done, ncols)
                    results.append(h2.eval_polynomial_batch(pc[:b], xh[:b]))
                    h2d += b * n * 32; d2h += b * 32
                    done += b
            elif kind == "lincomb":
                per_set = max(1, npolys_total // tr["shplonk_sets"])
                for _ in range(count):
                    h2.poly_lincomb(pick(per_set), lin_scalars[:per_set])
                h2d += count * per_set * n * 32; d2h += count * n * 32
            elif kind == "kate_division":
                for i, c_ in enumerate(pick(count)):
                    h2.kate_division(c_, xh[i])
                h2d += count * n * 32; d2h += count * n * 32
        return h2d, d2h

    def barrier():
        if world > 1 and not sim:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1 or sim:
            return ms
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    if args.profile_one_step:          # for `ncu`: setup + exactly one device-resident step, nothing else
        step_device()
        torch.cuda.synchronize()
        print("one step done")
        return

    parity_ops = None
    if not args.no_parity_gate:
        parity_ops = parity_gate()
        barrier()

    # ---- device-resident timing (library-side event profiling OFF: nothing but the kernels in the timed region)
    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(args.warmup):
        step_device()
    barrier()
    t_reg0 = time.time()
    l0 = nat.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        pts = step_device()
    e1.record()
    issue_ms = (time.time() - t_reg0) * 1e3 / args.steps     # host time to ENQUEUE a step (close to ms_per_step means the host issue rate is the limiter)
    barrier()
    sampler.mark(t_reg0, time.time())
    launches = nat.launch_count() - l0
    ms_dev = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, pts, evals, quotient["h"])
    # ---- same steps again with per-kernel-class CUDA events (roofline leg; not part of `value`)
    nat.check(L.b200_profile_enable(1))
    coll["on"] = True
    for _ in range(args.steps):
        step_device(serial=True)       # one stream, trace order: per-class event times must not overlap
    barrier()
    coll["on"] = False
    coll_ms = sum(a.elapsed_time(b) for a, b in coll["events"]) / args.steps
    prof = {}
    for cls, name in ((0, "msm_accumulate"), (1, "msm_total"), (2, "ntt"), (4, "msm_recode"), (5, "msm_tail"), (6, "quotient_eval")):
        ms, cnt = C.c_double(0), C.c_uint64(0)
        nat.check(L.b200_profile_read(cls, C.byref(ms), C.byref(cnt)))
        prof[name] = (ms.value, cnt.value)
    nat.check(L.b200_profile_enable(0))

    # ---- end-to-end (host buffers through the C ABI)
    e2e_steps = max(1, min(args.steps, 3))
    step_host()
    barrier()
    t0 = time.perf_counter()
    t_reg0 = time.time()
    for _ in range(e2e_steps):
        h2d, d2h, _ = step_host()
    barrier()
    ms_e2e = max_over_ranks((time.perf_counter() - t0) * 1e3) / e2e_steps
    sampler.mark(t_reg0, time.time())
    clocks = sampler.summary()

    # ---- the host-pointer (pageable) path of the minimal drop-in; one warm-up + one or two timed steps (it is PCIe bound)
    e2e_hp = None
    if world == 1 and not args.no_host_pointer_e2e and ext_k <= 23:
        step_host_pointer()
        hp_steps = 2 if k <= 18 else 1
        t0 = time.perf_counter()
        for _ in range(hp_steps):
            hp_h2d, hp_d2h = step_host_pointer()
        e2e_hp = {"value": round((time.perf_counter() - t0) / hp_steps, 6), "unit": "s", "h2d_bytes_per_step": int(hp_h2d), "d2h_bytes_per_step": int(hp_d2h), "steps": hp_steps,
                  "how": "host-pointer entry points only (b200_msm_batch, b200_ifft_batch, b200_evaluate_h on coefficient columns, b200_poly_eval_batch, ...) on "
                         "pageable numpy buffers; every operand and result crosses PCIe on every call (INTEGRATION.md §2a)"}
    # ---- N > 1: ONE process (rank 0) owning all N devices through b200_init_multi, same host-pointer trace; the library deals
    #      columns / splits bases / shards transforms itself (device workers).  The other ranks idle on the rendezvous store.
    in_process = None
    if world > 1 and not sim and not args.no_host_pointer_e2e and ext_k <= 23:
        store = dist.distributed_c10d._get_default_store()
        if rank == 0:
            try:
                g_lag.release(); g_coef.release()
                nat.shutdown()
                nat.check(L.b200_init_multi(C.c_int(world)))
                nat._inited = True
                g_lag, g_coef = h2.Bases(srs_host[0]), h2.Bases(srs_host[1])
                step_host_pointer()
                t0 = time.perf_counter()
                hp_h2d, hp_d2h = step_host_pointer()
                in_process = {"value": round(time.perf_counter() - t0, 6), "unit": "s", "n_devices": world, "h2d_bytes_per_step": int(hp_h2d), "d2h_bytes_per_step": int(hp_d2h),
                              "how": "one process, b200_init_multi(%d): the host-pointer trace with the library dealing batch columns over its device workers "
                                     "(MSM, iNTT, coset NTT, evaluation batches); evaluate_h and the single-column stages run on device 0" % world}
            except Exception as exc:      # never lose the main line to the extra figure
                in_process = {"error": str(exc)[:300]}
            store.set("b200_inproc_done", "1")
        else:
            store.wait(["b200_inproc_done"])

    pairs, ntt_elts = count_units(ops, n, tr)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    # dominant kernel: MSM bucket accumulation.  Algorithmic bytes = 32 B scalar + 64/b B shared base per pair
    # (SURVEY.md §8d), per launch = pairs in that launch; summed over the step and divided by the summed kernel time.
    my_msm_cols = 0
    gidx = 0
    for kind, count in ops:
        if kind.startswith("msm"):
            my_msm_cols += len(mine(count, gidx))
        gidx += count
    acc_ms, acc_cnt = prof["msm_accumulate"]
    win = cold["windows"]                           # windows per scalar = bucket additions per (scalar, base) pair
    launch_cols = my_msm_cols * args.steps / max(acc_cnt, 1)
    alg_bytes_per_launch = launch_cols * n * (32.0 + 64.0 / max(launch_cols, 1.0))
    achieved = alg_bytes_per_launch / ((acc_ms / max(acc_cnt, 1)) * 1e-3) / 1e9 if acc_ms > 0 else 0.0
    # DRAM traffic of the dominant kernel from the committed `ncu --set full` capture of this same command (k = 17 only)
    traffic = None
    try:
        cap_path = os.path.join(ROOT, "profiles", "r02_ncu_full_bench_step_k17.json")
        if not os.path.exists(cap_path):
            cap_path = os.path.join(ROOT, "profiles", "r01_ncu_full_bench_step_k17.json")
        cap = json.load(open(cap_path))["k_accumulate"]
        if k == 17 and tname == "conv2d_mnist" and world == 1:
            rd, wr = cap["dram__bytes_read.sum"]["per_launch"], cap["dram__bytes_write.sum"]["per_launch"]
            traffic = int(sum(rd + wr) * 1e9 / len(rd))
    except Exception:
        pass
    msm_ms = prof["msm_total"][0] / args.steps
    ntt_ms = prof["ntt"][0] / args.steps
    line = {
        "metric": "prove_time_s", "value": round(ms_dev / 1e3, 6), "unit": "s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms_dev, 3), "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
        "dtype": "u32 limbs (254-bit Montgomery integers mod BN254 r/p)", "data": "synthetic",
        "config": make_config(k, tname),
        "parallelism": ("columns round-robin over %d GPU(s), one process per GPU" % world) if not sim else
                       ("SIMULATED rank 0 of %d on one GPU: that rank's share of every stage, exchanges skipped — a profiling aid, not a bench value" % world),
        "host_issue_ms_per_step": round(issue_ms, 3),
        "schedule": ("two streams: iNTT + coset NTT of the %d witness-only columns on a low-priority side stream (second host thread) while the commitment phases run; "
                     "joined before evaluate_h; steps do not overlap each other" % n_early) if overlap else "one stream, trace order",
        "l2": "inputs larger than L2: %d MB of columns + %d MB tables per step" % (ncols * n * 32 >> 20, (2 * n * 64 * win) >> 20),
        "parity_checked": parity_ops is not None, "parity_ops": parity_ops,
        "e2e": {"value": round(ms_e2e / 1e3, 6), "unit": "s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": e2e_steps},
        "e2e_host_pointer": e2e_hp, "in_process": in_process, "cold_start": cold,
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"kernel": "k_accumulate (MSM bucket accumulation)", "bound": "hbm", "achieved": round(achieved, 2), "peak": hbm_peak, "unit": "GB/s",
                     "frac": round(achieved / hbm_peak, 5), "traffic": traffic, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": int(alg_bytes_per_launch), "avg_launch_ms": round(acc_ms / max(acc_cnt, 1), 4),
                     "kernel_share_of_step": round(acc_ms / args.steps / ms_dev, 4) if ms_dev > 0 else None,
                     "issue_bound": {"what": "the integer-multiply roofline of the SM: 16 32-bit product words / clk / sub-partition = 148 x 64 x 1.965 GHz = 18.6 T words/s (IMAD = 1 word, IMAD.WIDE = 2 words, "
                                             "carries free; profiles/r02_pipe_probe2_carry_cost.txt).  One bucket addition (XYZZ += affine) = 6 multiplications x 264 words + one two-product multiplication "
                                             "with a single reduction (392) + 2 squarings of 36 products (208 each) = 2392 words",
                                     "adds_per_s": round(my_msm_cols * n * win / (acc_ms / args.steps * 1e-3), 1) if acc_ms > 0 else None,
                                     "words_per_s": round(my_msm_cols * n * win * 2392 / (acc_ms / args.steps * 1e-3), 1) if acc_ms > 0 else None,
                                     "peak_words_per_s": 148 * 64 * 1.965e9,
                                     "frac": round(my_msm_cols * n * win * 2392 / (acc_ms / args.steps * 1e-3) / (148 * 64 * 1.965e9), 4) if acc_ms > 0 else None},
                     "note": "integer-issue bound (254-bit modular arithmetic), not HBM bound: see DESIGN.md"},
        "msm_pairs_per_s": round(pairs / world / (msm_ms * 1e-3), 1) * world if msm_ms > 0 else None,
        "ntt_elts_per_s": round(ntt_elts / world / (ntt_ms * 1e-3), 1) * world if ntt_ms > 0 else None,
        "msm_ms_per_step": round(msm_ms, 3), "ntt_ms_per_step": round(ntt_ms, 3),
        "kernel_class_ms_per_step": {name: round(v[0] / args.steps, 3) for name, v in prof.items()},
        "collectives_ms_per_step": {"rank0_total": round(coll_ms, 3), "calls_per_step": len(coll["events"]) // max(1, args.steps),
                                    "what": "all_to_all per evaluate_h column group, all_gather of h slabs, all_gather of commitments (CUDA events on rank 0's stream; includes waiting for the slowest rank)"},
    }
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(k, tname)
        print(json.dumps(line), flush=True)
    if world > 1 and not sim:
        dist.barrier()
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle ("port" of halo2's Rayon algorithms) on the host cores, running the WHOLE trace for real
class CpuTrace:
    """One proof's op trace on the CPU: every op instance of trace_ops() is executed (restated halo2 algorithms in oracle/,
    persistent thread pool), nothing is multiplied by a count.  Inputs are built once, outside the timed steps."""

    def __init__(self, k, tname, threads=None):
        from oracle import oracle as orc
        self.orc, self.k, self.tname = orc, k, tname
        self.threads = threads or orc.host_threads()
        self.n = 1 << k
        self.tr = TRACES[tname]
        self.ops = trace_ops(self.tr)
        self.ext_k = k + self.tr["ext_bits"]
        self.ncols = min(max(c for _, c in self.ops), 64)
        self.bases = [orc.gen_bases(self.n, seed=5, threads=self.threads), orc.gen_bases(self.n, seed=55, threads=self.threads)]
        self.cols = [orc.gen_scalars(self.n, seed=6 + i) for i in range(self.ncols)]
        self.xs = orc.gen_scalars(self.ncols, seed=7)
        self.one = orc.fr_one()
        self.group = QUOTIENT_GROUP if self.ext_k <= 23 else 16
        self.programs = {}
        self.per_op = {}

    def step(self):
        orc, tr, th, k, ext_k = self.orc, self.tr, self.threads, self.k, self.ext_k
        pick = lambda cnt: [self.cols[i % self.ncols] for i in range(cnt)]
        per = {}
        t_step = time.perf_counter()
        coeffs = None
        for kind, count in self.ops:
            t0 = time.perf_counter()
            if kind == "msm_lagrange" or kind == "msm_coeff":
                b = self.bases[0 if kind == "msm_lagrange" else 1]
                for c in pick(count):
                    orc.msm(c, b, th)
            elif kind == "batch_invert":
                for c in pick(count):
                    orc.batch_invert(c)
            elif kind in ("prefix_product", "prefix_sum"):
                for c in pick(count):
                    orc.prefix_scan(c, self.one, kind == "prefix_product")
            elif kind == "intt":
                coeffs = [orc.lagrange_to_coeff(c, k, th) for c in pick(count)]
            elif kind == "quotient":
                ncoset = n_coset_columns(tr)
                hq = np.zeros((1 << ext_k, 4), np.uint64)
                for g0 in range(0, ncoset, self.group):
                    m = min(self.group, ncoset - g0)
                    exts = [orc.coeff_to_extended(coeffs[(g0 + j) % len(coeffs)], ext_k, th) for j in range(m)]
                    if m not in self.programs:
                        self.programs[m] = gate_program(m).arrays()
                    loads, consts, prog = self.programs[m]
                    hq = orc.quotient_eval(exts + [hq], k, ext_k, loads, consts, prog, th)
                orc.extended_to_coeff(orc.divide_by_vanishing(hq, k, ext_k), ext_k, th)
            elif kind == "eval":
                for i, c in enumerate(pick(count)):
                    orc.eval_polynomial(c, self.xs[i % self.ncols])
            elif kind == "lincomb":
                per_set = max(1, (tr["advice"] + tr["fixed"] + tr["perm_cols"] + tr["perm_z"] + 2 * tr["lookups"] + 1 + tr["quotient_pieces"]) // tr["shplonk_sets"])
                for _ in range(count):
                    acc = self.cols[0]
                    for j in range(1, per_set):
                        acc = orc.poly_op("axpy", acc, self.cols[j % self.ncols], self.xs[j % self.ncols], threads=th)
            elif kind == "kate_division":
                for i, c in enumerate(pick(count)):
                    orc.kate_division(c, self.xs[i % self.ncols])
            per[kind] = per.get(kind, 0.0) + time.perf_counter() - t0
        self.per_op = {kk: round(v, 4) for kk, v in per.items()}
        return time.perf_counter() - t_step


def cpu_baseline(k, tname):
    """cpu_baseline of the GPU line: ONE whole trace step on the host cores (the first execution also warms the thread pool and
    page-faults the buffers in, so it is a slight over-estimate; `--impl reference` reports warmed steps)."""
    ct = CpuTrace(k, tname)
    v = ct.step()
    return {"value": round(v, 4), "unit": "s", "cores": ct.threads, "kind": "port",
            "sample": "1 whole trace step, every op instance executed (restated halo2 algorithms, oracle/bn254_oracle.c; not the Rust binary)",
            "per_op_s": ct.per_op}


def run_reference(args):
    """The reference arm: the CPU port executing whole trace steps in a real loop.  A k = 17 step takes tens of seconds on 128
    cores, so the loop is bounded by --cpu-budget seconds of wall time: at most `--warmup` (capped at 1) untimed + `--steps` timed
    steps, never fewer than one timed step; `steps` / `warmup` in the line are what actually ran."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    k = args.k
    tname = args.trace or CONFIG_FOR_K.get(k, "conv2d_mnist")
    t_all = time.perf_counter()
    ct = CpuTrace(k, tname)
    budget = max(args.cpu_budget, 1.0)
    warm = 0
    vals = []
    if args.warmup > 0:
        first = ct.step()
        warm = 1
        if first > budget / 2:          # the step is too long to afford a discarded warm-up: count it
            vals.append(first)
            warm = 0
    while len(vals) < max(1, args.steps):
        if vals and (time.perf_counter() - t_all) + 1.1 * max(vals) > budget:
            break
        vals.append(ct.step())
    v = sum(vals) / len(vals)
    base = {"value": round(v, 4), "unit": "s", "cores": ct.threads, "kind": "port",
            "sample": "%d whole trace step(s) timed after %d warm-up step(s), every op instance executed (restated halo2 algorithms, oracle/bn254_oracle.c; "
                      "not the Rust binary); requested --steps %d --warmup %d, bounded by --cpu-budget %.0f s" % (len(vals), warm, args.steps, args.warmup, budget),
            "per_step_s": [round(x, 3) for x in vals], "per_op_s": ct.per_op}
    line = {"impl": "reference", "metric": "prove_time_s", "value": round(v, 4), "unit": "s", "n_gpus": args.gpus, "steps": len(vals), "warmup": warm,
            "ms_per_step": round(v * 1e3, 1), "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
            "dtype": "u64 limbs (254-bit Montgomery integers)", "data": "synthetic",
            "config": make_config(k, tname),
            "cpu_baseline": base,
            "e2e": {"value": round(v, 4), "unit": "s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--k", type=int, default=17)
    ap.add_argument("--trace", default=None, choices=[None] + list(TRACES))
    ap.add_argument("--cpu-budget", type=float, default=150.0, help="--impl reference: wall-clock bound of the whole run in seconds")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity-gate", action="store_true", help="skip the oracle comparison of the timed inputs (profiling runs only; the line says parity_checked: false)")
    ap.add_argument("--no-host-pointer-e2e", action="store_true")
    ap.add_argument("--profile-one-step", action="store_true", help="setup + one device step only (for ncu launch lists)")
    ap.add_argument("--no-overlap", action="store_true", help="single-stream schedule (trace order), for A/B against the two-stream schedule")
    ap.add_argument("--simulate-rank-of", type=int, default=0, help="profiling aid: run rank 0's share of an N-way run on ONE GPU (collectives skipped); the line is marked SIMULATED")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32 digits of the wire limbs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
