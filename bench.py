#!/usr/bin/env python
"""bench.py — RISC-V cycles proven per second for the SP1 v6 core-shard hot path on B200.

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torchrun, one rank per GPU)
  python bench.py --impl reference ...                     (CPU arm: the oracle port on the host cores)

A "step" proves one batch of `--inflight` synthetic shards per GPU (default 6 for S2, each on its own library context + CUDA stream +
host transcript thread, so that the latency-bound sumcheck tails of one shard overlap the NTT / Poseidon2 kernels of another);
a shard = workload S2 by default (~1.9e8 trace cells = 2^22 cycles at 45 cells/cycle): main-trace jagged commit (RS-encode NTT +
Poseidon2 Merkle) followed by the phases listed in config.phases.  Per-phase times and the roofline lines are taken from a
shard proven ALONE (kernels_ms_per_shard_alone).
`value` is timed with the trace resident in HBM; `e2e` is the same step through the C ABI with the trace in pinned host
memory (H2D inside the timed region, proof D2H).  Shards are independent: ranks never communicate in the data path
(weak scaling); the only collectives are the barrier and the max-over-ranks of the elapsed time.
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

from sp1_b200 import workload as W  # noqa: E402

PHASES_DONE = ["commit(main): rs_encode + poseidon2 merkle", "logup-gkr: grind(12) + fraction circuit + 21 layer sumchecks + openings",
               "zerocheck: constraint bytecode interpreter, 22 rounds over all chips",
               "jagged open: hadamard sumcheck + branching-program sumcheck",
               "stacked/basefold open: batch + 21 fold rounds + 2 grinds + 124 queries"]
LEAF_TRAFFIC_BYTES_PER_LAUNCH = 3.191007e9 + 0.265294e9  # dram read + write of the 95-column S2c launch, profiles/ncu_leaf_hash_r02.txt (ncu --set full)
PHASES_MISSING = []  # the step is the whole prove_shard_with_data body (shard.rs:650-792) on synthetic AIRs


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi sampling during the timed region (B200_PROFILING.md recipe)"""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self.t.join(timeout=2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        mx = max(int(r[1]) for r in self.rows if r[1].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons, "samples": len(self.rows)}


def _oracle_threads(L):
    """one OpenMP thread per physical core this process may use: launchers such as torchrun export OMP_NUM_THREADS=1, and two
    threads per core (SMT) measured 5x slower on the oracle's barrier-heavy loops"""
    try:
        ncpu = len(os.sched_getaffinity(0))
        try:
            sib = open("/sys/devices/system/cpu/cpu0/topology/thread_siblings_list").read().strip()
            smt = 2 if ("," in sib or "-" in sib) else 1
        except OSError:
            smt = 1
        L.orc_set_num_threads(max(1, ncpu // smt))
    except (AttributeError, OSError):
        pass
    return int(L.orc_num_threads())


class OracleShard:
    """One synthetic shard (same machine, same chip heights as the GPU arm when scale == 1) set up for the CPU oracle:
    traces generated once (not timed); prove() = setup commit + the whole prove_shard_with_data body, verifier skipped."""

    def __init__(self, workload_name, scale=1.0):
        from tests import oracle_lib as O
        from sp1_b200 import synth_air as SA
        self.O, self.L = O, O.lib()
        self.cores = _oracle_threads(self.L)
        self.mach = W.synthetic_machine(workload_name, seed=42, scale=scale)
        self.params = W.params_of(workload_name)
        rng = np.random.default_rng(7)
        self.mains, self.preps = [], []
        for sp in self.mach["specs"]:
            m_, p_ = SA.synth_trace(rng, sp.h, sp.g, sp.wp, 12345, extra_cols=sp.extra, extra_prep=sp.extra_prep)
            self.mains.append(m_); self.preps.append(p_)
        self.pv = O.to_monty(np.array([12345, 5, 6, 7]))
        self.cells = W.area_of(self.mach["main_shapes"])
        self.cycles = self.cells / W.CELLS_PER_CYCLE

    def prove(self):
        import ctypes
        ch = self.O.Challenger()
        self.L.orc_set_skip_verify(1)
        t0 = time.time()
        self.O.prove_shard_verify(self.mach["blob"], [s_[0] for s_ in self.mach["specs"]], self.mains, self.preps, self.mach["names"],
                                  self.pv, self.params["log_stacking_height"], self.params["max_log_row_count"], ch)
        wall = time.time() - t0
        self.L.orc_set_skip_verify(0)
        t = (ctypes.c_double * 5)()
        self.L.orc_shard_times(t)
        return wall, dict(zip(("setup_commit", "main_commit", "logup_gkr", "zerocheck", "jagged_open"), [round(x, 3) for x in t]))


CPU_KIND_NOTE = ("oracle C++ port with OpenMP (scalar Montgomery arithmetic, no AVX-512 packing) - a NAIVE port, not the Rust/AVX-512 "
                 "Plonky3 prover: `cargo` is probed at run time and is absent in this image")


def _cargo_probe():
    import shutil
    return shutil.which("cargo") is not None


def cpu_baseline(workload_name):
    """cpu_baseline of the GPU arm: the oracle port on the host cores proving a BOUNDED sample of the workload (the same
    synthetic machine with every chip height scaled down to ~4 M cells; the protocol parameters stay the core ones, so the fixed
    costs - 2^21-row stacking, 22 sumcheck rounds, grinds, 124 queries - weigh more than in a full shard: same_config is false;
    the like-for-like figure is the `--impl reference` arm, which proves the full workload)."""
    full = W.synthetic_machine(workload_name, seed=42)
    sh = OracleShard(workload_name, scale=(1 << 22) / W.area_of(full["main_shapes"]))
    wall, phases = sh.prove()
    return {"value": sh.cycles / wall, "unit": "cycles/s", "cores": sh.cores, "kind": "port", "same_config": False,
            "cargo_present": _cargo_probe(), "phases_s": phases,
            "sample": f"same machine, heights scaled to {sh.cells} main cells ({sh.cycles:.0f} cycles): whole shard proof "
                      f"(setup commit + prove_shard body) in {wall:.1f}s; {CPU_KIND_NOTE}"}


def run_reference(args):
    """CPU arm, like for like: the oracle port proves the SAME workload as the GPU arm (same machine, same chip heights, core
    parameters) on all host cores.  One step = one whole shard proof; the arm times as many steps as fit a wall budget (at least 2,
    at most --steps) and reports the median, the spread, and how many steps it actually timed."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t_gen = time.time()
    sh = OracleShard(args.workload, scale=1.0)
    t_gen = time.time() - t_gen
    budget = float(os.environ.get("SP1B200_REF_BUDGET_S", "180"))
    walls, phases = [], None
    t_start = time.time()
    while len(walls) < max(1, args.steps):
        w_, phases = sh.prove()
        walls.append(w_)
        if len(walls) >= 2 and time.time() - t_start + float(np.median(walls)) > budget:
            break
    med = float(np.median(walls))
    v = sh.cycles / med
    cb = {"value": v, "unit": "cycles/s", "cores": sh.cores, "kind": "port", "same_config": True, "cargo_present": _cargo_probe(),
          "phases_s": phases,
          "sample": f"the full {args.workload} shard ({sh.cells} main cells = {sh.cycles:.0f} cycles), {len(walls)} timed proofs: "
                    f"median {med:.1f}s, min {min(walls):.1f}s, max {max(walls):.1f}s; {CPU_KIND_NOTE}"}
    print(json.dumps({"impl": "reference", "metric": "riscv_cycles_proven_per_second_core", "value": v, "unit": "cycles/s",
                      "n_gpus": args.gpus, "steps": len(walls), "steps_requested": args.steps, "warmup": 0, "warmup_requested": args.warmup,
                      "ms_per_step": med * 1e3, "higher_is_better": True,
                      "scaling": "weak", "vs_baseline": None, "dtype": "u32 KoalaBear (Montgomery) / ext4", "data": "synthetic",
                      "config": workload_config(args.workload, sh.cells, sh.cycles, len(sh.mach["specs"]), default_inflight(args)),
                      "cpu_baseline": cb, "spread": {"min_s": min(walls), "max_s": max(walls), "median_s": med, "n": len(walls)},
                      "trace_generation_s": round(t_gen, 1),
                      "e2e": {"value": v, "unit": "cycles/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def default_inflight(args):
    """shards proven concurrently per GPU (measured: 13.7 GB per calibrated 2^22-cycle context, 26-32 GB per full shard; S2c: 73.5 / 74.4 /
    75.5 / 75.2 M cycles/s at five / six / seven / eight in flight, six keeps 8 ranks x 6 host transcript threads within a 64-core host;
    S3c 73.4 M cycles/s at three, 78.1 M at four in flight)"""
    return args.inflight if args.inflight > 0 else {"S1": 5, "S2": 6, "S1c": 5, "S2c": 6, "R1": 5, "tiny": 4, "tinyc": 4, "tinyr": 4}.get(args.workload, 4)


def workload_config(workload, cells, cycles, n_chips, inflight):
    """the `config` object both arms print"""
    ls = W.params_of(workload)["log_stacking_height"]
    padded = ((cells + (1 << ls) - 1) >> ls) << ls
    c = {"workload": f"{workload}: {W.WORKLOADS[workload][1]}; main area {cells} cells = {cycles:.0f} cycles/shard "
                     f"(cells/45), {n_chips} chips (synthetic AIR bytecode + LogUp interactions), {padded >> ls} stacked columns of 2^{ls}, blowup 4, "
                     f"124 queries, 16+5+12 PoW bits",
         "phases": PHASES_DONE, "phases_not_yet_in_step": PHASES_MISSING}
    # identical in both arms (the driver compares the two config objects): the GPU-arm notes are stated for the GPU arm
    c["inflight"] = f"GPU arm: {inflight} shard(s) in flight per GPU per step (one context + stream each); CPU arm: one shard at a time on all host cores"
    c["l2"] = "GPU arm: working set (>= 3 GB codeword per shard) exceeds the 126 MB L2 between iterations"
    return c


DUMP_CAP_BYTES = 64 << 20


def dump_outputs(d, arrays):
    """--dump-outputs: write each uint32 array as <d>/<name>.npy in float64 (exact for 32-bit words), so that two builds can be compared
    output for output.  If all of them together exceed DUMP_CAP_BYTES, each keeps the same share of its words: a fixed, seeded sample of
    its flattened positions, in increasing order."""
    os.makedirs(d, exist_ok=True)
    total = sum(a.size for a in arrays.values()) * 8
    for name, a in arrays.items():
        if total > DUMP_CAP_BYTES:
            a = a.reshape(-1)
            a = a[np.sort(np.random.default_rng(0).choice(a.size, max(1, a.size * DUMP_CAP_BYTES // total), replace=False))]
        np.save(os.path.join(d, name + ".npy"), a.astype(np.float64))


def ref_kernels_leg(lib, n_cols, dev):
    """Head to head on this box: the REFERENCE's own CUDA kernels (oracle/_ref, compiled unmodified from sp1-gpu/crates/sys; launch
    shapes of its Rust host code) against this library's kernel-level entry points, on identical device buffers of the S2 commit
    shape.  Outside every timed region; a checker-side measurement, never part of the product path.  ratio = ref_ms / repo_ms."""
    import ctypes as C
    import torch
    from tests import ref_lib as R
    if not R.available():
        return {"unavailable": "oracle/_ref/libsp1ref.so not built"}
    R.lib()

    class TB:  # torch tensor seen as a device buffer by the reference launcher
        def __init__(self, t):
            self.t = t; self.ptr = C.c_void_p(t.data_ptr())
    g = torch.Generator(device=dev); g.manual_seed(5)
    out = {}
    log_h, lb = 21, 2
    msg = torch.randint(0, W.P, (n_cols, 1 << log_h), dtype=torch.int32, device=dev, generator=g)
    cw_ref = torch.empty((n_cols, 1 << (log_h + lb)), dtype=torch.int32, device=dev)
    cw = torch.empty_like(cw_ref)
    torch.cuda.synchronize()

    def best(fn, reps=3):
        v = []
        for _ in range(reps):
            v.append(fn())
        return min(v)
    # RS-encode
    ref_ms = best(lambda: R.batch_coset_dft(None, lb, d_in=TB(msg), d_out=TB(cw_ref), shape=(n_cols, 1 << log_h))[1])

    def mine_rs():
        lib.rs_encode(msg, cw, n_cols, log_h, lb); lib.sync()
        return lib.phase_ms("rs_encode")
    my_ms = best(mine_rs)
    torch.cuda.synchronize()
    same = bool(torch.equal(cw, cw_ref))
    out["rs_encode"] = {"shape": f"{n_cols} cols 2^21 -> 2^23", "ref_ms": ref_ms, "repo_ms": my_ms, "ratio": ref_ms / my_ms, "bit_identical": same}
    del cw_ref
    # Merkle: leaf hash + compress layers over the codeword
    h = log_h + lb
    nd = (2 << h) - 1
    dg_ref = torch.empty(nd * 8, dtype=torch.int32, device=dev)
    dg = torch.empty(nd * 8, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    r_leaf, r_comp = 1e30, 1e30
    for _ in range(3):
        _, (a_, b_) = R.merkle_tree((n_cols, 1 << h), d_mat=TB(cw), d_digests=TB(dg_ref))
        r_leaf, r_comp = min(r_leaf, a_), min(r_comp, b_)
    m_leaf, m_tot = 1e30, 1e30
    for _ in range(3):
        root, _c = lib.merkle_commit(cw, n_cols, h, d_layers=dg); lib.sync()
        m_leaf, m_tot = min(m_leaf, lib.phase_ms("merkle.leaf_hash")), min(m_tot, lib.phase_ms("merkle_commit"))
    torch.cuda.synchronize()
    root_ref = dg_ref[:8].cpu().numpy().view(np.uint32)
    out["leaf_hash"] = {"shape": f"{n_cols} cols x 2^23 rows", "ref_ms": r_leaf, "repo_ms": m_leaf, "ratio": r_leaf / m_leaf}
    out["compress_tree"] = {"shape": "2^23 leaves, 23 layers", "ref_ms": r_comp, "repo_ms": m_tot - m_leaf, "ratio": r_comp / (m_tot - m_leaf),
                            "root_identical": bool((root_ref == root).all())}
    out["note"] = ("reference kernels: leafHashPacked + compress (sys/lib/merkle_tree/merkle_tree.cu:27-94, launch shapes of "
                   "merkle_tree/src/single_layer.rs:109-150), batch_coset_dft (sys/include/ntt/sppark.cuh:49-107); CUDA events, best of 3; "
                   "repo compress_tree = merkle_commit - leaf_hash phases")
    return out


def run_queue(args):
    """--job queue (BASELINE config 5 / SURVEY.md 8e "S5"): `--shards` full shards with DISTINCT heights and traces (seeds 42+i) are
    placed round-robin on the ranks (the reference's controller hands ProveShard tasks to free workers, crates/prover/src/worker/
    client.rs:29-69), every rank's in-flight contexts pull their rank's shards from a host queue, each shard's trace goes H2D from
    pinned memory through the upload slots, and all proofs are gathered to rank 0 (the input of the recursion tree) with one NCCL
    gather - all inside the timed region.  Total work is fixed: strong scaling."""
    import torch
    import torch.distributed as dist
    from sp1_b200 import Lib
    from sp1_b200 import shards as SH
    from sp1_b200 import synth_air as SA
    from sp1_b200.lib import HostChallenger

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torchrun for N > 1)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n_shards, distinct = args.shards, min(args.distinct, args.shards)
    args.inflight = default_inflight(args)
    base = W.synthetic_machine(args.workload, seed=42)
    pv0 = 12345
    pv = ((np.array([pv0, 5, 6, 7], dtype=np.uint64) << np.uint64(32)) % np.uint64(W.P)).astype(np.uint32)
    # the distinct shard inputs this rank can be asked for: variant v = shard index % distinct (heights from seed 42+v)
    mine = SH.shards_of_rank(n_shards, rank, world)
    variants = sorted({i % distinct for i in mine})
    h_traces, heights_of, cycles_of = {}, {}, {}
    for v in variants:
        mv = W.synthetic_machine(args.workload, seed=42 + v)
        assert mv["names"] == base["names"] and [s_[1:] for s_ in mv["specs"]] == [s_[1:] for s_ in base["specs"]]
        heights_of[v] = [s_[0] for s_ in mv["specs"]]
        cycles_of[v] = W.area_of(mv["main_shapes"]) / W.CELLS_PER_CYCLE
        parts = [SA.synth_trace_cuda(sp.h, sp.g, sp.wp, pv0, SH.shard_seed(42, v) + k, dev, extra_cols=sp.extra, extra_prep=sp.extra_prep)[0] for k, sp in enumerate(mv["specs"])]
        d = torch.cat(parts)
        h_traces[v] = torch.empty(d.shape, dtype=torch.int32, pin_memory=True)
        h_traces[v].copy_(d)
        del parts, d
    # every variant's cycle count is needed for the total (a pure function of the seed)
    per = {v: W.area_of(W.shard_shapes(args.workload, seed=42 + v)[1]) for v in range(distinct)}
    pre_cells = W.area_of(base["main_shapes"]) - W.area_of(W.shard_shapes(args.workload, seed=42)[1])   # precompile table (same in every variant)
    total_cycles = sum(per[i % distinct] + pre_cells for i in range(n_shards)) / W.CELLS_PER_CYCLE
    # preprocessed tables are the same for every shard (their heights depend on the workload only)
    preps = [SA.synth_trace_cuda(sp.h, sp.g, sp.wp, pv0, SH.shard_seed(0, 0) + k, dev, extra_cols=sp.extra, extra_prep=sp.extra_prep)[1] for k, sp in enumerate(base["specs"]) if sp.wp]
    d_prep = torch.cat(preps).contiguous()
    prep_rows = [s_.h for s_ in base["specs"] if s_.wp]
    prep_cols = [1 + s_.extra_prep for s_ in base["specs"] if s_.wp]
    torch.cuda.synchronize()
    provers = []
    for _ in range(args.inflight):
        l_ = Lib(device=local, **W.params_of(args.workload))
        m_ = l_.machine_create(base["blob"])
        _, p_ = l_.jagged_commit_dense(d_prep, prep_rows, prep_cols)
        provers.append((l_, m_, p_))
    chal0 = HostChallenger().st.copy()
    names = base["names"]
    # the job moves every shard's trace over PCIe: measure this rank's host->device bandwidth (pinned, 256 MiB, best of 3) so that the
    # limiter can be named from the same run
    probe_h = torch.empty(64 << 20, dtype=torch.int32, pin_memory=True)
    probe_d = torch.empty(64 << 20, dtype=torch.int32, device=dev)
    h2d_gbs = 0.0
    for _ in range(3):
        a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a_.record(); probe_d.copy_(probe_h, non_blocking=True); b_.record(); torch.cuda.synchronize()
        h2d_gbs = max(h2d_gbs, probe_h.numel() * 4 / (a_.elapsed_time(b_) / 1e3) / 1e9)
    del probe_h, probe_d
    h2d_min = -SH.max_over_ranks(-h2d_gbs, dev)
    h2d_max = SH.max_over_ranks(h2d_gbs, dev)

    def worker(who, q, proofs, busy):
        l_, m_, p_ = provers[who]
        nxt = q.pop()
        if nxt is None:
            return
        slot = 0
        d_nxt = l_.upload_begin(h_traces[nxt % distinct], slot)
        t0 = time.time()
        while nxt is not None:
            cur, d_cur = nxt, d_nxt
            nxt = q.pop()
            if nxt is not None:
                slot ^= 1
                d_nxt = l_.upload_begin(h_traces[nxt % distinct], slot)   # the next shard's H2D overlaps this shard's proof
            st = chal0.copy()
            proofs[cur] = l_.prove_shard(m_, p_, d_cur, heights_of[cur % distinct], names, pv, st)
        busy[who] = time.time() - t0

    def run_once(n):
        q = SH.ShardQueue(n, rank, world)
        proofs, busy = {}, [0.0] * len(provers)
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        if world > 1:
            dist.barrier()
        for l_, _, _ in provers:
            l_.sync()
        torch.cuda.synchronize()
        e0.record()
        ths = [threading.Thread(target=worker, args=(w_, q, proofs, busy)) for w_ in range(len(provers))]
        [t.start() for t in ths]
        [t.join() for t in ths]
        for l_, _, _ in provers:
            l_.sync()
        e1.record()
        allp = SH.gather_proofs(proofs, dst=0, device=dev)
        torch.cuda.synchronize()
        e2.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        return e0.elapsed_time(e2), e1.elapsed_time(e2), allp, busy

    run_once(min(n_shards, world * len(provers) * 2))   # slot allocation and pool growth are setup: one small untimed pass
    with ClockSampler(local) as cs:
        ms, gather_ms, allp, busy = run_once(n_shards)
    clocks = cs.summary()
    ms_all = SH.max_over_ranks(ms, dev)
    launches = sum(l_.launch_count() for l_, _, _ in provers)
    out = None
    if rank == 0:
        assert sorted(allp) == list(range(n_shards)), "rank 0 did not receive every shard's proof"
        proof_bytes = int(sum(v.size for v in allp.values()) * 4)
        h2d = int(sum(h_traces[i % distinct].numel() * 4 for i in mine))
        v = total_cycles / (ms_all / 1e3)
        out = {"metric": "riscv_cycles_proven_per_second_core", "value": v, "unit": "cycles/s", "n_gpus": world, "steps": 1, "warmup": 1,
               "ms_per_step": ms_all, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
               "dtype": "u32 KoalaBear (Montgomery) / ext4", "data": "synthetic", "job": "queue",
               "config": {"workload": f"S5: {n_shards} shards of {args.workload} ({W.WORKLOADS[args.workload][1]}), {distinct} distinct height sets / traces "
                                      f"(seeds 42+i), {total_cycles:.0f} cycles in total; round-robin over {world} rank(s), {len(provers)} contexts per rank "
                                      "pulling from the rank's host queue; traces H2D per shard from pinned memory; proofs gathered to rank 0",
                          "phases": PHASES_DONE, "l2": "working set exceeds L2"},
               "e2e": {"value": v, "unit": "cycles/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": proof_bytes,
                       "note": "the job is end to end by construction: per-shard H2D, proof D2H and the gather are inside the timed region; "
                               "h2d bytes are rank 0's"},
               "gather": {"ms_incl_wait_for_slowest_rank": gather_ms, "proof_bytes_total": proof_bytes,
                          "how": "all_gather of the (index, length) table + one NCCL gather of padded words; rank 0 enters the collective when ITS "
                                 "shards are done, so this time includes waiting for the slowest rank"},
               "rank0_context_busy_s": [round(b, 3) for b in busy], "gpu_launches": int(launches), "clocks": clocks,
               "h2d_probe_gb_per_s": {"min_over_ranks": h2d_min, "max_over_ranks": h2d_max, "how": "pinned 256 MiB host->device copy, best of 3, per rank"},
               "bytes_per_shard": int(h_traces[variants[0]].numel() * 4),
               "limiter": "static placement: %d shards per rank over %d contexts = %d waves (the last one partly empty), plus rank 0 waiting inside the gather "
                          "for the slowest rank; the traces need %.1f GB/s of H2D per GPU to keep the provers busy and the measured pinned rate is "
                          "%.1f-%.1f GB/s per GPU, so the transfer is hidden behind the proofs"
                          % (len(mine), len(provers), -(-len(mine) // len(provers)), h_traces[variants[0]].numel() * 4 / 1e9 / 0.124, h2d_min, h2d_max)}
        print(json.dumps(out))
    for l_, m_, p_ in provers:
        l_.jagged_round_free(p_); l_.machine_free(m_); l_.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="S2c", choices=list(W.WORKLOADS),
                    help="S2c (default): the sha-bench-like 2^22-cycle shard with CALIBRATED chips (constraint counts and LogUp message "
                         "statistics read off the reference's Rust eval functions, sp1_b200/chip_stats.json); S2: the same shapes with the "
                         "light round-1 chip template")
    ap.add_argument("--no-light-line", action="store_true", help="skip the side-by-side run of the light-template workload")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-kernels", action="store_true", help="skip the head-to-head timing of the reference's own CUDA kernels (oracle/_ref)")
    ap.add_argument("--inflight", type=int, default=0,
                    help="shards proven concurrently per GPU (one library context + stream + host thread each): the latency-bound "
                         "sumcheck tails of one shard overlap the NTT / Poseidon2 kernels of another")
    ap.add_argument("--e2e-mode", default="pipelined", choices=["pipelined", "serial"],
                    help="pipelined: H2D of step i+1 overlaps the proof of step i (upload slots); serial: plain host pointer per step")
    ap.add_argument("--job", default="step", choices=["step", "queue"],
                    help="step: the driver's contract (K identical steps, weak scaling); queue: --shards distinct shards through a host queue with "
                         "per-shard H2D and a proof gather to rank 0 (strong scaling, BASELINE config 5)")
    ap.add_argument("--shards", type=int, default=64)
    ap.add_argument("--distinct", type=int, default=16, help="--job queue: number of distinct (heights, trace) sets the shards cycle over")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step returned to each in-flight caller of prove_shard (rank 0) as "
                         "DIR/<name>.npy in float64: proof_words and challenger_state [inflight, ...] of the device-resident steps, "
                         "e2e_proof_words and e2e_challenger_state of the e2e steps; at most 64 MB in all (larger: a fixed, seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    if args.job == "queue":
        return run_queue(args)

    import torch
    import torch.distributed as dist
    from sp1_b200 import Lib
    from sp1_b200.lib import HostChallenger

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torchrun for N > 1)"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    params = W.params_of(args.workload)
    lib = Lib(device=local, **params)
    stream = torch.cuda.ExternalStream(lib.stream(), device=dev)

    from sp1_b200 import synth_air as SA
    from sp1_b200 import shards as SH
    # one shard per rank per step (weak scaling): rank r proves shard r of a world-sized batch of independent shards
    my_shard = SH.shards_of_rank(world, rank, world)[0]
    mach = W.synthetic_machine(args.workload, seed=42)
    specs, names = mach["specs"], mach["names"]
    heights = [s_[0] for s_ in specs]
    cells = W.area_of(mach["main_shapes"])
    cycles = cells / W.CELLS_PER_CYCLE
    pv0 = 12345
    pv = ((np.array([pv0, 5, 6, 7], dtype=np.uint64) << np.uint64(32)) % np.uint64(W.P)).astype(np.uint32)
    mains, preps = [], []
    for i, sp in enumerate(specs):
        m_, p_ = SA.synth_trace_cuda(sp.h, sp.g, sp.wp, pv0, SH.shard_seed(0, my_shard) + i, dev, extra_cols=sp.extra, extra_prep=sp.extra_prep)
        mains.append(m_)
        if sp.wp:
            preps.append(p_)
    d_main = torch.cat(mains).contiguous()
    d_prep = torch.cat(preps).contiguous()
    del mains, preps
    h_main = torch.empty(d_main.shape, dtype=torch.int32, pin_memory=True)
    h_main.copy_(d_main)
    torch.cuda.synchronize()
    # setup (not timed; reference: AirProver::setup uploads the machine and commits the preprocessed traces once per program)
    machine = lib.machine_create(mach["blob"])
    prep_rows = [s_.h for s_ in specs if s_.wp]
    prep_cols = [1 + s_.extra_prep for s_ in specs if s_.wp]
    _, h_prep = lib.jagged_commit_dense(d_prep, prep_rows, prep_cols)
    # further in-flight provers on the same GPU: own context (stream, mailbox, upload slots), own machine / preprocessed commit
    # default: as many shards in flight as the device memory comfortably holds (measured: ~24 GB per S2 context at the pool's high
    # water mark; throughput saturates at 5-6 contexts), never more than 5
    args.inflight = default_inflight(args)
    provers = [(lib, machine, h_prep)]
    for _ in range(1, args.inflight):
        l2 = Lib(device=local, **params)
        m2 = l2.machine_create(mach["blob"])
        _, p2 = l2.jagged_commit_dense(d_prep, prep_rows, prep_cols)
        provers.append((l2, m2, p2))
    chal0 = HostChallenger().st.copy()
    LS = params["log_stacking_height"]
    padded_cells = ((cells + (1 << LS) - 1) >> LS) << LS

    phase_names = ["commit.rs_encode", "commit.merkle", "merkle.leaf_hash", "shard.commit", "gkr.circuit", "gkr.rounds", "gkr.openings", "gkr.total", "gkr.host_wait", "gkr.host_interaction", "gkr.host_transcript",
                   "zerocheck.total", "zerocheck.host_wait", "zerocheck.host_math", "zerocheck.host_setup", "jagged.little_poly", "jagged.sumcheck", "jagged.eval_sumcheck", "open.batch", "open.fri_rounds",
                   "open.queries", "open.total", "jagged.total", "shard.total"]
    acc = {}

    def step(src, record=False, who=0):
        """-> (proof words, final challenger state): what a caller of prove_shard receives"""
        l_, m_, p_ = provers[who]
        st = chal0.copy()
        proof = l_.prove_shard(m_, p_, src, heights, names, pv, st)
        if record and who == 0:
            for n in phase_names:
                v = l_.phase_ms(n)
                if v >= 0:
                    acc[n] = acc.get(n, 0.0) + v
        return proof, st

    def run_steps(who, src, k, pipelined_upload, out):
        l_ = provers[who][0]
        if pipelined_upload:
            nxt = l_.upload_begin(src, 0)
            for i in range(k):
                cur = nxt
                if i + 1 < k:
                    nxt = l_.upload_begin(src, (i + 1) & 1)
                out[who] = step(cur, record=True, who=who)
        else:
            for _ in range(k):
                out[who] = step(src, record=True, who=who)

    def sync_all():
        for l_, _, _ in provers:
            l_.sync()
        torch.cuda.synchronize()

    def timed(src, k, pipelined_upload=False):
        """k steps, each step = one shard per in-flight prover; pipelined_upload: src is the pinned host buffer, every shard's H2D
        goes through the library's double-buffered upload slots (C ABI sp1b200_upload_begin) so that the copy of the next shard
        overlaps the proof of the current one — all copies are inside the timed region.
        -> (ms, launches, [(proof words, challenger state) of the last step, per in-flight prover])"""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if world > 1:
            dist.barrier()
        sync_all()
        l0 = sum(l_.launch_count() for l_, _, _ in provers)
        e0.record(stream)
        out = [None] * len(provers)
        if len(provers) == 1:
            run_steps(0, src, k, pipelined_upload, out)
        else:
            ths = [threading.Thread(target=run_steps, args=(w, src, k, pipelined_upload, out)) for w in range(len(provers))]
            for t in ths:
                t.start()
            for t in ths:
                t.join()
        sync_all()
        e1.record(stream)
        sync_all()
        if world > 1:
            dist.barrier()
        ms = SH.max_over_ranks(e0.elapsed_time(e1), dev)
        return ms, sum(l_.launch_count() for l_, _, _ in provers) - l0, out

    if os.environ.get("SP1B200_PROFILE_RANGE") == "1":   # ncu --profile-from-start off: skip the torch trace synthesis and the setup
        torch.cuda.cudart().cudaProfilerStart()
    # warm-up in the same concurrent shape as the timed steps (the stream-ordered memory pool has to grow to its steady size)
    if args.warmup:
        timed(d_main, args.warmup)
    acc.clear()
    # per-phase / per-kernel times (roofline lines): ONE shard proven alone, outside the throughput measurement
    PHASE_REPS = 2
    for _ in range(PHASE_REPS):
        step(d_main, record=True, who=0)
    sync_all()
    phases = {k: v / PHASE_REPS for k, v in acc.items()}
    acc.clear()
    with ClockSampler(local) as cs:
        ms_dev, launches, last_dev = timed(d_main, args.steps)
        acc.clear()
        if args.e2e_mode == "pipelined":
            for l_, _, _ in provers:
                l_.upload_begin(h_main, 0); l_.upload_begin(h_main, 1); l_.sync()   # slot allocation is setup, not a step
        ms_e2e, _, last_e2e = timed(h_main, args.steps, pipelined_upload=(args.e2e_mode == "pipelined"))
    clocks = cs.summary()
    proof_bytes = last_dev[0][0].nbytes
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"proof_words": np.stack([p for p, _ in last_dev]), "challenger_state": np.stack([s for _, s in last_dev]),
                                         "e2e_proof_words": np.stack([p for p, _ in last_e2e]), "e2e_challenger_state": np.stack([s for _, s in last_e2e])})

    total_cycles = cycles * world * len(provers)  # every rank proves `inflight` shards of the same size per step (weak scaling)
    value = total_cycles * args.steps / (ms_dev / 1e3)
    e2e = total_cycles * args.steps / (ms_e2e / 1e3)
    hbm, peak_src = peaks()
    ntt_ms = phases.get("commit.rs_encode", float("nan"))
    ach = 20.0 * padded_cells / (ntt_ms / 1e3) / 1e9
    merkle_ms = phases.get("commit.merkle", float("nan"))
    leaf_ms = phases.get("merkle.leaf_hash", float("nan"))
    n_stacked = padded_cells >> LS
    leaf_bytes = (4 * n_stacked + 32) * (1 << (LS + 2))
    leaf_perms = (1 << (LS + 2)) * ((n_stacked + 7) // 8)
    leaf_gbs = leaf_bytes / (leaf_ms / 1e3) / 1e9
    perms = (1 << (LS + 2)) * ((n_stacked + 7) // 8) + (1 << (LS + 2))
    out = {
        "metric": "riscv_cycles_proven_per_second_core", "value": value, "unit": "cycles/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32 KoalaBear (Montgomery) / ext4", "data": "synthetic",
        "config": workload_config(args.workload, cells, cycles, len(specs), len(provers)),
        "e2e": {"value": e2e, "unit": "cycles/s", "h2d_bytes_per_step": int(cells * 4) * len(provers), "d2h_bytes_per_step": int(proof_bytes) * len(provers),
                "ms_per_step": ms_e2e / args.steps,
                "note": "host trace in pinned memory -> sp1b200_upload_begin (two device slots, copy stream) -> sp1b200_prove_shard; "
                        "the copy of step i+1 overlaps the proof of step i, every step's copy and proof read-back are inside the timed region"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"kernel": "leaf_hash_kernel (Poseidon2 sponge over the 2^23 codeword rows of the main commit; largest share of the step)",
                     "bound": "hbm", "achieved": leaf_gbs, "peak": hbm, "unit": "GB/s", "frac": leaf_gbs / hbm,
                     "traffic": LEAF_TRAFFIC_BYTES_PER_LAUNCH, "algorithmic_bytes_per_launch": leaf_bytes, "peak_source": peak_src,
                     "limiter": "the fmaheavy integer-multiply pipe, not HBM: 12 Poseidon2 permutations per 412-byte row; ncu shows "
                                "sm__pipe_fmaheavy_cycles_active 90 %, fmalite 0 %, alu 61 % (profiles/ncu_p2_pipes_r02.txt): every IMAD* "
                                "instruction of the permutation (3 434 pipe slots per permutation after the round-2 s-box change, 3 724 before) "
                                "runs on that one pipe; register-resident permutations reach 5.02 Gperm/s (tools/p2_modes.cu), see DESIGN.md section 3.1",
                     "gperm_per_s": leaf_perms / (leaf_ms / 1e3) / 1e9, "register_resident_gperm_per_s": 5.02,
                     "note": "algorithmic bytes = (4 B x stacked columns + 32 B digest) x 2^23 rows per launch; CUDA events on the library "
                             "stream (phase merkle.leaf_hash); traffic = dram read+write of the same launch under ncu --set full (profiles/)"},
        "roofline_rs_encode": {"kernel": "rs_encode (rs_step_a_fast<10> + rs_step_b_2048), all stacked columns of the main commit",
                               "bound": "hbm", "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm,
                               "traffic": {"rs_step_a_fast<10>": 32.3e6, "rs_step_b_2048": 76.4e6, "per": "launch pair = 2 columns (cold cache under ncu)",
                                           "algorithmic": 83.9e6},
                               "peak_source": peak_src,
                               "note": "algorithmic 20 B/cell (4 B read + 16 B codeword write); integer-pipe bound (46 modular products per cell), see DESIGN.md"},
        "kernels_ms_per_shard_alone": phases,
        "inflight": len(provers), "ms_per_shard": ms_dev / args.steps / len(provers),
        "gpu_mem_used_gb": round((torch.cuda.mem_get_info(dev)[1] - torch.cuda.mem_get_info(dev)[0]) / 2**30, 1),
        "poseidon2": {"leaf+compress_perms_per_step": int(perms), "gperm_per_s": perms / (merkle_ms / 1e3) / 1e9,
                      "note": "INT32-ALU bound (see DESIGN.md), not HBM bound"},
    }
    for l_, m_, p_ in provers[1:]:
        l_.jagged_round_free(p_)
        l_.machine_free(m_)
        l_.close()
    del d_main, h_main
    torch.cuda.empty_cache()
    if rank == 0:
        if world == 1 and not args.no_light_line and args.workload in W.BASE_OF:
            # side by side: the same shard shapes with the light round-1 chip template, measured by a child process now that this
            # process has released its shards (same code path, fewer steps; not part of `value`)
            try:
                lib.jagged_round_free(h_prep); lib.machine_free(machine); h_prep = machine = None
                cp = subprocess.run([sys.executable, os.path.abspath(__file__), "--workload", W.BASE_OF[args.workload], "--steps", str(min(args.steps, 5)),
                                     "--warmup", "3", "--no-cpu-baseline", "--no-ref-kernels", "--no-light-line", "--inflight", str(args.inflight)],
                                    capture_output=True, text=True, timeout=600)
                lj = json.loads(cp.stdout.strip().splitlines()[-1])
                out["light_workload"] = {"workload": lj["config"]["workload"], "value": lj["value"], "e2e": lj["e2e"]["value"], "unit": "cycles/s",
                                         "ms_per_shard": lj["ms_per_shard"], "kernels_ms_per_shard_alone": lj["kernels_ms_per_shard_alone"],
                                         "note": "same shard shapes, light chip template (round-1 headline workload): ~4 constraints per 6 columns, "
                                                 "1-3 values per interaction on a third of the column groups"}
            except Exception as e:
                out["light_workload"] = {"unavailable": f"failed: {e}"}
        if world == 1 and not args.no_ref_kernels:
            try:
                out["vs_ref_kernels"] = ref_kernels_leg(lib, int(n_stacked), dev)
            except Exception as e:  # the reference kernels are a checker-side bar; the GPU numbers stand without them
                out["vs_ref_kernels"] = {"unavailable": f"failed: {e}"}
        if world == 1 and not args.no_cpu_baseline:
            try:
                out["cpu_baseline"] = cpu_baseline(args.workload)
            except Exception as e:  # the oracle is a checker; the GPU numbers stand without it
                out["cpu_baseline"] = {"value": None, "unit": "cycles/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e}"}
        print(json.dumps(out))
    if h_prep is not None:
        lib.jagged_round_free(h_prep)
        lib.machine_free(machine)
    lib.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
