#!/usr/bin/env python
"""bench.py -- routing decisions/s of the EPP scheduling cycle on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload config3] [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the whole hot path (prefix-block hashing -> index lookup / global-stop match -> load scoring
-> weighted sum -> arg-max pick [-> decider -> prefill pick]) over one batch of synthetic requests.
  value     decisions/s with the batch already resident in HBM (device-pointer batch through the C ABI)
  e2e       the same metric through the C ABI with HOST (pinned) buffers: the H2D copy of every prompt byte and the
            D2H copy of every decision record are inside the timed region
  roofline  dominant kernel: algorithmic bytes per launch / CUDA-event launch time vs MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the oracle (C restatement of the reference Go loops, kind "port") on the host cores, bounded sample
--impl reference: times the reference's CPU algorithm (the oracle port; Go is not installable here) on all host cores.
Multi-GPU (--gpus N under torchrun): N independent replicas, each with the full index and its own batch (weak
scaling, no data-path collective); time = max over ranks.
--dump-outputs DIR: after the timed steps, rank 0 writes the decisions of the last timed step as DIR/<field>.npy (see
_dump_decisions); the inputs depend only on the arguments, so two builds can be compared file by file.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

# stdout carries exactly ONE JSON line: NCCL's log (communicator set-up at NCCL_DEBUG=INFO) goes to stderr instead,
# unchanged, so that the driver can still read it
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True        # the benchmark leaves the source tree as it found it (it may be read-only)

METRIC = "routing decisions/sec at 4K-token prompts x 4,096 endpoints"
UNIT = "decisions/s"


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) >= 8:
                self.rows.append(f)

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for f in self.rows:
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v == "Active":
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def _bind_to_gpu_numa_node(local_rank: int):
    """Run this rank (and first-touch its pinned staging buffers) on the NUMA node its GPU hangs off, so 8 ranks do not
    pull their H2D traffic across the socket interconnect.  Returns (node, all_cpus) or (None, all_cpus)."""
    all_cpus = os.sched_getaffinity(0)
    try:
        import torch
        pr = torch.cuda.get_device_properties(local_rank)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return None, all_cpus
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= all_cpus
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node, all_cpus
    except Exception:
        pass
    return None, all_cpus


def _pinned(nbytes: int, lib):
    p = C.c_void_p()
    rc = lib.epp_host_alloc(nbytes, C.byref(p))
    if rc != 0:
        raise RuntimeError("epp_host_alloc failed")
    return p, np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(nbytes,))


DUMP_MAX_ROWS = 1 << 19                 # 8 arrays x 8 B x 2^19 rows = 32 MiB


def _dump_decisions(out_dir: str, dec: np.ndarray):
    """--dump-outputs: the epp_decision records a caller of the timed path receives, one float64 array per field
    (endpoint ids are u32 and scores f64, both exact in float64), plus request.npy, the batch row of each entry.
    Batches above DUMP_MAX_ROWS requests are written as a fixed seeded sample of rows."""
    rows = np.arange(dec.shape[0])
    if rows.size > DUMP_MAX_ROWS:
        rows = np.sort(np.random.default_rng(0).choice(rows.size, DUMP_MAX_ROWS, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "request.npy"), rows.astype(np.float64))
    for name in dec.dtype.names:
        np.save(os.path.join(out_dir, name + ".npy"), dec[name][rows].astype(np.float64))


def _workload(name: str, R: int | None):
    from tools import tracegen as tg
    w = tg.baseline_configs()[name]
    if R:
        w = w.scaled(R=R, name=w.name)
    return w


def _config_json(w, n_gpus, extra=None):
    scor = ",".join(f"{ {0: 'prefix', 1: 'kv-util', 2: 'queue', 3: 'load-aware'}[k]}*{wt:g}" for k, wt, _ in w.primary_scorers)
    c = {"workload": f"{w.name}: {w.E} endpoints, {w.T}-token prompts ({w.prompt_bytes} B, {w.blocks} blocks of "
                     f"{w.block_size_tokens * 4} B), batch {w.R} requests per GPU, scorers {scor}"
                     + (f", P/D two-stage pick ({w.n_prefill} prefill endpoints, nonCachedTokens {w.non_cached_tokens})"
                        if w.prefill_scorers else ""),
         "endpoints": w.E, "prompt_tokens": w.T, "batch_requests_per_gpu": w.R, "block_size_tokens": w.block_size_tokens,
         "max_prefix_blocks": w.max_prefix_blocks,
         "l2": f"inputs are {w.R * w.prompt_bytes / 2**20:.0f} MiB per step per GPU, larger than the 126 MB L2 (no flush needed)",
         "parallelism": f"{n_gpus} independent replicas (index replicated, requests sharded; no data-path collective)",
         "trace_seed": hex(w.seed)}
    if extra:
        c.update(extra)
    return c


def _best_thread_count(run, n_max: int):
    """The host may expose more logical CPUs than it lets this container use: probe a few thread counts on a short
    sample and keep the fastest (the baseline must be the CPU's best, not an oversubscribed run).  Returns the winner
    and the whole table {threads: decisions/s} (the rate moves a lot from box to box)."""
    cands = sorted({max(1, n_max >> k) for k in range(0, 6)} | {min(n_max, 8)}, reverse=True)
    best, best_rate, table = cands[0], 0.0, {}
    for nt in cands:
        rate = run(nt)
        table[str(nt)] = round(rate, 1)
        if rate > best_rate * 1.05:
            best, best_rate = nt, rate
    return best, table


def cpu_baseline(w, trace, n_threads: int, target_s: float = 12.0, tokens: np.ndarray | None = None):
    """Oracle (port of the reference Go loops) on the host cores over a bounded sample of the same workload."""
    from tools import workload_setup as helpers
    from oracle import pyoracle as orc
    pool, ix, primary, prefill, _ = helpers.setup_oracle(orc, w, trace)
    n = int(min(w.R, tokens.shape[0] if tokens is not None else w.R))
    tk = tokens[:n] if tokens is not None else trace.requests(0, n)[0]
    probe_n = min(n, max(16 * n_threads, 2048))

    def probe(nt):
        t0 = time.perf_counter()
        helpers.oracle_decisions(orc, w, pool, ix, primary, prefill, tk[:probe_n], nt)
        return probe_n / (time.perf_counter() - t0)

    probe(n_threads)                                   # warm caches / page in
    nt, table = _best_thread_count(probe, n_threads)
    passes, dt = 0, 0.0
    odec = None
    while dt < target_s and passes < 1000:      # repeat the batch until ~target_s of CPU work has been timed
        t0 = time.perf_counter()
        odec, _ = helpers.oracle_decisions(orc, w, pool, ix, primary, prefill, tk, nt)
        dt += time.perf_counter() - t0
        passes += 1
    n_total = n * passes
    return {"value": n_total / dt, "unit": UNIT, "cores": nt, "kind": "port", "threads_probed": table,
            "sample": f"{passes} passes over the first {n} requests of the step's batch ({n_total} decisions), "
                      f"{nt} host threads (fastest of the probed counts; os.cpu_count() = {n_threads}), {dt:.2f} s; "
                      "C restatement of the reference Go loops (oracle/epp_oracle.c) -- the Go toolchain is not "
                      "installable here"}, odec


def run_reference(args, rank, world):
    if rank != 0:
        return
    from tools import tracegen as tg
    w = _workload(args.workload, args.requests)
    trace = tg.Trace(w)
    n_threads = os.cpu_count() or 1
    from tools import workload_setup as helpers
    from oracle import pyoracle as orc
    orc.build()
    pool, ix, primary, prefill, _ = helpers.setup_oracle(orc, w, trace)
    # thread count: the fastest of a few probed counts (the box may oversubscribe its logical CPUs)
    probe = trace.requests(0, min(w.R, max(16 * n_threads, 2048)))[0]

    def probe_rate(nt):
        t0 = time.perf_counter()
        helpers.oracle_decisions(orc, w, pool, ix, primary, prefill, probe, nt)
        return probe.shape[0] / (time.perf_counter() - t0)

    probe_rate(n_threads)
    n_cpu = n_threads
    n_threads, table = _best_thread_count(probe_rate, n_threads)
    # size one step so that (warmup + steps) steps take about 60 s in total
    per_req = 1.0 / probe_rate(n_threads)
    n = int(min(w.R, max(n_threads, 60.0 / max(1, args.steps + args.warmup) / per_req)))
    n = max(n_threads, (n // n_threads) * n_threads)
    tokens = trace.requests(0, n)[0]
    for _ in range(args.warmup):
        helpers.oracle_decisions(orc, w, pool, ix, primary, prefill, tokens, n_threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        helpers.oracle_decisions(orc, w, pool, ix, primary, prefill, tokens, n_threads)
    dt = time.perf_counter() - t0
    val = n * args.steps / dt
    sample = (f"each step = first {n} requests of the workload's batch on {n_threads} host threads (fastest of the probed "
              f"counts; os.cpu_count() = {n_cpu}); C restatement of the reference Go loops (oracle/epp_oracle.c), Go "
              "toolchain unavailable")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64 (XXH64) + f64 (scores)", "data": "synthetic",
        "config": _config_json(w, args.gpus),
        "reference_step_requests": n,
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": n_threads, "kind": "port", "sample": sample,
                         "threads_probed": table},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def index_write_leg(args, w, trace, dev_tokens, dev_dec, local_rank, epp, helpers, orc_mod):
    """SURVEY 8(f).1 -- PreRequest at batch rate: schedule a batch, index its picks ON THE DEVICE (indexer.Add + LRU
    eviction for 65 536 x 256 hashes), bring the read table up to date.  The engine's index is seeded through
    indexer.Add (not a snapshot), LRU capacity is the reference default (31 250 per endpoint).  Two tie rules:
    the reproducible random one (tie_seed != 0, what a deployment runs: tied requests spread over the arg-max set like
    the reference's shuffle) and the deterministic lowest-slot one (tie_seed = 0: EVERY cold request of a batch picks
    the same endpoint, millions of Adds to one LRU -- the worst case for the write side).  The CPU number beside it is
    the oracle's indexer (one mutex, like indexer.go) applying a bounded sample of the same Adds."""
    import torch
    from tools import tracegen as tg
    role, kv, waiting, running = trace.pool()
    out = {"what": "epp_schedule(keep_hashes) + epp_index_add_picked + epp_index_commit per config-3 batch (65 536 picks x up to 256 block hashes)"}
    hs = es = cuts = None
    for label, seed in (("random_ties", 0x7153ED), ("lowest_slot_ties", 0)):
        eng = helpers.make_engine(w, device=local_rank, tie_seed=seed)
        eng.register_model(tg.MODEL)
        eng.pool_set(np.arange(w.E, dtype=np.uint32), role, kv, waiting, running)
        fh, _ = eng.hash_prompts(trace.family_tokens(), uniform_len=w.prompt_bytes)
        hs, es = trace.index_pairs(fh)
        order = np.argsort(es, kind="stable")
        hs, es = hs[order], es[order]
        cuts = np.flatnonzero(np.diff(es)) + 1
        for seg_h, seg_e in zip(np.split(hs, cuts), np.split(es, cuts)):
            if len(seg_e):
                eng.index_add(int(seg_e[0]), seg_h)
        if args.index_fill > 0:                      # production-size index: every endpoint's LRU (nearly) full
            fhs, _ = helpers.filler_pairs(w.E, args.index_fill)
            for e in range(w.E):
                eng.index_add(e, fhs[e * args.index_fill:(e + 1) * args.index_fill])
        eng.index_commit()
        cycles = []
        R = w.R
        for k in range(4):
            torch.cuda.synchronize()
            t_all = time.perf_counter()
            eng.schedule(dev_tokens, uniform_len=w.prompt_bytes, detail=False, out=dev_dec, keep_hashes=True)
            t0 = time.perf_counter()
            eng.index_add_picked()
            eng.index_commit()
            t1 = time.perf_counter()
            st = eng.stats()
            cycles.append({"schedule_ms": (t0 - t_all) * 1e3, "apply_ms": st["last_index_apply_ms"], "build_ms": st["last_index_build_ms"],
                           "write_wall_ms": (t1 - t0) * 1e3, "cycle_wall_ms": (t1 - t_all) * 1e3,
                           "hashes_added": int(st["last_index_items"]), "pairs_after": int(st["index_pairs"]),
                           "read_table": "patched from the change log" if st["last_index_patched"] else "bulk rebuild"})
        last = cycles[-1]
        dec = epp.decisions_from_torch(dev_dec)
        ok = dec["status"] == 0
        out[label] = {"tie_seed": seed, "cycles": cycles,
                      "full_cycle_decisions_per_s": R / (last["cycle_wall_ms"] * 1e-3),
                      "adds_per_s": last["hashes_added"] / (last["apply_ms"] * 1e-3),
                      "adds_per_s_incl_read_table": last["hashes_added"] / (last["write_wall_ms"] * 1e-3),
                      "distinct_endpoints_picked": int(np.unique(dec["pick"][ok]).shape[0]),
                      "max_picks_on_one_endpoint": int(np.bincount(dec["pick"][ok].astype(np.int64)).max()),
                      "kernels_per_apply": int(eng.stats()["last_index_launches"]),
                      "store_device_bytes": int(eng.stats()["device_bytes"])}
        if label == "lowest_slot_ties" and orc_mod is not None:
            # CPU: the oracle's indexer applying the Adds of the first requests of the same batch to the same seeded index
            ix = orc_mod.Indexer()
            for seg_h, seg_e in zip(np.split(hs, cuts), np.split(es, cuts)):
                if len(seg_e):
                    ix.add(seg_h, int(seg_e[0]))
            n_s = min(R, 8192)
            hh, nb = eng.hash_prompts(dev_tokens[:n_s], uniform_len=w.prompt_bytes)
            hh = hh.cpu().numpy().view(np.uint64) if hasattr(hh, "cpu") else hh
            nb = nb.cpu().numpy() if hasattr(nb, "cpu") else nb
            t0 = time.perf_counter()
            tot = 0
            for r in range(n_s):
                if dec["status"][r] == 0:
                    ix.add(hh[r, : nb[r]], int(dec["pick"][r]))
                    tot += int(nb[r])
            dt = time.perf_counter() - t0
            out["cpu_adds_per_s"] = tot / dt
            out["cpu_sample"] = f"oracle indexer (C port of indexer.go Add + golang-lru), 1 thread, Adds of the first {n_s} requests"
        eng.close()
    return out


def run_gpu(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    import epp_b200 as epp
    from tools import workload_setup as helpers
    from tools import tracegen as tg

    torch.cuda.set_device(local_rank)
    numa_node, all_cpus = _bind_to_gpu_numa_node(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    epp.build.build()
    tg.build()
    w = _workload(args.workload, args.requests)
    trace = tg.Trace(w)
    lib = epp.capi.load()
    R, nbytes = w.R, w.R * w.prompt_bytes

    # this rank's batch: requests [rank*R, (rank+1)*R) of the seeded trace, generated straight into pinned memory
    pin_ptr, pin = _pinned(nbytes, lib)
    host_tokens = pin.view(np.uint32).reshape(R, w.T)
    trace.requests(rank * R, R, out=host_tokens)
    dev_tokens = torch.empty((R, w.T), dtype=torch.int32, device="cuda")
    dev_tokens.copy_(torch.from_numpy(host_tokens.view(np.int32)))
    dec_ptr, dec_pin = _pinned(R * 32, lib)
    host_dec = dec_pin.view(epp.DECISION_DTYPE)
    dev_dec = torch.empty((R, 32), dtype=torch.uint8, device="cuda")

    eng = helpers.make_engine(w, device=local_rank)
    helpers.setup_engine(eng, w, trace, filler_per_endpoint=args.index_fill)
    st0 = eng.stats()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sched_kw = dict(uniform_len=w.prompt_bytes)
    if args.pitch_pad:
        pitch = w.prompt_bytes + args.pitch_pad
        padded = torch.zeros((R, pitch), dtype=torch.uint8, device="cuda")
        padded[:, : w.prompt_bytes] = dev_tokens.view(torch.uint8).view(R, w.prompt_bytes)
        dev_tokens = padded
        offs = (torch.arange(R + 1, dtype=torch.int64, device="cuda") * pitch)
        lens = torch.full((R,), w.prompt_bytes, dtype=torch.int64, device="cuda")
        sched_kw = dict(offsets=offs, lengths=lens)
        torch.cuda.synchronize()
    # ---- value: inputs resident in HBM.  K batches are enqueued back to back (EPP_BATCH_ASYNC) and timed on the
    # device with CUDA events recorded on the engine's launch stream; the wall clock around the same region is kept
    # as a cross-check.  The clock sampler runs from the warm-up to the end of the per-kernel pass below.
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup):
        eng.schedule(dev_tokens, detail=False, out=dev_dec, **sched_kw)
    barrier()
    t0 = time.perf_counter()
    eng.event_record(0)
    for _ in range(args.steps):
        eng.schedule(dev_tokens, detail=False, out=dev_dec, asynchronous=True, **sched_kw)
    eng.event_record(1)
    eng.synchronize()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    timed_ms = eng.event_elapsed_ms()
    timed_launches = int(eng.stats()["last_kernel_launches"]) * args.steps      # kernels of one async batch x K
    if args.dump_outputs and rank == 0:
        _dump_decisions(args.dump_outputs, epp.decisions_from_torch(dev_dec))
    barrier()
    wall = max_over_ranks(wall)
    timed_ms = max_over_ranks(timed_ms)
    value = world * R * args.steps / (timed_ms * 1e-3)
    # ---- the same loop for >= 1 s (a burst of K steps is only a few ms): what the clocks settle at
    n_sus = max(args.steps, int(1.1e3 / max(timed_ms / args.steps, 1e-3)))
    barrier()
    eng.event_record(0)
    for _ in range(n_sus):
        eng.schedule(dev_tokens, detail=False, out=dev_dec, asynchronous=True, **sched_kw)
    eng.event_record(1)
    eng.synchronize()
    sus_ms = max_over_ranks(eng.event_elapsed_ms())
    value_sustained = world * R * n_sus / (sus_ms * 1e-3)
    dev_dec_async = epp.decisions_from_torch(dev_dec)      # what the timed (pipelined, detail-less) configuration decided
    # ---- per-kernel pass: the same K steps again, one at a time, each kernel bracketed by CUDA events on the launch
    # stream (roofline.launch_ms); repeated until the clock sampler has seen the GPU under this load
    kms = np.zeros(8)
    dev_ms = 0.0
    launches = 0
    probes = postings = 0
    t_k = time.perf_counter()
    n_k = 0
    while n_k < args.steps or (len(sampler.rows) < 5 and time.perf_counter() - t_k < 3.0):
        eng.schedule(dev_tokens, detail=False, out=dev_dec, **sched_kw)
        st = eng.stats()
        kms += np.array(st["last_kernel_ms"])
        dev_ms += st["last_kernels_ms"]
        launches = st["last_kernel_launches"] * args.steps
        probes, postings = st["last_probes"], st["last_postings"]
        n_k += 1
    kms *= args.steps / n_k
    dev_ms *= args.steps / n_k
    dev_ms = max_over_ranks(dev_ms)
    clocks = sampler.stop()

    # ---- e2e: host buffers through the C ABI (H2D of the prompts + D2H of the decisions inside the timed region)
    e2e_steps = max(1, min(args.steps, 10))
    e2e_wall, e2e_value, h2d_peak = float("nan"), None, None
    if not args.no_e2e:
        for _ in range(max(1, min(args.warmup, 3))):
            eng.schedule(host_tokens, uniform_len=w.prompt_bytes, detail=False, out=host_dec)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            eng.schedule(host_tokens, uniform_len=w.prompt_bytes, detail=False, out=host_dec)
        torch.cuda.synchronize()
        e2e_wall = max_over_ranks(time.perf_counter() - t0)
        barrier()
        e2e_value = world * R * e2e_steps / e2e_wall
        # sanity: device-pointer and host-pointer paths agree
        np.testing.assert_array_equal(dev_dec_async, host_dec)
        # what the link can do: a plain pinned -> device copy of the same bytes, timed with CUDA events
        pin_t = torch.from_numpy(host_tokens.view(np.int32))
        stage = torch.empty_like(dev_tokens[:, : w.T]) if args.pitch_pad else torch.empty_like(dev_tokens)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        best = float("inf")
        for _ in range(4):
            barrier()
            ev0.record()
            stage.copy_(pin_t, non_blocking=True)
            ev1.record()
            ev1.synchronize()
            best = min(best, ev0.elapsed_time(ev1))
        h2d_peak = nbytes / (max_over_ranks(best) * 1e-3) / 1e9
        del stage

    # ---- small batches: ONE synchronous epp_schedule call per batch on the raw C ABI, pinned host buffers in and out
    # (what a flush of the micro-batcher costs): median latency, decisions compared with the e2e batch's
    small = None
    if rank == 0 and not args.no_e2e:
        import ctypes as C
        small = {"how": "median of 200 synchronous epp_schedule calls per size, pinned host prompts in / decisions out, "
                        "raw C ABI (ctypes), same engine and index as `value`", "us": {}, "us_p99": {}, "decisions_equal_e2e_batch": True}
        sb = epp.capi.Batch()
        sb.uniform_len = w.prompt_bytes
        sb.data = host_tokens.ctypes.data
        small_dec = np.zeros(256, dtype=epp.DECISION_DTYPE)
        for n in (1, 16, 256):
            sb.n_requests = n
            call = lambda: lib.epp_schedule(eng._h, C.byref(sb), small_dec.ctypes.data_as(C.c_void_p), None, 0)
            for _ in range(20):
                assert call() == 0
            ts = []
            for _ in range(200):
                t0 = time.perf_counter()
                call()
                ts.append(time.perf_counter() - t0)
            small["us"][str(n)] = float(np.median(ts) * 1e6)
            small["us_p99"][str(n)] = float(np.percentile(ts, 99) * 1e6)
            small["decisions_equal_e2e_batch"] &= bool((small_dec[:n] == host_dec[:n]).all())
        small["launches_per_call"] = int(eng.stats()["last_kernel_launches"])

    full_index = None
    if world == 1 and not args.no_full_index and args.index_fill == 0:
        full_index = full_index_leg(args, w, trace, dev_tokens, dev_dec, dev_dec_async, local_rank, sched_kw, args.steps, epp, helpers)
        full_index["vs_small_index"] = full_index["value"] / value
    sharded = None
    if world > 1 and not args.no_sharded:
        sharded = sharded_leg(args, rank, world, local_rank, max(3, min(args.steps, 10)), 3)
    if rank == 0:
        peak, peak_src = _peaks()
        kms /= args.steps
        # dominant kernel = k_hash_fused (reads every prompt byte once).  Its share of the algorithmic bytes
        # A(r) = 4*T_eff + 16*P(r) + 4*M(r) + 16 + 16*E/R (SURVEY.md 8(d)) is the token term 4*T_eff.
        t_eff = min(w.T, w.block_size_tokens * w.max_prefix_blocks)
        token_bytes = R * 4 * t_eff
        algo_total = token_bytes + 16 * probes + 4 * postings + 16 * R + 16 * w.E
        dom_ms = kms[1]
        achieved = token_bytes / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
        ncu_traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            try:
                ncu_traffic = json.load(open(tpath)).get(f"{w.name}:k_hash_fused")
            except Exception:
                pass
        n_threads = os.cpu_count() or 1
        os.sched_setaffinity(0, all_cpus)            # the CPU leg gets every host core again
        cpu, odec = cpu_baseline(w, trace, n_threads, tokens=host_tokens) if not args.no_cpu else ({"value": None}, None)
        # ---- parity IN THIS RUN: the decisions of the timed configurations (async device batches; host-buffer e2e batches)
        # against the oracle decisions the CPU leg just computed for the same batch
        parity = None
        if odec is not None:
            def same(dec):
                ok = odec["status"] == 0
                pf = dec["prefill_pick"].astype(np.int64)
                pf[pf == 0xFFFFFFFF] = -1
                return bool((dec["status"] == odec["status"]).all()
                            and (dec["pick"][ok].astype(np.int64) == odec["pick"][ok]).all()
                            and (dec["score"][ok].view(np.uint64) == odec["score"][ok].view(np.uint64)).all()
                            and (dec["tie_count"][ok].astype(np.int64) == odec["tie_count"][ok]).all()
                            and (pf[ok] == odec["prefill_pick"][ok]).all())
            parity = {"requests_checked": int(odec.shape[0]), "fields": "status, pick, score bits, tie_count, prefill_pick",
                      "async_device_batches_vs_oracle": same(dev_dec_async[: odec.shape[0]]),
                      "e2e_host_batches_vs_oracle": same(host_dec[: odec.shape[0]]) if not args.no_e2e else None}
        index_write = None
        if world == 1 and not args.no_index_write:
            try:
                from oracle import pyoracle as _orc
                _orc.build()
            except Exception:
                _orc = None
            index_write = index_write_leg(args, w, trace, dev_tokens, dev_dec, local_rank, epp, helpers, None if args.no_cpu else _orc)
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": timed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64 (XXH64) + f64 (scores)", "data": "synthetic",
            "config": _config_json(w, world),
            "numa_node_of_rank0": numa_node,
            "value_sustained": value_sustained,
            "sustained": {"steps": n_sus, "seconds": sus_ms * 1e-3, "ms_per_step": sus_ms / n_sus},
            "parity_in_run": parity,
            "full_index": full_index,
            "sharded": sharded,
            "timing": "CUDA events on the engine launch stream around K back-to-back (EPP_BATCH_ASYNC) batches, max over ranks",
            "wall_ms_per_step": wall / args.steps * 1e3,
            "device_ms_per_step": dev_ms / args.steps,
            "kernel_ms_per_step": {"k_hash_fused (lengths+digests+chain)": kms[1] + kms[0] + kms[2], "match+score+pick (k_match_pick_sparse + overflow pass)": kms[3]},
            "kernel_times_how": "synchronous device batches, every kernel bracketed by CUDA events on the engine's stream",
            "algorithmic_bytes_per_step": int(algo_total),
            "algorithmic_gbs_whole_step": algo_total / (timed_ms / args.steps * 1e-3) / 1e9,
            "whole_step_frac_of_peak": (algo_total / (timed_ms / args.steps * 1e-3) / 1e9) / peak if peak else None,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(nbytes), "d2h_bytes_per_step": int(R * 32),
                    "steps": e2e_steps, "ms_per_step": e2e_wall / e2e_steps * 1e3,
                    "h2d_peak_gbs": h2d_peak,
                    "h2d_peak_how": "plain pinned -> device copy of the same bytes (torch copy_, CUDA events, best of 4), same run",
                    "achieved_gbs": (nbytes + R * 32) / (e2e_wall / e2e_steps) / 1e9 if e2e_value else None,
                    "frac_of_pcie": ((nbytes + R * 32) / (e2e_wall / e2e_steps) / 1e9) / h2d_peak if e2e_value and h2d_peak else None},
            "small_batch_latency": small,
            "gpu_launches": int(timed_launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "k_hash_fused", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak if peak else None, "traffic": ncu_traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": int(token_bytes),
                         "launch_ms": dom_ms},
            "cpu_baseline": cpu,
            "index_write": index_write,
            "index": {"pairs": st0["index_pairs"], "slots": st0["index_slots"], "filler_per_endpoint": args.index_fill,
                      "device_bytes": st0["device_bytes"], "probes_per_step": int(probes),
                      "postings_per_step": int(postings)},
        }
        print(json.dumps(out), flush=True)
    eng.close()
    lib.epp_host_free(pin_ptr)
    lib.epp_host_free(dec_ptr)
    if world > 1:
        dist.destroy_process_group()


def sharded_leg(args, rank, world, local_rank, steps, warmup, dump_dir=None):
    """BASELINE config 5: the endpoint index sharded across the GPUs (4 096 endpoints per GPU, E = 4 096 x N), every
    rank schedules the same batch of R requests; per batch two small exchanges (presence masks, best records) over
    NVLink peer memory (default) or NCCL (--sharded-nccl).  torch.distributed must be initialised when world > 1.
    Returns the result dict on rank 0, None elsewhere.  value = R decisions per step (the ranks decide TOGETHER).
    dump_dir: where rank 0 writes the decisions of the last timed step (_dump_decisions)."""
    import importlib

    import torch
    import torch.distributed as dist

    import epp_b200 as epp
    from tools import workload_setup as helpers
    from tools import tracegen as tg
    sh = importlib.import_module("llm-d-inference-scheduler_b200.sharded")

    base = tg.baseline_configs()["config5"]
    w = base.scaled(E=4096 * world, R=args.requests or base.R, name="config5")
    trace = tg.Trace(w)
    R = w.R
    host = np.empty((R, w.T), dtype=np.uint32)
    trace.requests(0, R, out=host)
    dev_tokens = torch.from_numpy(host.view(np.int32)).cuda()
    eng = helpers.make_engine(w, device=local_rank)
    eng.register_model(tg.MODEL)
    lo, hi = sh.shard_range(rank, world, w.E)
    eng.shard_set(lo, hi)
    role, kv, waiting, running = trace.pool()
    eng.pool_set(np.arange(w.E, dtype=np.uint32), role, kv, waiting, running)
    fh, _ = eng.hash_prompts(trace.family_tokens(), uniform_len=w.prompt_bytes)
    hs, es = trace.index_pairs(fh)
    keep = (es >= lo) & (es < hi)
    eng.index_load_snapshot(hs[keep], es[keep])
    d = dist if world > 1 else None

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    use_p2p = not args.sharded_nccl
    if use_p2p:
        sh.connect_p2p(eng, R, d)             # CUDA IPC handles of the exchange buffers: the only collective, once
        out_dec = torch.empty((R, 32), dtype=torch.uint8, device="cuda")
        step = lambda: sh.schedule_sharded_p2p(eng, dev_tokens, w.prompt_bytes, out=out_dec)
    else:
        step = lambda: sh.schedule_sharded(eng, dev_tokens, w.prompt_bytes, d)
    for _ in range(warmup):
        dec = step()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record()
    for _ in range(steps):
        dec = step()
    ev1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    if dump_dir and rank == 0:
        _dump_decisions(dump_dir, epp.decisions_from_torch(dec))
    barrier()
    if world > 1:
        t = torch.tensor([wall], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        wall = float(t.item())
    parity = None
    if rank == 0:
        # the sharded decisions must equal what ONE engine holding the whole index decides
        n_chk = min(R, 4096)
        full = helpers.make_engine(w, device=local_rank)
        full.register_model(tg.MODEL)
        full.pool_set(np.arange(w.E, dtype=np.uint32), role, kv, waiting, running)
        full.index_load_snapshot(hs, es)
        ref_dec, _ = full.schedule(host[:n_chk], uniform_len=w.prompt_bytes, detail=False)
        got = epp.decisions_from_torch(dec)[:n_chk]
        parity = bool((got["status"] == ref_dec["status"]).all() and (got["pick"] == ref_dec["pick"]).all()
                      and (got["score"].view(np.uint64) == ref_dec["score"].view(np.uint64)).all()
                      and (got["tie_count"] == ref_dec["tie_count"]).all())
        full.close()
    res = None
    if rank == 0:
        W = (w.max_prefix_blocks + 31) // 32
        res = {"value": R * steps / wall, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
               "ms_per_step": wall / steps * 1e3, "timing": "host clock around K blocking steps, max over ranks (every step ends with a stream synchronisation)",
               "endpoints": w.E, "batch_requests": R,
               "exchange": ("NVLink peer memory: masks OR-reduced and best records merged straight out of the peers' buffers by "
                            "the engine's own kernels (CUDA IPC, release/acquire flags; no NCCL on the data path)" if use_p2p
                            else "NCCL all-gathers + torch OR (--sharded-nccl)"),
               "exchange_bytes_per_rank_per_step": {"presence_masks": int(R * W * 4), "best_records": int(R * 24)},
               "decisions_ok": int((epp.decisions_from_torch(dec)["status"] == 0).sum()),
               "parity_vs_unsharded": parity, "parity_requests_checked": min(R, 4096),
               "config": _config_json(w, world, {
                   "parallelism": f"endpoint index sharded over {world} GPUs (4096 endpoints each); every rank schedules the same batch"})}
    eng.close()
    del dev_tokens
    torch.cuda.empty_cache()
    return res


def run_gpu_sharded(args, rank, world, local_rank):
    """--workload config5: only the endpoint-sharded leg, as its own JSON line."""
    import torch
    import torch.distributed as dist

    import epp_b200 as epp
    from tools import tracegen as tg

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    epp.build.build()
    tg.build()
    res = sharded_leg(args, rank, world, local_rank, args.steps, args.warmup, dump_dir=args.dump_outputs)
    if rank == 0:
        out = {"metric": METRIC + " (endpoint-sharded index)", "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
               "dtype": "u64 (XXH64) + f64 (scores)", "data": "synthetic"}
        out.update(res)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def full_index_leg(args, w, trace, dev_tokens, dev_dec, ref_dec, local_rank, sched_kw, steps, epp, helpers):
    """The same batch against a PRODUCTION-SIZE index: every endpoint's LRU full (31 250 blocks per endpoint, the
    reference default, approximateprefix/types.go:110) -> 1.29e8 pairs, a table far larger than L2.  The filler
    hashes never match a prompt, so the decisions must not change."""
    import torch
    per = 31250
    eng = helpers.make_engine(w, device=local_rank)
    t0 = time.perf_counter()
    helpers.setup_engine(eng, w, trace, filler_per_endpoint=per)
    setup_s = time.perf_counter() - t0
    st = eng.stats()
    for _ in range(3):
        eng.schedule(dev_tokens, detail=False, out=dev_dec, **sched_kw)
    torch.cuda.synchronize()
    eng.event_record(0)
    for _ in range(steps):
        eng.schedule(dev_tokens, detail=False, out=dev_dec, asynchronous=True, **sched_kw)
    eng.event_record(1)
    eng.synchronize()
    ms = eng.event_elapsed_ms() / steps
    same = bool((epp.decisions_from_torch(dev_dec).view(np.uint8) == ref_dec.view(np.uint8)).all())
    eng.schedule(dev_tokens, detail=False, out=dev_dec, **sched_kw)
    k = eng.stats()["last_kernel_ms"]
    out = {"value": w.R / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps, "filler_per_endpoint": per,
           "index_pairs": int(st["index_pairs"]), "index_slots": int(st["index_slots"]),
           "index_table_bytes": int(st["index_slots"]) * 32, "device_bytes": int(st["device_bytes"]),
           "decisions_equal_to_small_index": same, "setup_s": setup_s,
           "kernel_ms": {"hash": k[0] + k[1] + k[2], "match+score+pick": k[3]}}
    eng.close()
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="config3", choices=["config1", "config2", "config3", "config4", "config5"])
    ap.add_argument("--requests", type=int, default=0, help="override the batch size R (0 = the config's)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--sharded-nccl", action="store_true",
                    help="config5: exchange masks / records with NCCL all-gathers instead of the peer-memory kernels")
    ap.add_argument("--no-index-write", action="store_true", help="skip the index write-side leg (SURVEY 8(f).1)")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer e2e leg (profiling runs only)")
    ap.add_argument("--no-full-index", action="store_true", help="skip the production-size-index leg")
    ap.add_argument("--no-sharded", action="store_true", help="N > 1: skip the endpoint-sharded (config 5) leg")
    ap.add_argument("--index-fill", type=int, default=0,
                    help="extra never-matching index entries per endpoint (31250 = every endpoint's LRU full: 1.28e8 pairs, "
                         "a table far larger than L2); decisions are unchanged")
    ap.add_argument("--pitch-pad", type=int, default=0,
                    help="experiment: lay the device-resident prompts out with this many pad bytes between requests")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the decisions of the last timed step as DIR/<field>.npy (float64) to compare builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the CUDA engine decided: it needs --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.workload == "config5":
        run_gpu_sharded(args, rank, world, local_rank)
        return
    run_gpu(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
