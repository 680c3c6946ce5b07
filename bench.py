#!/usr/bin/env python3
"""bench.py — ECDSA-P256 verifies/s at batch = 64K (BASELINE.json configs[1]) on N B200s.

A "step" is one pass of the hot path over one 65,536-signature batch PER GPU (batches shard embarrassingly, so per-GPU
work is fixed as N grows: weak scaling); with N > 1 every step ends with the all-gather of the packed verdict bitmask
over NCCL, issued by the engine itself (sbv_gather_verdicts_device: k_pack_bits + ncclAllGather, ordered behind the step on its stream) —
the only exchange the path has.  No PyTorch kernel runs inside a step.

  value      device-timed, inputs already resident in HBM (16 rotating copies = 168 MB > L2), steps rotating over 4 streams
  e2e        the same metric through the C ABI with pinned HOST buffers (sbv_verify_batch; sbv_verify_batch_ranked when
             N > 1, i.e. INCLUDING the gather): H2D of the 160 B/item batch and D2H of the verdicts inside the timed region
  roofline   dominant kernel (k_verify_kt: the fixed-base kernel the repeated keys of the batch take): achieved wide-MAC/s
             (canonical W = 272,256 MAC32 per verify, SURVEY §8d) over its CUDA-event duration vs the IMAD.WIDE peak probed
             in the same run; given for the isolated launch and for the pipelined steps; HBM fraction beside it
  cpu_baseline  OpenSSL ECDSA_do_verify (oracle/, the stand-in for Go crypto/ecdsa — no Go toolchain exists here) on all
             host cores, same batch, rank 0 / N=1 only
  extras     the other BASELINE configs, each checked against the oracle in the run: C3 (SHA-256 + verify, 1M requests),
             C4 (n=16 commit-vote quorum stream, 262,144 signatures, sharded by instance over the ranks), C5 (mixed curves)

`--impl reference` times the CPU implementation alone (the reference arm).
`--dump-outputs DIR` writes the verdicts of the last timed step as float32 .npy files; the inputs are seeded, so two
builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH = 65536
KEYS = 1024
MAC32_PER_VERIFY = 272_256       # SURVEY.md §8d canonical count (P-256)
MAC32_PER_VERIFY_P384 = 902_880
EXECUTED_MAC32_PER_VERIFY = 68 * (8 * 64 + 3 * 36) + (2 * 64 + 36)   # fixed-base path, P-256 (DESIGN.md §6)
BYTES_PER_VERIFY = 161           # 160 B in + 1 B out
N_COPIES = 16                    # rotating input copies: 16 x 10.5 MB > 126 MB L2
N_LANES = int(os.environ.get("SBV_BENCH_LANES", "4"))   # CUDA streams the device-timed steps rotate over
METRIC = "ECDSA-P256 verifies/sec at batch=64K"
WORKLOAD = "C2: ECDSA-P256 batch verify, 65,536 synthetic sigs per GPU, 1,024 keys, 1/16 corrupted"


def base_config(world):
    """The workload — the same dict, key for key, in both arms (the driver compares them)."""
    return {"workload": WORKLOAD, "batch_per_gpu": BATCH, "keys": KEYS, "seed": "1 + 1000*rank", "sharding": f"batch-parallel x{world}",
            "l2": f"GPU arm: {N_COPIES} rotating input copies per rank (168 MB > 126 MB L2), no flush needed; CPU arm: the rank-0 batch (10.5 MB) every step"}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    # (no power.draw: the power sensor read is the one query that can hold the GPU for milliseconds)
    Q = ("index,clocks.sm,clocks.max.sm,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.rows = []
        self.marks = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def mark(self):
        self.marks.append(time.perf_counter())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        lo, hi = (self.marks + [0, 1e30])[:2] if len(self.marks) >= 2 else (0, 1e30)
        sm, mx, reasons, sm_all = [], [], set(), []
        for ts, row in self.rows:
            f = [x.strip() for x in row.split(",")]
            if len(f) < 8:
                continue
            try:
                v, m = float(f[1]), float(f[2])
            except ValueError:
                continue
            sm_all.append(v)
            mx.append(m)
            if lo - 0.06 <= ts <= hi + 0.06:     # samples taken while the timed region ran
                sm.append(v)
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        use = sorted(sm or sm_all)
        return {"sm_mhz": use[len(use) // 2] if use else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_total": len(sm_all)}


def make_workload(rank: int):
    import oracle  # corpus generator + CPU baseline live in the oracle package (test/bench infrastructure)
    from oracle import corpus
    return corpus.make_batch(oracle.P256, n=BATCH, K=KEYS, seed=1 + 1000 * rank)


def run_reference(args, rank, world):
    """Reference arm: the CPU implementation of the path on the box's host cores."""
    if rank != 0:
        return
    import oracle
    b = make_workload(0)
    cores = oracle.ncores()
    keys = b["keys"]
    for _ in range(max(args.warmup, 1)):
        oracle.bench_verify(oracle.P256, b["r"][:8192], b["s"][:8192], keys, b["key_idx"][:8192], b["digest"][:8192], nthreads=cores)
    total = 0.0
    for _ in range(args.steps):
        t, ok = oracle.bench_verify(oracle.P256, b["r"], b["s"], keys, b["key_idx"], b["digest"], nthreads=cores)
        total += t
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"verdicts": ok})
    value = BATCH * args.steps / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "verifies/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32 limbs (integer)", "data": "synthetic",
        "config": base_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": "verifies/s", "cores": cores, "kind": "port",
                         "sample": f"{args.steps} x the full 65,536-signature batch of rank 0, OpenSSL 3.0 ECDSA_do_verify (stand-in for Go crypto/ecdsa)"},
        "e2e": {"value": value, "unit": "verifies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def pack_bits(ok):
    import numpy as np
    return np.packbits(ok.astype(np.uint8), bitorder="little").view(np.uint32)


def dump_outputs(out_dir, arrays):
    """Writes each array as out_dir/<name>.npy in float32 (verdicts are 0/1, so the conversion is exact): what the timed
    path returned in its last step, for comparing two builds output for output on the same seeded inputs."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a, dtype=np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="sbv", choices=["sbv", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the verdicts of the last one as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    import consensus_b200 as sbv
    import oracle

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    b = make_workload(rank)
    eng = sbv.Engine(devices=[local_rank])
    # one-process-per-GPU: the engines form their own NCCL communicators (one channel per concurrent stream / caller);
    # torch.distributed only carries the 128-byte ids and the final max-over-ranks
    # caller threads of the e2e leg: four keep one GPU busy; on the 8-GPU box three measured better than four
    # (profiles/r02_scaling.txt: the ranks' synchronous calls meet in a gather every call, and more callers per rank made
    # the slowest rank slower), so N = 8 runs with three
    e2e_threads = int(os.environ.get("SBV_BENCH_E2E_THREADS", "4" if world <= 4 else "3"))
    n_channels = N_LANES + e2e_threads
    if world > 1:
        for ch in range(n_channels):
            uid = torch.zeros(128, dtype=torch.uint8, device=dev)
            if rank == 0:
                uid.copy_(torch.frombuffer(bytearray(sbv.Engine.comm_unique_id()), dtype=torch.uint8))
            dist.broadcast(uid, 0)
            got = eng.comm_init_rank(bytes(uid.cpu().numpy().tobytes()), world, rank)
            assert got == ch

    fields = ("r", "s", "qx", "qy", "digest")
    host = {k: torch.from_numpy(np.ascontiguousarray(b[k])).pin_memory() for k in fields}
    copies = [{k: host[k].to(dev, non_blocking=True) for k in fields} for _ in range(N_COPIES)]
    d_ok = torch.zeros(BATCH, dtype=torch.uint8, device=dev)
    words = BATCH // 32
    stream = torch.cuda.current_stream().cuda_stream
    # Consecutive steps are independent batches, so they are enqueued round-robin on four streams: the latency-bound
    # heads of step i+1 (key grouping, table construction, scalar preparation) overlap the verify kernel of step i.
    # Every step still does all of its work; the timed region is bracketed by events on the main stream that wait for all.
    lanes = [torch.cuda.Stream(device=dev) for _ in range(N_LANES)]
    d_oks = [torch.zeros(BATCH, dtype=torch.uint8, device=dev) for _ in range(N_LANES)]
    d_masks = [torch.zeros(world * words, dtype=torch.int32, device=dev) for _ in range(N_LANES)]

    def device_step(i, pipelined=True):
        c = copies[i % N_COPIES]
        if not pipelined:
            eng.verify_batch_device(sbv.P256, BATCH, c["r"].data_ptr(), c["s"].data_ptr(), c["qx"].data_ptr(), c["qy"].data_ptr(),
                                    c["digest"].data_ptr(), 32, d_ok.data_ptr(), stream=stream)
            return
        k = i % N_LANES
        eng.verify_batch_device(sbv.P256, BATCH, c["r"].data_ptr(), c["s"].data_ptr(), c["qx"].data_ptr(), c["qy"].data_ptr(),
                                c["digest"].data_ptr(), 32, d_oks[k].data_ptr(), stream=lanes[k].cuda_stream)
        if world > 1:   # engine-side pack + NCCL all-gather, on the step's own stream and channel
            eng.gather_verdicts_device(k, d_oks[k].data_ptr(), BATCH, d_masks[k].data_ptr(), stream=lanes[k].cuda_stream)

    def join_lanes():
        for lane in lanes:
            torch.cuda.current_stream().wait_stream(lane)

    def fork_lanes():
        for lane in lanes:
            lane.wait_stream(torch.cuda.current_stream())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- correctness gate: the verdicts of this run must equal the oracle's ----
    want = oracle.verify_batch(oracle.P256, b["r"], b["s"], b["qx"], b["qy"], b["digest"])
    device_step(0, pipelined=False)
    torch.cuda.synchronize()
    if not np.array_equal(d_ok.cpu().numpy(), want):
        raise SystemExit("bench: GPU verdicts differ from the oracle — refusing to report a number")
    want_mask_all = None
    if world > 1:   # what every rank's gathered mask must hold: the packed oracle verdicts of all ranks
        mine = torch.from_numpy(pack_bits(want).view(np.int32).copy()).to(dev)
        allm = torch.zeros(world * words, dtype=torch.int32, device=dev)
        dist.all_gather_into_tensor(allm, mine)
        want_mask_all = allm.cpu().numpy()

    # ---- device-timed value ----
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()          # before the warm-up and the barrier: the fork of nvidia-smi is nobody's timed region
    for i in range(args.warmup):
        device_step(i)
    join_lanes()
    barrier()
    launches0 = eng.kernel_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.mark()
    e0.record()
    fork_lanes()
    diag = os.environ.get("SBV_BENCH_DIAG", "0") != "0"   # per-step completion events cost 4-5 % of the throughput (profiles/r02_variants.md): off by default
    step_done = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps if diag else 0)]
    for i in range(args.steps):
        device_step(args.warmup + i)
        if diag:
            step_done[i].record(lanes[(args.warmup + i) % N_LANES])   # diagnostic only: when each step finished (timing_diag below)
    join_lanes()
    e1.record()
    torch.cuda.synchronize()
    sampler.mark()
    done_ms = sorted(e0.elapsed_time(ev) for ev in step_done) or [0.0]
    gaps = sorted(b - a for a, b in zip([0.0] + done_ms[:-1], done_ms))
    timing_diag = None if not diag else {"step_completion_gap_ms": {"median": gaps[len(gaps) // 2], "p99": gaps[min(len(gaps) - 1, int(len(gaps) * 0.99))], "max": gaps[-1]},
                   "first_step_done_ms": done_ms[0], "step_done_ms": [round(x, 3) for x in done_ms[:64]],
                   "note": "gaps between consecutive step completions inside the timed region (all streams merged): a max far above the median is a "
                           "stall of the whole device (e.g. a management query), not arithmetic"}
    launches = eng.kernel_launches - launches0
    barrier()
    dev_ms = max_over_ranks(e0.elapsed_time(e1))
    for k in range(N_LANES):
        if not np.array_equal(d_oks[k].cpu().numpy(), want):
            raise SystemExit("bench: pipelined verdicts differ from the oracle")
        if world > 1 and not np.array_equal(d_masks[k].cpu().numpy(), want_mask_all):
            raise SystemExit("bench: gathered verdict mask differs from the packed oracle verdicts of all ranks")
    if args.dump_outputs and rank == 0:
        # the lane of the last timed step; the registered-key leg below reuses these buffers
        last = (args.warmup + args.steps - 1) % N_LANES
        outputs = {"verdicts": d_oks[last].cpu().numpy()}
        if world > 1:   # the gathered mask every rank receives, one 0/1 entry per item of all ranks
            outputs["gathered_verdicts"] = np.unpackbits(d_masks[last].cpu().numpy().view(np.uint8), bitorder="little")
        dump_outputs(args.dump_outputs, outputs)
    clocks = sampler.stop() if rank == 0 else None
    value = world * BATCH * args.steps / (dev_ms * 1e-3)

    # single-stream steps (no overlap): step latency, and the CUDA-event duration of the dominant kernel
    # (kernel durations are only meaningful when launches do not share the SMs)
    eng.profile_enable(True)
    l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0.record()
    for i in range(20):
        device_step(i, pipelined=False)
    l1.record()
    torch.cuda.synchronize()
    step_latency_ms = l0.elapsed_time(l1) / 20
    prep_ms, verify_ms, pairs = eng.profile_read()
    eng.profile_enable(False)

    # ---- end-to-end through the C ABI with pinned host buffers ----
    # Host threads each keep one synchronous call in flight (the reference calls its Verifier from concurrent goroutines,
    # view.go:537-541 / consensus.go:302-306); every call does H2D of its 160 B/item batch, the whole pipeline and the
    # D2H of its verdicts — and, with N > 1, the NCCL all-gather of the packed verdicts plus the D2H of the gathered mask.
    E2E_THREADS = e2e_threads
    ptr = {k: host[k].data_ptr() for k in fields}
    host_oks = [torch.zeros(BATCH, dtype=torch.uint8).pin_memory() for _ in range(E2E_THREADS)]
    host_masks = [torch.zeros(world * words, dtype=torch.int32).pin_memory() for _ in range(E2E_THREADS)]

    def e2e_calls(tid, count):
        for _ in range(count):
            if world == 1:
                eng.verify_batch_ptr(sbv.P256, BATCH, ptr["r"], ptr["s"], ptr["qx"], ptr["qy"], ptr["digest"], 32, host_oks[tid].data_ptr())
            else:
                eng.verify_batch_ranked_ptr(N_LANES + tid, sbv.P256, BATCH, ptr["r"], ptr["s"], ptr["qx"], ptr["qy"], ptr["digest"], 32,
                                            host_oks[tid].data_ptr(), host_masks[tid].data_ptr())

    def e2e_run(total, nthreads=E2E_THREADS):
        ths = [threading.Thread(target=e2e_calls, args=(t, total // nthreads + (t < total % nthreads))) for t in range(nthreads)]
        for t in ths: t.start()
        for t in ths: t.join()

    e2e_run(2 * args.warmup)
    barrier()
    t0 = time.perf_counter()
    e2e_run(args.steps)
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    for tid in range(E2E_THREADS):
        if not np.array_equal(host_oks[tid].numpy(), want):
            raise SystemExit("bench: e2e verdicts differ from the oracle")
        if world > 1 and not np.array_equal(host_masks[tid].numpy(), want_mask_all):
            raise SystemExit("bench: e2e gathered mask differs from the packed oracle verdicts of all ranks")
    e2e_value = world * BATCH * args.steps / e2e_s
    # one caller, one call at a time: the latency-bound form of the same number
    barrier()
    t0 = time.perf_counter()
    e2e_calls(0, 20)
    e2e_single = world * BATCH * 20 / max_over_ranks(time.perf_counter() - t0)

    # ---- registered-key path (extra, NOT the headline): keys registered once with sbv_set_keys.  Same signatures;
    # expected verdicts recomputed against the registered key of each item.
    reg = None
    try:
        keys = b["keys"]
        t0 = time.perf_counter()
        eng.set_keys(np.zeros(KEYS, np.uint8), keys.reshape(KEYS, 2, 32))
        set_keys_first_s = time.perf_counter() - t0      # includes the first allocation of the table memory
        t0 = time.perf_counter()
        eng.set_keys(np.zeros(KEYS, np.uint8), keys.reshape(KEYS, 2, 32))
        set_keys_s = time.perf_counter() - t0
        want_reg = oracle.verify_batch(oracle.P256, b["r"], b["s"], np.ascontiguousarray(keys[b["key_idx"], :32]),
                                       np.ascontiguousarray(keys[b["key_idx"], 32:]), b["digest"])
        d_slot = torch.from_numpy(b["key_idx"].astype(np.int32)).to(dev)

        def reg_step(i, pipelined=True):
            c = copies[i % N_COPIES]
            st, out = (stream, d_ok) if not pipelined else (lanes[i % N_LANES].cuda_stream, d_oks[i % N_LANES])
            eng.verify_registered_device(sbv.P256, BATCH, d_slot.data_ptr(), c["r"].data_ptr(), c["s"].data_ptr(), c["digest"].data_ptr(), 32,
                                         out.data_ptr(), stream=st)
        for i in range(args.warmup):
            reg_step(i, pipelined=False)
        torch.cuda.synchronize()
        if not np.array_equal(d_ok.cpu().numpy(), want_reg):
            raise RuntimeError("registered-key verdicts differ from the oracle")
        barrier()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        fork_lanes()
        for i in range(args.steps):
            reg_step(i)
        join_lanes()
        r1.record()
        barrier()
        reg_ms = max_over_ranks(r0.elapsed_time(r1))
        for k in range(N_LANES):
            if not np.array_equal(d_oks[k].cpu().numpy(), want_reg):
                raise RuntimeError("pipelined registered-key verdicts differ from the oracle")
        q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        q0.record()
        for i in range(20):
            reg_step(i, pipelined=False)
        q1.record()
        torch.cuda.synchronize()
        reg = {"value": world * BATCH * args.steps / (reg_ms * 1e-3), "unit": "verifies/s", "ms_per_step": reg_ms / args.steps,
               "step_latency_ms": q0.elapsed_time(q1) / 20, "keys": KEYS, "set_keys_seconds": set_keys_s, "set_keys_first_call_seconds": set_keys_first_s,
               "note": "sbv_set_keys + sbv_verify_registered: per-key tables (8-bit signed windows, 264 KiB/key) built once per verification sequence"}
    except Exception as ex:  # the extra must never take the headline down
        reg = {"error": str(ex)}

    # ---- roofline of the dominant kernel ----
    mad_peak = eng.probe_mad_rate()                      # wide MAC32/s, measured in this run
    hbm_gbs, hbm_src = load_peaks()
    k_ms = verify_ms / max(pairs, 1)                     # average launch duration of the dominant kernel (CUDA events, isolated steps)
    mac_rate = BATCH * MAC32_PER_VERIFY / (k_ms * 1e-3)
    roofline = {
        "bound": "int32-mad (IMAD.WIDE issue rate; neither hbm nor tensor binds this path)",
        "kernel": "k_gpart + k_verify_kt<P256,5> (the two halves of the fixed-base verification of the key-grouped pipeline: u1*G, then the key's windows)", "achieved": mac_rate / 1e12, "peak": mad_peak / 1e12,
        "unit": "TMAC32/s", "frac": mac_rate / mad_peak if mad_peak else None, "peak_source": "sbv_probe_mad_rate, same run",
        "kernel_ms": k_ms, "prep_and_grouping_ms": prep_ms / max(pairs, 1), "step_latency_ms": step_latency_ms,
        "frac_whole_step_isolated": BATCH * MAC32_PER_VERIFY / (step_latency_ms * 1e-3) / mad_peak if mad_peak else None,
        "frac_pipelined": value / world * MAC32_PER_VERIFY / mad_peak if mad_peak else None,
        # what the two kernels actually execute: 68 mixed additions of 8 products (64 MAC32) + 3 squarings (36 MAC32) and the
        # final check, per verify — against the same wide-MAD peak
        "executed_mac32_per_verify": EXECUTED_MAC32_PER_VERIFY,
        "frac_executed": BATCH * EXECUTED_MAC32_PER_VERIFY / (k_ms * 1e-3) / mad_peak if mad_peak else None,
        "note": "W = 272,256 MAC32 is SURVEY §8d's canonical double-scalar multiplication; the key-grouped pipeline does less arithmetic per "
                "verify than the canonical algorithm (no doublings for repeated keys), so the fraction can exceed 1",
        "traffic": None, "algorithmic_bytes_per_launch": BATCH * BYTES_PER_VERIFY,
        "hbm": {"achieved": BATCH * BYTES_PER_VERIFY / (k_ms * 1e-3) / 1e9, "peak": hbm_gbs, "unit": "GB/s",
                "frac": BATCH * BYTES_PER_VERIFY / (k_ms * 1e-3) / 1e9 / hbm_gbs, "peak_source": hbm_src},
    }
    tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            roofline["traffic"] = tj.get("dram_bytes_per_launch")
            roofline["traffic_source"] = tj.get("source")
        except Exception:
            pass

    cfg = base_config(world)
    execution = dict({         # how THIS arm runs the workload (kept out of `config` so that both arms' configs are identical)
                "pipelining": f"consecutive steps rotate over {N_LANES} CUDA streams; unpipelined step latency in step_latency_ms",
                "exchange": "engine-side k_pack_bits + ncclAllGather of the packed verdict bitmask per step, ordered behind the step on its stream (run on the channel's high-priority stream)" if world > 1 else "none (1 GPU)",
                "key_grouping": "on (threshold 16): per-key fixed-base tables rebuilt inside every step"})
    line = {
        "metric": METRIC, "value": value, "unit": "verifies/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32 limbs (integer)", "data": "synthetic", "config": cfg, "execution": execution,
        "e2e": {"value": e2e_value, "unit": "verifies/s", "h2d_bytes_per_step": 160 * BATCH * world,
                "d2h_bytes_per_step": (BATCH + (world * words * 4 if world > 1 else 0)) * world,
                "callers": E2E_THREADS, "single_caller_value": e2e_single, "includes_gather": world > 1},
        "step_latency_ms": step_latency_ms, "gpu_launches": int(launches), "roofline": roofline, "clocks": clocks, "timing_diag": timing_diag, "registered_keys": reg,
    }

    if not args.no_extras:
        try:
            line["extras"] = run_extras(eng, sbv, oracle, np, torch, dev, rank, world, local_rank, mad_peak, hbm_gbs, dist, max_over_ranks, barrier)
        except Exception as ex:
            line["extras"] = {"error": repr(ex)}

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = oracle.ncores()
        reps = 4
        tot = 0.0
        for _ in range(reps):
            t, okc = oracle.bench_verify(oracle.P256, b["r"], b["s"], b["keys"], b["key_idx"], b["digest"], nthreads=cores)
            tot += t
        line["cpu_baseline"] = {"value": BATCH * reps / tot, "unit": "verifies/s", "cores": cores, "kind": "port",
                                "sample": f"{reps} x the full 65,536-signature batch; OpenSSL 3.0 ECDSA_do_verify on pre-built keys "
                                          "(stand-in for Go crypto/ecdsa: no Go toolchain)"}
    eng.close()
    if rank == 0 and world == 1:
        # consensus tx/s at n=4 (BASELINE configs[0]): in-process normal-path simulator, 1,000 txs,
        # RequestBatchMaxCount = 100; accept-all (= stock naive_chain) vs per-call CPU verifier vs GPU verifier
        sim = os.path.join(ROOT, "consensus_b200", "host", "sim")
        try:
            out = subprocess.run([sim, "1000", "100", "1"], capture_output=True, text=True, timeout=300)
            line["consensus_n4"] = json.loads(out.stdout.strip().splitlines()[-1])
        except Exception as ex:
            line["consensus_n4"] = {"error": str(ex)}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_extras(eng, sbv, oracle, np, torch, dev, rank, world, local_rank, mad_peak, hbm_gbs, dist, max_over_ranks, barrier):
    """The other BASELINE configs, each verified against the oracle inside the run.  C4 runs at every N (sharded by
    instance over the ranks, `reached` bitmask gathered by the engine over NCCL); C3 and C5 at N = 1."""
    from oracle import corpus
    from oracle import ecdsa_ref as ref
    ex = {}
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()

    def best_of(fn, reps=3):
        for _ in range(8):      # one warm-up call per scratch set of the engine (each grows its buffers on first use)
            fn()
        best = 1e30
        for _ in range(reps):
            barrier()
            t0 = time.perf_counter()
            fn()
            best = min(best, max_over_ranks(time.perf_counter() - t0))
        return best

    # ---- C4: n=16, f=5, Q=11: 17,476 instances x 15 foreign votes = 262,140 commit votes (+4 padding votes) ----
    I, NV = 17476, 15
    tile = corpus.make_batch(oracle.P256, n=BATCH, K=16, seed=61, corrupt_rate=16)     # 16 consenter keys
    want_tile = oracle.verify_batch(oracle.P256, tile["r"], tile["s"], tile["qx"], tile["qy"], tile["digest"])
    total = I * NV + 4
    rep4 = lambda a: np.ascontiguousarray(np.concatenate([a] * 4)[:total])
    inst = np.concatenate([np.repeat(np.arange(I, dtype=np.uint32), NV), np.full(4, I - 1, np.uint32)])
    g = ref.DRBG(6)
    sender = ((np.arange(total) % NV) + 1).astype(np.uint16)
    signer = sender.copy()
    dm = np.ones(total, np.uint8)
    dm[-4:] = 0                                           # padding votes
    rnd = np.frombuffer(b"".join(g.block(i) for i in range((total + 31) // 32)), np.uint8)[:total]
    dup = (rnd % 29) == 0
    sender[dup] = np.roll(sender, 1)[dup]                 # duplicate sender: the second vote must not count
    signer[dup] = sender[dup]
    wrong_signer = (rnd % 31) == 1
    signer[wrong_signer] = (signer[wrong_signer] % NV) + 1 + (signer[wrong_signer] % NV == sender[wrong_signer] - 1)
    dm[(rnd % 37) == 2] = 0                               # wrong digest
    ok_all = rep4(want_tile)
    self_id = np.zeros(I, np.uint16)                      # node 0 counts the votes of nodes 1..15
    want_cnt, want_reached = ref.count_commit_votes_batch(inst, sender, signer, dm, ok_all, I, 10, self_id)
    # shard by instance over the ranks (instance ids local to the rank's shard: every engine counts from 0)
    from consensus_b200 import sharding
    vlo, vhi, ilo, ihi, local_inst = sharding.shard_votes(inst, I, rank, world)
    sl = slice(vlo, vhi)
    F = {k: pin(rep4(tile[k])[sl]) for k in ("r", "s", "qx", "qy", "digest")}
    cols = [pin(local_inst), pin(sender[sl]), pin(signer[sl]), pin(dm[sl]), pin(self_id[ilo:ihi])]
    nv, ni = vhi - vlo, ihi - ilo
    ok_h, cnt_h, rch_h = pin(np.zeros(nv, np.uint8)), pin(np.zeros(ni, np.uint32)), pin(np.zeros(ni, np.uint8))
    wi = (I // world + 1 + 31) // 32
    d_rch_all = torch.zeros(world * wi, dtype=torch.int32, device=dev)
    vp = ctypes.c_void_p

    def c4():
        eng._check(eng._lib.sbv_verify_quorum(eng._h, ctypes.c_uint8(0), ctypes.c_size_t(nv), vp(F["r"].data_ptr()), vp(F["s"].data_ptr()),
                                              vp(F["qx"].data_ptr()), vp(F["qy"].data_ptr()), vp(F["digest"].data_ptr()), ctypes.c_uint8(32),
                                              vp(cols[0].data_ptr()), vp(cols[1].data_ptr()), vp(cols[2].data_ptr()), vp(cols[3].data_ptr()),
                                              ctypes.c_size_t(ni), vp(cols[4].data_ptr()), ctypes.c_uint32(10), vp(ok_h.data_ptr()),
                                              vp(cnt_h.data_ptr()), vp(rch_h.data_ptr())), "sbv_verify_quorum")
        if world > 1:   # every rank learns which instances reached quorum: one NCCL all-gather of the packed bits
            packed = np.zeros(wi * 4, np.uint8)
            pb = np.packbits(rch_h.numpy(), bitorder="little")
            packed[:pb.size] = pb
            mine = torch.from_numpy(packed.view(np.int32).copy())
            d_rch_all[rank * wi:(rank + 1) * wi].copy_(mine, non_blocking=True)
            eng.gather_words_device(0, d_rch_all.data_ptr(), wi, stream=torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()

    t = best_of(c4)
    good = (np.array_equal(ok_h.numpy(), ok_all[sl]) and np.array_equal(cnt_h.numpy(), want_cnt[ilo:ihi]) and np.array_equal(rch_h.numpy(), want_reached[ilo:ihi]))
    if world > 1:
        allw = d_rch_all.cpu().numpy().view(np.uint8)
        for r_ in range(world):
            a, bnd = I * r_ // world, I * (r_ + 1) // world
            bits = np.unpackbits(allw[r_ * wi * 4:(r_ + 1) * wi * 4], bitorder="little")[:bnd - a]
            good = good and np.array_equal(bits, want_reached[a:bnd])
    ex["c4_quorum_stream"] = {"workload": "C4: n=16 f=5 Q=11 commit votes, 17,476 instances x 15 votes = 262,144 signatures per batch (whole job), 16 consenter keys, "
                                          "Byzantine votes: bad signature / wrong digest / duplicate sender / signer != sender",
                              "votes": total, "instances": I, "e2e_s": t, "value": total / t, "unit": "votes/s", "n_gpus": world, "scaling": "strong",
                              "through": "sbv_verify_quorum (pinned host buffers: H2D of the votes, verify, count, D2H of verdicts / counts / reached)"
                                         + (" + engine NCCL all-gather of the reached bitmask" if world > 1 else ""),
                              "reached": int(want_reached.sum()), "bit_exact_vs_oracle": bool(good),
                              "roofline_frac_canonical": total / t * MAC32_PER_VERIFY / (mad_peak * world) if mad_peak else None}
    if world > 1 or rank != 0:
        return ex

    # ---- C3: SHA-256 digest + ECDSA verify fused, 1,048,576 requests of 256 B, 4,096 client keys ----
    T16 = 16
    msgs1, off1 = corpus.make_requests(BATCH, seed=5, fixed_len=256)
    dig1 = oracle.sha256_batch(msgs1, off1)
    d, kxy = corpus.make_keys(oracle.P256, 4096, seed=71)
    kidx = (np.arange(BATCH) % 4096).astype(np.uint32)
    r1, s1 = oracle.sign_batch(oracle.P256, d, kidx, dig1, corpus._blocks(73, BATCH, 32, b"k"))
    bad = (np.arange(BATCH) % 16) == 5
    msgs1 = msgs1.copy()
    msgs1[np.nonzero(bad)[0] * 256 + 17] ^= 0x40          # "flip one payload bit" class
    want1 = oracle.verify_batch(oracle.P256, r1, s1, kxy[kidx, :32].copy(), kxy[kidx, 32:].copy(), oracle.sha256_batch(msgs1, off1))
    n3 = BATCH * T16
    rep = lambda a: np.ascontiguousarray(np.tile(a, (T16, 1)))
    M, OFF = pin(np.tile(msgs1, T16)), pin(np.arange(n3 + 1, dtype=np.uint64) * 256)
    R, S, QX, QY = pin(rep(r1)), pin(rep(s1)), pin(rep(kxy[kidx, :32])), pin(rep(kxy[kidx, 32:]))
    ok3 = pin(np.zeros(n3, np.uint8))

    def c3():
        eng._check(eng._lib.sbv_hash_verify_batch(eng._h, ctypes.c_uint8(0), ctypes.c_size_t(n3), vp(M.data_ptr()), vp(OFF.data_ptr()), vp(R.data_ptr()),
                                                  vp(S.data_ptr()), vp(QX.data_ptr()), vp(QY.data_ptr()), None, vp(ok3.data_ptr())), "sbv_hash_verify_batch")
    t = best_of(c3)
    eng.profile_enable(True)
    c3()
    p_ms, v_ms, pairs = eng.profile_read()
    eng.profile_enable(False)
    blocks = 5 * n3          # 256 B + 9 -> 5 blocks of 64 B
    ex["c3_sha256_verify_1m"] = {"workload": "C3: SHA-256 digest + ECDSA-P256 verify fused, 1,048,576 requests of 256 B, 4,096 client keys, 1/16 with a flipped payload bit",
                                 "requests": n3, "e2e_s": t, "value": n3 / t, "unit": "requests/s",
                                 "through": "sbv_hash_verify_batch, pinned host buffers (H2D of 268 MB of requests + 128 B/item inside; keys first, "
                                            "then 4 chunks of 262,144 requests uploaded on a second stream while the previous chunk is hashed and verified)",
                                 "chunks": 4, "verify_kernel_ms_last_chunk": v_ms / max(pairs, 1), "bit_exact_vs_oracle": bool(np.array_equal(ok3.numpy(), np.tile(want1, T16))),
                                 "roofline_frac_canonical": n3 / t * MAC32_PER_VERIFY / mad_peak if mad_peak else None,
                                 "sha256_algorithmic_bytes": blocks * 64 + 32 * n3,
                                 "h2d_gbs": (n3 * (256 + 8 + 128)) / t / 1e9}

    # ---- f2: one large message (a multi-MiB Proposal.Digest, types.go:50-69) is ONE sequential SHA-256 chain: a single GPU
    # thread against a single host core — measured so that the decision (the host keeps single large digests, the engine
    # takes batches) rests on numbers
    big = np.frombuffer(np.random.Generator(np.random.PCG64(77)).bytes(10 << 20), np.uint8)
    boff = np.array([0, big.size], np.uint64)
    t0 = time.perf_counter(); dg = eng.sha256_batch(big, boff); t_gpu = time.perf_counter() - t0
    t0 = time.perf_counter(); want_dg = oracle.sha256_batch(big, boff, nthreads=1); t_cpu = time.perf_counter() - t0
    many_off = (np.arange(1025, dtype=np.uint64) * 10240)      # the same bytes as 1,024 requests of 10 KiB: a batch
    t0 = time.perf_counter(); dg_many = eng.sha256_batch(big[:1024 * 10240], many_off); t_many = time.perf_counter() - t0
    ex["f2_large_single_digest"] = {"bytes": int(big.size), "gpu_one_thread_s": t_gpu, "host_one_core_s": t_cpu,
                                    "same_bytes_as_1024_messages_gpu_s": t_many, "bit_exact_vs_oracle": bool(np.array_equal(dg, want_dg)) and
                                    bool(np.array_equal(dg_many, oracle.sha256_batch(big[:1024 * 10240], many_off))),
                                    "decision": "a lone multi-MiB digest is a single dependent chain: it stays with the caller (the reference computes "
                                                "Proposal.Digest itself, view.go:435); the engine hashes batches"}

    # ---- C5: mixed-curve consenter batch, 65,536 signatures, curve tag = DRBG bit (~50/50), 512 keys per curve ----
    tile5 = 8192
    b256 = corpus.make_batch(oracle.P256, n=tile5, K=512, seed=81, corrupt_rate=16)
    b384 = corpus.make_batch(oracle.P384, n=tile5, K=512, seed=82, corrupt_rate=16)
    w256 = oracle.verify_batch(oracle.P256, b256["r"], b256["s"], b256["qx"], b256["qy"], b256["digest"])
    w384 = oracle.verify_batch(oracle.P384, b384["r"], b384["s"], b384["qx"], b384["qy"], b384["digest"])
    g5 = ref.DRBG(9)
    tag = (np.frombuffer(b"".join(g5.block(i) for i in range(BATCH // 32)), np.uint8)[:BATCH] & 1).astype(np.uint8)
    f48 = {k: np.zeros((BATCH, 48), np.uint8) for k in ("r", "s", "qx", "qy")}
    dg = np.zeros((BATCH, 32), np.uint8)
    want5 = np.zeros(BATCH, np.uint8)
    i0, i1 = np.nonzero(tag == 0)[0], np.nonzero(tag == 1)[0]
    j0, j1 = np.arange(i0.size) % tile5, np.arange(i1.size) % tile5
    for k in f48:
        f48[k][i0, 16:] = b256[k][j0]
        f48[k][i1] = b384[k][j1]
    dg[i0], dg[i1] = b256["digest"][j0], b384["digest"][j1]
    want5[i0], want5[i1] = w256[j0], w384[j1]
    P = {k: pin(v) for k, v in f48.items()}
    TAG, DG, ok5 = pin(tag), pin(dg), pin(np.zeros(BATCH, np.uint8))

    def c5():
        eng._check(eng._lib.sbv_verify_mixed(eng._h, ctypes.c_size_t(BATCH), vp(TAG.data_ptr()), vp(P["r"].data_ptr()), vp(P["s"].data_ptr()),
                                             vp(P["qx"].data_ptr()), vp(P["qy"].data_ptr()), vp(DG.data_ptr()), vp(ok5.data_ptr())), "sbv_verify_mixed")
    t = best_of(c5)
    n256, n384 = int(i0.size), int(i1.size)
    ex["c5_mixed_curve_64k"] = {"workload": "C5: mixed-curve consenter batch, 65,536 signatures (P-256 / P-384 by DRBG bit), 512 keys per curve, 1/16 corrupted",
                                "n": BATCH, "p256": n256, "p384": n384, "e2e_s": t, "value": BATCH / t, "unit": "verifies/s",
                                "through": "sbv_verify_mixed, pinned host buffers", "bit_exact_vs_oracle": bool(np.array_equal(ok5.numpy(), want5)),
                                "roofline_frac_canonical": (n256 * MAC32_PER_VERIFY + n384 * MAC32_PER_VERIFY_P384) / t / mad_peak if mad_peak else None}
    return ex


if __name__ == "__main__":
    main()
