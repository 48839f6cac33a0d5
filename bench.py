#!/usr/bin/env python
"""bench.py -- headline benchmark of the per-read FASTQ batch path on B200.

Workload (BASELINE.json configs[4], the config the metric is quoted on): fused
trim-by-quality (Q20) + demultiplex of paired-end 2x150 bp reads against a 384-sample dual-index
sheet (10+10 bp, literal '+', 8 bp UMI -> 29-character barcodes), synthetic FASTQ generated on the
device.  The 1 B-pair job does not fit any memory, so it is streamed: a "step" is one batch of
`--pairs` read pairs per GPU (weak scaling: every rank processes its own contiguous pair range).

  value     reads/s over all ranks with inputs resident in HBM (CUDA events on the kernels' stream): one step = the two
            fused trim+demultiplex passes AND the device-side per-sample compaction of both mates (one contiguous
            output run per sample) -- the whole hot path of the north star.  `value_demux_passes_only` is round 1's
            definition (the two passes without the compaction, which round 1 did on the host); `value_breakdown`
            gives the parts in ms per step
  e2e       the same metric through the C ABI with HOST buffers: pinned H2D upload, kernels, compaction, D2H
            of the per-sample streams (compacted buffers + slice tables), 3 slots in flight, the host thread
            and its pinned buffers on the GPU's NUMA node
  configs   device time, algorithmic bytes and roofline fraction of BASELINE configs[0..3] as well
  roofline  algorithmic bytes (input once + output once) / average device time of the dominant
            kernel, against MEASURED_PEAKS.json
  cpu_baseline  the CPU oracle (port of the reference; the Rust reference cannot be built here)

`--impl reference` times that oracle on all host cores instead (rank 0 only).

`--dump-outputs DIR` writes what the caller of the timed step received after its last step (rank 0) as
DIR/<name>.npy; the inputs are the same seeded batch in every run, so two builds compare output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import random
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree (it may be read-only)

READ_LEN = 150
MIN_BASEQ = 20
N_SAMPLES = 384


def make_sheet(n_samples=N_SAMPLES, seed=2024):
    """i7(10)+i5(10)+UMI(8): 20 literal bases with pairwise Hamming distance >= 3."""
    rng = random.Random(seed)
    codes = []
    while len(codes) < n_samples:
        c = bytes(rng.choice(b"ACGT") for _ in range(20))
        if all(sum(a != b for a, b in zip(c, d)) >= 3 for d in codes):
            codes.append(c)
    return [c[:10] + b"+" + c[10:] + b"U" * 8 for c in codes]


def sheet_text(bcs):
    return b"".join(b"S%03d\t%s\n" % (i, b) for i, b in enumerate(bcs))


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons of one GPU while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows = index, False, []

    def run(self):
        try:
            p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                  "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
        except Exception:
            return
        self.proc = p
        for line in p.stdout:
            self.rows.append([x.strip() for x in line.split(",")])
            if self.stop_flag:
                break
        p.terminate()

    def finish(self):
        self.stop_flag = True
        time.sleep(0.15)
        if hasattr(self, "proc"):
            self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
            except Exception:
                continue
            for k, nm in enumerate(names):
                if len(r) > 2 + k and r[2 + k].lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------- reference arm
def _oracle_shard(args):
    sheet, r1, r2 = args
    from oracle import pyoracle as O
    t1, t2 = O.trim_by_quality(r1, MIN_BASEQ), O.trim_by_quality(r2, MIN_BASEQ)
    res = O.demultiplex(sheet, t1[1], t2[1])
    return res["identified"]


def cut_pairs(buf: bytes, n_pairs: int, parts: int):
    """Splits a FASTQ buffer of n_pairs records into `parts` pieces at record boundaries."""
    lines = buf.split(b"\n")
    per = (n_pairs + parts - 1) // parts
    out = []
    for k in range(parts):
        seg = lines[4 * k * per:4 * min((k + 1) * per, n_pairs)]
        if seg:
            out.append(b"\n".join(seg) + b"\n")
    return out


def time_oracle(sheet, r1, r2, n_pairs, procs, steps, warmup):
    """Oracle = fasta demultiplex sheet <(fasta trim by quality R1 20) <(fasta trim by quality R2 20),
    in memory, `procs` independent shards in parallel (the reference itself is single-threaded)."""
    import multiprocessing as mp
    from oracle import pyoracle as O
    O.build()
    s1, s2 = cut_pairs(r1, n_pairs, procs), cut_pairs(r2, n_pairs, procs)
    jobs = [(sheet, a, b) for a, b in zip(s1, s2)]
    times = []
    if procs == 1:
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            _oracle_shard(jobs[0])
            if it >= warmup:
                times.append(time.perf_counter() - t0)
    else:
        with mp.get_context("fork").Pool(procs) as pool:
            for it in range(warmup + steps):
                t0 = time.perf_counter()
                pool.map(_oracle_shard, jobs)
                if it >= warmup:
                    times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    return 2.0 * n_pairs / dt, dt


def synth_pair(eng, n_pairs, first_pair, seed=5):
    n1 = eng.synth(0, n_pairs, seed=seed, first_pair=first_pair, read_len=READ_LEN, mate=1, with_bc=True)
    n2 = eng.synth(1, n_pairs, seed=seed, first_pair=first_pair, read_len=READ_LEN, mate=2, with_bc=True)
    return n1, n2


def host_pairs(bcs, n_pairs, first_pair=0, seed=5, threads=None):
    """Both mates of `n_pairs` read pairs from the HOST twin of the device generator (oracle/synth_host.c):
    the same bytes as Engine.synth for the same (seed, range), without loading the product's library."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import pyoracle as O
    O.build()
    threads = threads or max(1, min(os.cpu_count() or 1, 32))
    per = (n_pairs + threads - 1) // threads
    jobs = [(m, first_pair + k * per, max(0, min(per, n_pairs - k * per))) for m in (1, 2) for k in range(threads)]
    with ThreadPoolExecutor(threads) as ex:  # (ctypes releases the GIL)
        parts = list(ex.map(lambda j: O.synth_fastq(j[2], seed=seed, first_pair=j[1], read_len=READ_LEN, mate=j[0],
                                                    barcodes=bcs), jobs))
    return b"".join(parts[:threads]), b"".join(parts[threads:])


def run_reference(args, rank):
    if rank != 0:
        return
    bcs = make_sheet()
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, 64))
    n_pairs = args.ref_pairs_per_core * procs
    r1, r2 = host_pairs(bcs, n_pairs)  # input creation only: no GPU, no libseqkit_b200.so in this arm
    rps, dt = time_oracle(sheet_text(bcs), r1, r2, n_pairs, procs, args.steps, max(args.warmup, 1))
    line = {
        "impl": "reference", "metric": "reads_per_s", "value": rps, "unit": "reads/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "gbases_per_s": rps * READ_LEN / 1e9,
        "config": workload_config(args.pairs),
        "cpu_baseline": {"value": rps, "unit": "reads/s", "cores": procs, "kind": "port",
                         "sample": "%d pairs per step (bounded sample of the workload), %d independent shards "
                                   "(oracle/fasta_oracle.c, in memory, no gzip); input from oracle/synth_host.c"
                                   % (n_pairs, procs)},
        "e2e": {"value": rps, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit_line(line)


def workload_config(pairs, note=None):
    cfg = {"workload": "BASELINE configs[4]: fused trim-by-quality(Q%d)+demultiplex, paired-end 2x%d bp, %d samples, "
                       "dual index 10+10 bp + 8 bp UMI (29-char barcodes incl. '+'), <=1 mismatch; 1B-pair job streamed "
                       "in batches" % (MIN_BASEQ, READ_LEN, N_SAMPLES),
           "pairs_per_gpu_per_step": pairs, "read_len": READ_LEN, "samples": N_SAMPLES, "min_baseq": MIN_BASEQ,
           "l2": "inputs per step (>1 GB per stream) exceed the 126 MB L2; no flush needed"}
    if note:
        cfg["note"] = note
    return cfg


# ---------------------------------------------------------------------------------------------- our arm
_REAL_STDOUT = None


def emit_line(line):
    """The one JSON line of the contract, on the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    # Libraries print banners on stdout (NCCL: its version line); the contract is ONE line there.  File
    # descriptor 1 is pointed at stderr for the whole run and the JSON line goes to the saved descriptor.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pairs", type=int, default=8_000_000, help="read pairs per GPU per step (device-resident)")
    ap.add_argument("--e2e-pairs", type=int, default=1_000_000, help="read pairs per host batch in the e2e leg")
    ap.add_argument("--cpu-pairs", type=int, default=400_000, help="bounded sample for the 1-core CPU baseline")
    ap.add_argument("--ref-pairs-per-core", type=int, default=100_000)
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--cli-pairs", type=int, default=200_000,
                    help="bounded sample for the files+gzip end-to-end leg (the `fasta` binary; 0 = skip)")
    ap.add_argument("--cli-pairs-large", type=int, default=2_000_000,
                    help="pairs of the files+gzip leg's second, larger run of the `fasta` binary (0 = skip)")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-configs", action="store_true", help="no device-time legs for BASELINE configs[0..3]")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32 / float64, ~34 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    from seqkit_b200 import Engine, _lib as L

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: seqkit_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    bcs = make_sheet()
    P = args.pairs
    steps, warm = args.steps, max(args.warmup, 3)
    cfg_reads = 0 if args.skip_configs else 10_000_000  # configs[1] wants 10 M single-end reads resident
    eng = Engine(device=local_rank, max_stream_bytes=max(P * 410, cfg_reads * 345) + (1 << 20),
                 max_records=max(P, cfg_reads), n_slots=1, max_samples=N_SAMPLES, aux_streams=False)
    lib = eng.lib
    eng.set_sheet(bcs)
    n1, n2 = synth_pair(eng, P, rank * P)  # weak scaling: rank r owns pairs [r*P, (r+1)*P)
    opts = L.DemuxOpts(MIN_BASEQ, 0, 0, 0, 0)
    stream = torch.cuda.ExternalStream(lib.sk_slot_stream(eng.ctx, 0), device=local_rank)

    def step(compact=True):
        rc = lib.sk_demultiplex(eng.ctx, 0, C.byref(opts))
        if rc == 0 and compact:
            rc = lib.sk_demux_compact(eng.ctx, 0)
        if rc != 0:
            raise RuntimeError("sk_demultiplex / sk_demux_compact failed: %s" % lib.sk_last_error(eng.ctx).decode())

    # the one collective of the path: per-sample counts merged over NVLink with a single NCCL all-reduce
    comm = C.c_void_p()
    if world > 1:
        idbuf = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            raw = C.create_string_buffer(128)
            assert lib.sk_nccl_unique_id(eng.ctx, raw) == 0, lib.sk_last_error(eng.ctx)
            idbuf = torch.frombuffer(bytearray(raw.raw), dtype=torch.uint8).clone()
        idbuf = idbuf.cuda()
        dist.broadcast(idbuf, 0)
        raw = bytes(idbuf.cpu().numpy().tobytes())
        assert lib.sk_nccl_comm_init(eng.ctx, raw, world, rank, C.byref(comm)) == 0, lib.sk_last_error(eng.ctx)

    for _ in range(warm):
        step()
    if world > 1:  # the first all-reduce sets up NCCL's channels: part of the warm-up, like the first launches
        assert lib.sk_allreduce_counts(eng.ctx, 0, comm) == 0, lib.sk_last_error(eng.ctx)
    res = eng.wait()
    assert res.status == 0 and res.n_records == P, (res.status, res.n_records)
    # sk_result.reserved: bit0 = the warp engine ran, bit1 = it was re-run on the general engine, bit3 = compacted
    assert (res.reserved & 3) == 1, "bench workload must run on the warp engine without a re-run (got %d)" % res.reserved
    assert res.reserved & 8, "the per-sample compaction must have run"
    pairs_done = res.n_records

    def timed(n_steps, compact):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record(stream)
        for _ in range(n_steps):
            step(compact)
        if world > 1:
            assert lib.sk_allreduce_counts(eng.ctx, 0, comm) == 0, lib.sk_last_error(eng.ctx)
        ev1.record(stream)
        barrier()
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    ms_total = timed(steps, True)  # the whole step: both demultiplex passes + the per-sample compaction of both mates
    res = eng.wait()
    assert res.status == 0 and res.reserved & 8, (res.status, res.reserved)
    launches = res.gpu_launches * steps
    counts = (C.c_uint64 * (N_SAMPLES + 2))()
    lib.sk_download_counts(eng.ctx, 0, counts)
    if world > 1:
        assert counts[N_SAMPLES] == P * world, "all-reduced total_reads must cover every rank"
    clocks = sampler.finish()
    if args.dump_outputs and rank == 0:  # before the passes below reuse the slot's buffers
        dump_outputs(args.dump_outputs, eng, L, res, counts)
    ms_step = ms_total / steps
    value = 2.0 * P * world / (ms_step * 1e-3)
    ms_with_compaction = ms_step
    ms_demux_only = timed(steps, False) / steps  # round 1's definition: the two passes alone
    res_d = eng.wait()
    assert res_d.status == 0

    # per-kernel device time (CUDA events around each launch, on the launching stream)
    lib.sk_set_profiling(eng.ctx, 1)
    pass_ms = [0.0, 0.0]
    prof_steps = min(steps, 20)
    for _ in range(prof_steps):
        step(False)
        r = eng.wait()
        pass_ms[0] += r.pass_ms[0] / prof_steps
        pass_ms[1] += r.pass_ms[1] / prof_steps
    lib.sk_set_profiling(eng.ctx, 0)
    bytes_pass = [n1 + res.out_bytes[0], n2 + res.out_bytes[1]]
    dom = 0 if pass_ms[0] >= pass_ms[1] else 1
    peak, peak_src = peaks()
    achieved = bytes_pass[dom] / (pass_ms[dom] * 1e-3) / 1e9
    if os.environ.get("SK_NO_WARP", "0") not in ("", "0"):  # the general engine instead of the warp engine
        kname = lambda k: "sk_chunk_kernel<OP_DEMUX%d>" % (k + 1)
    else:
        kname = lambda k: "sk_warp_kernel<OP_DEMUX%d>" % (k + 1)
    # DRAM traffic of the dominant kernel from this round's committed ncu capture (dram__bytes_read + write,
    # 1 M pairs per launch), scaled to this launch's pairs; null when the summary is missing
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            tj = json.load(f)
        traffic = tj["dram_bytes_per_launch"]["DEMUX%d" % (dom + 1)] * (P / float(tj["pairs_per_launch"]))
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "kernel": kname(dom), "peak_source": peak_src,
                "algorithmic_bytes_per_launch": bytes_pass[dom], "ms_per_launch": pass_ms[dom],
                "other_kernel": {"kernel": kname(1 - dom), "ms_per_launch": pass_ms[1 - dom],
                                 "achieved": bytes_pass[1 - dom] / (pass_ms[1 - dom] * 1e-3) / 1e9},
                "step_bytes": sum(bytes_pass), "step_achieved": sum(bytes_pass) / (ms_demux_only * 1e-3) / 1e9,
                # SURVEY 8(d): against the nominal figure of the north star as well (~8 TB/s)
                "frac_of_nominal_8000_gbs": achieved / 8000.0}
    identified = counts[N_SAMPLES + 1]
    out_bytes = [int(res.out_bytes[0]), int(res.out_bytes[1])]
    compact_ms = ms_with_compaction - ms_demux_only
    breakdown = {"demux1_ms": pass_ms[0], "demux2_ms": pass_ms[1], "compact_ms": compact_ms,
                 "step_ms": ms_step, "step_ms_demux_passes_only": ms_demux_only,
                 "compact": {"kernels": "sk_compact_hist/cols/bases/addr/move_kernel, both mates",
                             "algorithmic_bytes": 2 * sum(out_bytes),  # the emitted bytes once more in and out
                             "achieved": 2 * sum(out_bytes) / (max(compact_ms, 1e-6) * 1e-3) / 1e9,
                             "frac": 2 * sum(out_bytes) / (max(compact_ms, 1e-6) * 1e-3) / 1e9 / peak}}
    value_demux_only = 2.0 * P * world / (ms_demux_only * 1e-3)
    configs = None
    # the path's other two operators on the same resident mate-1 stream (BASELINE configs[0] / [1] shapes):
    # device time per launch and algorithmic bytes (input once + output once), for the record
    if rank == 0:
        lib.sk_set_profiling(eng.ctx, 1)
        other = {}
        for name, fn in (("trim_by_quality", lib.sk_trim_by_quality), ("mask_by_quality", lib.sk_mask_by_quality)):
            ms, ob = 0.0, 0
            reps = 5
            for i in range(reps + 1):
                assert fn(eng.ctx, 0, MIN_BASEQ, 0) == 0, lib.sk_last_error(eng.ctx)
                r = eng.wait()
                assert r.status == 0 and r.n_records == P, (name, r.status, r.n_records)
                if i:
                    ms += r.pass_ms[0] / reps
                    ob = int(r.out_bytes[0])
                    eng_bits = int(r.reserved)  # 1: warp engine, 2: re-run on the general engine
            opn = "TRIM" if name.startswith("trim") else "MASK"
            ws = os.environ.get("SK_WARP_STREAM")  # default: both on the warp engine (trim: + scan + gather kernels)
            on_warp = os.environ.get("SK_NO_WARP", "0") in ("", "0") and ws not in ("", "0")
            kn = ("sk_warp_kernel<OP_%s>" if on_warp else "sk_chunk_kernel<OP_%s>") % opn
            if on_warp and opn == "TRIM" and os.environ.get("SK_TRIM_GATHER") not in ("", "0"):
                kn += " + sk_tile_sum_kernel + sk_tile_scan_kernel + sk_tile_gather_kernel"
            other[name] = {"kernel": kn, "engine_bits": eng_bits,
                           "reads_per_launch": P, "ms_per_launch": ms, "algorithmic_bytes_per_launch": n1 + ob,
                           "achieved": (n1 + ob) / (ms * 1e-3) / 1e9, "frac": (n1 + ob) / (ms * 1e-3) / 1e9 / peak}
        roofline["other_ops"] = other
        if not args.skip_configs:
            try:
                configs = run_configs(eng, L, P, peak)
                configs["configs[3] add barcode"] = run_add_barcode_leg(local_rank, peak)
            except Exception as ex:  # reported extras: never cost the contract line
                configs = {"error": "%s: %s" % (type(ex).__name__, ex)}
        lib.sk_set_profiling(eng.ctx, 0)
    eng.close()

    # ---- bytes, not only counts: per-sample streams are a function of the pair range, whichever GPU / batching
    verify = None
    try:
        verify = verify_ranges(torch, L, bcs, local_rank, rank, world)
    except AssertionError:
        raise
    except Exception as ex:
        verify = {"error": "%s: %s" % (type(ex).__name__, ex)}

    # ---- e2e: host buffers through the C ABI, 3 slots in flight
    e2e = None
    if not args.skip_e2e:
        e2e = run_e2e(args, torch, L, bcs, local_rank, rank, world, barrier)

    # ---- CPU baseline (rank 0, N=1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        r1, r2 = host_pairs(bcs, args.cpu_pairs)
        rps, dt = time_oracle(sheet_text(bcs), r1, r2, args.cpu_pairs, 1, 1, 0)
        cpu = {"value": rps, "unit": "reads/s", "cores": 1, "kind": "port",
               "sample": "%d pairs (same generator), oracle/fasta_oracle.c trim x2 + demultiplex in memory, %.1f s"
                         % (args.cpu_pairs, dt)}

    # ---- files + gzip end to end (rank 0, N=1 only): the `fasta` binary beside the oracle's CLI
    e2e_files = None
    if rank == 0 and world == 1 and args.cli_pairs > 0:
        try:
            e2e_files = run_cli_leg(args, bcs, local_rank, with_cpu=not args.skip_cpu)
        except Exception as ex:  # a reported extra: never costs the contract line
            e2e_files = {"error": "%s: %s" % (type(ex).__name__, ex)}

    if rank == 0:
        line = {
            "metric": "reads_per_s", "value": value, "unit": "reads/s", "n_gpus": world, "steps": steps, "warmup": warm,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "config": workload_config(P), "gbases_per_s": value * READ_LEN / 1e9,
            "pairs_per_s": value / 2, "identified_fraction": identified / float(P * world),
            "bytes_per_step_per_gpu": {"in": [n1, n2], "out": out_bytes},
            "value_includes": "the two fused trim+demultiplex passes and the device-side per-sample compaction of both mates "
                              "(round 1 compacted on the host and quoted the two passes alone: value_demux_passes_only)",
            "value_demux_passes_only": value_demux_only, "value_breakdown": breakdown,
            "clocks": clocks, "gpu_launches": launches, "roofline": roofline, "e2e": e2e, "cpu_baseline": cpu,
            "e2e_files_gzip": e2e_files, "configs": configs, "verify": verify,
        }
        emit_line(line)
    if world > 1:
        dist.destroy_process_group()


def _nth_newline(buf, k):
    """Offset just past the k-th newline of buf (len(buf) if it has fewer)."""
    pos = 0
    for _ in range(k):
        j = buf.find(b"\n", pos)
        if j < 0:
            return len(buf)
        pos = j + 1
    return pos


def run_cli_leg(args, bcs, local_rank, with_cpu=True):
    """Third number of SURVEY 8(d): end to end WITH files and gzip.  The drop-in `fasta` binary
    (`demultiplex --trim-by-quality=Q`, its one-pass form of the benchmark's pipeline) reads two plain FASTQ
    files and writes one .fq.gz per sample and mate (block-parallel deflate on host threads; common.rs:49-81
    spawns one `gzip -c` child per file); beside it the oracle's CLI runs the reference's own three commands
    (trim R1, trim R2, demultiplex) on the same files, and every decompressed output file is compared.  Wall
    clock of the processes, CUDA context creation included; a bounded sample.  `large` repeats our side on ten
    times the pairs (start-up amortised; the single-threaded oracle would need minutes there)."""
    import shutil
    import tempfile
    from seqkit_b200 import Engine
    from oracle import pyoracle as O
    n = args.cli_pairs
    fasta = os.path.join(ROOT, "seqkit_b200", "fasta")
    if not os.path.exists(fasta):
        subprocess.check_call(["make", "-s", "-C", ROOT, "seqkit_b200/fasta"])
    O.build()
    oracle_cli = os.path.join(ROOT, "oracle", "_build", "fasta_oracle")
    r1, r2 = host_pairs(bcs, n, seed=11)
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    top = tempfile.mkdtemp(prefix="skbench_", dir=base)
    try:
        for name, data in (("sheet.tsv", sheet_text(bcs)), ("r1.fq", r1), ("r2.fq", r2)):
            with open(os.path.join(top, name), "wb") as f:
                f.write(data)
        env = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", str(local_rank)))

        def outputs(d):
            tot = 0
            for f in os.listdir(d):
                if f.endswith(".fq.gz"):
                    tot += os.path.getsize(os.path.join(d, f))
            return tot

        def settle(d):  # the reference does not wait for its gzip children (common.rs:49-81): wait for the files
            last, t_end = -1, time.time() + 60
            while time.time() < t_end:
                cur = outputs(d)
                if cur == last:
                    return cur
                last = cur
                time.sleep(0.2)
            return last

        # one untimed invocation on the first 2 000 pairs: the first CUDA process of a fresh box pays one-off costs
        # (driver and library page-in) that belong to the box, not to the run; its wall time is reported beside
        d_warm = os.path.join(top, "warm")
        os.mkdir(d_warm)
        cut1, cut2 = _nth_newline(r1, 8000), _nth_newline(r2, 8000)
        for name, data in (("w1.fq", r1[:cut1]), ("w2.fq", r2[:cut2])):
            with open(os.path.join(top, name), "wb") as f:
                f.write(data)
        t0 = time.perf_counter()
        subprocess.run([fasta, "demultiplex", "--trim-by-quality=%d" % MIN_BASEQ, "../sheet.tsv", "../w1.fq", "../w2.fq"],
                       cwd=d_warm, env=env, capture_output=True, timeout=600)
        dt_warm = time.perf_counter() - t0
        shutil.rmtree(d_warm, ignore_errors=True)
        d_ours = os.path.join(top, "ours")
        os.mkdir(d_ours)
        t0 = time.perf_counter()
        p = subprocess.run([fasta, "demultiplex", "--trim-by-quality=%d" % MIN_BASEQ, "../sheet.tsv", "../r1.fq", "../r2.fq"],
                           cwd=d_ours, env=env, capture_output=True, timeout=600)
        dt_ours = time.perf_counter() - t0
        if p.returncode != 0:
            raise RuntimeError("fasta demultiplex: exit %d: %s" % (p.returncode, p.stderr[-300:].decode("utf-8", "replace")))
        gz_ours = settle(d_ours)
        res = {"value": 2.0 * n / dt_ours, "unit": "reads/s", "seconds": dt_ours, "pairs": n,
               "warmup_invocation_seconds": dt_warm,
               "gz_bytes_out": gz_ours, "summary": p.stderr.decode("utf-8", "replace").strip().splitlines()[-1][:200],
               "note": "fasta demultiplex --trim-by-quality=%d sheet r1.fq r2.fq: process start, CUDA context, file "
                       "reads, kernels, compaction, %d .fq.gz files through block-parallel deflate (zlib level 4); wall clock"
                       % (MIN_BASEQ, 2 * N_SAMPLES)}
        if with_cpu:
            d_cpu = os.path.join(top, "cpu")
            os.mkdir(d_cpu)
            t0 = time.perf_counter()
            for m in ("1", "2"):
                with open(os.path.join(d_cpu, "t%s.fq" % m), "wb") as f:
                    subprocess.run([oracle_cli, "trim", "by", "quality", "../r%s.fq" % m, str(MIN_BASEQ)], cwd=d_cpu,
                                   stdout=f, check=True, timeout=900)
            q = subprocess.run([oracle_cli, "demultiplex", "../sheet.tsv", "t1.fq", "t2.fq"], cwd=d_cpu,
                               capture_output=True, timeout=900)
            dt_cpu = time.perf_counter() - t0
            gz_cpu = settle(d_cpu)
            same = None
            if q.returncode == 0:  # decompressed bytes of every output file, ours against the oracle's
                import gzip as _gz
                same = True
                for f in sorted(os.listdir(d_cpu)):
                    if f.endswith(".fq.gz"):
                        a = _gz.decompress(open(os.path.join(d_cpu, f), "rb").read())
                        try:
                            b = _gz.decompress(open(os.path.join(d_ours, f), "rb").read())
                        except Exception:
                            b = None
                        if a != b:
                            same = False
                            break
            res["cpu"] = {"value": 2.0 * n / dt_cpu, "unit": "reads/s", "seconds": dt_cpu, "cores": 1, "kind": "port",
                          "exit": q.returncode, "gz_bytes_out": gz_cpu, "outputs_identical": same,
                          "note": "oracle CLI, single-threaded: trim by quality R1, R2 to files, then demultiplex; it compresses its "
                                  "output files one after another (the reference runs its gzip -c children concurrently)"}
        if args.cli_pairs_large > n:  # throughput with the start-up amortised (ours only)
            nl = args.cli_pairs_large
            l1, l2 = host_pairs(bcs, nl, seed=12)
            for name, data in (("l1.fq", l1), ("l2.fq", l2)):
                with open(os.path.join(top, name), "wb") as f:
                    f.write(data)
            del l1, l2
            d_big = os.path.join(top, "big")
            os.mkdir(d_big)
            t0 = time.perf_counter()
            p = subprocess.run([fasta, "demultiplex", "--trim-by-quality=%d" % MIN_BASEQ, "../sheet.tsv", "../l1.fq", "../l2.fq"],
                               cwd=d_big, env=dict(env, SK_TIMING="1"), capture_output=True, timeout=600)
            dt_big = time.perf_counter() - t0
            tl = [x for x in p.stderr.decode("utf-8", "replace").splitlines() if "timing" in x]
            res["large"] = {"value": 2.0 * nl / dt_big, "unit": "reads/s", "seconds": dt_big, "pairs": nl, "exit": p.returncode,
                            "gz_bytes_out": settle(d_big), "phases": tl[-1] if tl else None, "host_cores": os.cpu_count()}
        return res
    finally:
        shutil.rmtree(top, ignore_errors=True)


def make_sheet_single(n_samples=96, length=8, seed=3):
    """configs[2]: 96 single-index 8-mers with pairwise Hamming distance >= 3 (greedy from the seed)."""
    rng = random.Random(seed)
    codes = []
    while len(codes) < n_samples:
        c = bytes(rng.choice(b"ACGT") for _ in range(length))
        if all(sum(a != b for a, b in zip(c, d)) >= 3 for d in codes):
            codes.append(c)
    return codes


def run_configs(eng, L, P, peak):
    """Device time, algorithmic bytes (input once + output once) and fraction of the measured HBM peak for
    BASELINE configs[0..3], on the main engine (profiling on: CUDA events around every pass)."""
    lib = eng.lib
    out = {}

    def stream_leg(fn, n, seed, reps):
        n_in = eng.synth(0, n, seed=seed, mate=1, with_bc=False)
        ms, ob, launches = 0.0, 0, 0
        for i in range(reps + 2):
            assert fn(eng.ctx, 0, MIN_BASEQ, 0) == 0, lib.sk_last_error(eng.ctx)
            r = eng.wait()
            assert r.status == 0 and r.n_records == n, (r.status, r.n_records)
            if i >= 2:
                ms += r.pass_ms[0] / reps
                ob, launches = int(r.out_bytes[0]), int(r.gpu_launches)
        b = n_in + ob
        return {"reads": n, "ms": ms, "launches": launches, "algorithmic_bytes": b, "achieved": b / (ms * 1e-3) / 1e9,
                "frac": b / (ms * 1e-3) / 1e9 / peak, "reads_per_s": n / (ms * 1e-3)}

    out["configs[0]"] = dict(stream_leg(lib.sk_trim_by_quality, 1_000_000, 1, 20),
                             workload="fasta trim by quality, 1 M single-end 150 bp reads, Q20 (launch-latency regime: "
                                      "trim kernel + tile sum + scan + gather)")
    out["configs[1]"] = dict(stream_leg(lib.sk_mask_by_quality, 10_000_000, 2, 5),
                             workload="fasta mask by quality, 10 M single-end 150 bp reads, 3'-decaying qualities, Q20")

    def demux_leg(bcs, fused, reps=5):
        eng.set_sheet(bcs)
        m1 = eng.synth(0, P, seed=7, mate=1, with_bc=True)
        m2 = eng.synth(1, P, seed=7, mate=2, with_bc=True)
        opts = L.DemuxOpts(fused, 0, 0, 0, 0)
        ms = [0.0, 0.0]
        for i in range(reps + 1):
            assert lib.sk_demultiplex(eng.ctx, 0, C.byref(opts)) == 0, lib.sk_last_error(eng.ctx)
            r = eng.wait()
            assert r.status == 0 and r.n_records == P and (r.reserved & 3) == 1, (r.status, r.n_records, r.reserved)
            if i:
                ms[0] += r.pass_ms[0] / reps
                ms[1] += r.pass_ms[1] / reps
        b = [m1 + int(r.out_bytes[0]), m2 + int(r.out_bytes[1])]
        return {"pairs": P, "ms": ms, "algorithmic_bytes": b, "achieved": [b[k] / (ms[k] * 1e-3) / 1e9 for k in range(2)],
                "frac": [b[k] / (ms[k] * 1e-3) / 1e9 / peak for k in range(2)], "reads_per_s": 2.0 * P / (sum(ms) * 1e-3),
                "identified_fraction": r.identified_reads / float(P)}

    out["configs[2]"] = dict(demux_leg(make_sheet_single(), -1),
                             workload="fasta demultiplex, paired-end 2x150 bp, 96-sample 8 bp single index, <=1 mismatch "
                                      "(50 M-pair job streamed in batches of `pairs`)")
    out["configs[3]"] = dict(demux_leg(make_sheet(), -1),
                             workload="fasta demultiplex (no trim), 384 samples, dual index 10+10 bp + 8 bp UMI; the "
                                      "`fasta add barcode` step of the chain is timed separately below")
    eng.set_sheet(make_sheet())
    return out


def run_add_barcode_leg(local_rank, peak, n=1_000_000):
    """configs[3], first step of the chain (README.md:44-47): `fasta add barcode reads.fq barcodes.fq` on 1 M reads
    (record table of the barcode file from its line table, then OP_ADDBC over the reads on the warp engine)."""
    from seqkit_b200 import Engine
    bcs = make_sheet()
    with Engine(device=local_rank, max_stream_bytes=n * 420 + (1 << 20), max_records=n, max_samples=N_SAMPLES,
                aux_streams=True) as eng:
        lib = eng.lib
        eng.set_sheet(bcs)
        m1 = eng.synth(0, n, seed=13, mate=1, with_bc=True)
        r1 = eng.download_in(0, m1)
        lines = r1.split(b"\n")
        obs = [ln[ln.rfind(b" BC:") + 4:] for ln in lines[0::4] if ln]
        bcfile = b"".join(b"@bc%07d\n%s\n+\n%s\n" % (i, b, b"I" * len(b)) for i, b in enumerate(obs))
        m1 = eng.synth(0, n, seed=13, mate=1, with_bc=False)
        eng.upload(2, bcfile)
        lib.sk_set_profiling(eng.ctx, 1)
        ms, reps, ob, ms_table = 0.0, 5, 0, 0.0
        for i in range(reps + 1):
            assert lib.sk_add_barcode(eng.ctx, 0, 0) == 0, lib.sk_last_error(eng.ctx)
            r = eng.wait()
            assert r.status == 0 and r.n_records == n, (r.status, r.n_records)
            if i:
                ms += (r.pass_ms[0] + r.pass_ms[2]) / reps
                ms_table += r.pass_ms[2] / reps
                ob = int(r.out_bytes[0])
        b = m1 + len(bcfile) + ob
        return {"reads": n, "ms": ms, "ms_barcode_table": ms_table, "engine_bits": int(r.reserved), "launches": int(r.gpu_launches), "algorithmic_bytes": b, "achieved": b / (ms * 1e-3) / 1e9,
                "frac": b / (ms * 1e-3) / 1e9 / peak, "reads_per_s": n / (ms * 1e-3),
                "workload": "fasta add barcode, 1 M reads + 1 M barcode records (i7+i5UMI on the sequence line)"}


def dump_outputs(out_dir, eng, L, res, counts, n_sample=1 << 22, seed=2024):
    """What the caller of the timed step receives, as DIR/<name>.npy:

      counts                  float64 [S + 2]  reads per sample, then total and identified reads
      mate{1,2}_sample_len    float64 [S]      bytes of each sample's output stream (the content of its .fq.gz file)
      mate{1,2}_sample_crc32  float64 [S]      CRC-32 of each sample's stream, so every byte is compared
      mate{1,2}_bytes         float32 [n]      a seeded sample of the bytes of the streams laid end to end in sheet
                                               order (sorted positions drawn from the streams' total length)

    The streams are read through the slice table: the padding between slices of the compacted buffer is not
    output and is never read."""
    import zlib
    import numpy as np
    lib, S = eng.lib, N_SAMPLES
    arrays = {"counts": np.array(counts[:S + 2], dtype=np.float64)}
    for m in range(2):
        ext = int(res.out_extent[m])
        buf = np.empty(max(ext, 1), dtype=np.uint8)
        sl = (L.Slice * (S + 1))()
        assert lib.sk_download_compact(eng.ctx, 0, m, buf.ctypes.data, ext) == 0, lib.sk_last_error(eng.ctx)
        assert lib.sk_download_slices(eng.ctx, 0, m, sl) == 0, lib.sk_last_error(eng.ctx)
        eng.wait()
        off = np.array([sl[s].offset for s in range(S)], dtype=np.int64)
        ln = np.array([sl[s].len for s in range(S)], dtype=np.int64)
        assert np.all(off + ln <= ext) and int(ln.sum()) == int(res.out_bytes[m]), "slice table and outcome disagree"
        mv = memoryview(buf)
        arrays["mate%d_sample_len" % (m + 1)] = ln.astype(np.float64)
        arrays["mate%d_sample_crc32" % (m + 1)] = np.array([zlib.crc32(mv[o:o + n]) for o, n in zip(off, ln)],
                                                           dtype=np.float64)
        total = int(ln.sum())
        pos = np.sort(np.random.default_rng(seed + m).integers(0, max(total, 1), size=min(n_sample, total)))
        start = np.cumsum(ln) - ln
        s = np.searchsorted(start, pos, side="right") - 1  # the sample whose stream holds each position
        arrays["mate%d_bytes" % (m + 1)] = buf[off[s] + pos - start[s]].astype(np.float32)
        del buf, mv
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    print("bench: wrote %d arrays (%.1f MB) to %s" % (len(arrays), sum(a.nbytes for a in arrays.values()) / 1e6, out_dir),
          file=sys.stderr)


def verify_ranges(torch, L, bcs, local_rank, rank, world, n=1_000_000):
    """Bytes, not only counts.  A CRC-32 of every per-sample output stream (compacted buffers + slices, both
    mates) of a pair range, chained over batches in batch order, so equal CRCs mean equal concatenated bytes.
    One GPU: the range in one batch against the same range in two half batches (the order contract of
    fasta_demultiplex.rs:196-238 across batches).  Several GPUs: every rank also recomputes the first `n` pairs
    of its right neighbour's range and the two ranks' CRCs are compared (outputs depend on the pair range,
    not on the GPU that ran it)."""
    import zlib
    from seqkit_b200 import Engine
    S = N_SAMPLES
    with Engine(device=local_rank, max_stream_bytes=n * 410 + (1 << 20), max_records=n, max_samples=S,
                aux_streams=False) as eng:
        lib = eng.lib
        eng.set_sheet(bcs)
        opts = L.DemuxOpts(MIN_BASEQ, 0, 0, 0, 0)

        def crcs(batches):
            acc = [[0] * S, [0] * S]
            for first, cnt in batches:
                synth_pair(eng, cnt, first)
                assert lib.sk_demultiplex(eng.ctx, 0, C.byref(opts)) == 0, lib.sk_last_error(eng.ctx)
                assert lib.sk_demux_compact(eng.ctx, 0) == 0, lib.sk_last_error(eng.ctx)
                r = eng.wait()
                assert r.status == 0 and r.n_records == cnt
                for m in range(2):
                    ext = int(r.out_extent[m])
                    buf = torch.empty(max(ext, 1), dtype=torch.uint8)
                    sl = (L.Slice * (S + 1))()
                    assert lib.sk_download_compact(eng.ctx, 0, m, buf.data_ptr(), ext) == 0
                    assert lib.sk_download_slices(eng.ctx, 0, m, sl) == 0
                    eng.wait()
                    mv = memoryview(buf.numpy())
                    for s in range(S):
                        acc[m][s] = zlib.crc32(mv[sl[s].offset:sl[s].offset + sl[s].len], acc[m][s])
            return acc

        P0 = rank * 8_000_000  # (any range will do; ranks use distinct ones)
        if world == 1:
            whole = crcs([(P0, n)])
            halves = crcs([(P0, n // 2), (P0 + n // 2, n - n // 2)])
            assert whole == halves, "per-sample streams of two half batches differ from the single batch"
            return {"ok": True, "pairs": n, "check": "CRC-32 of all %d per-sample streams: one batch == two half batches" % (2 * S)}
        import torch.distributed as dist
        mine = crcs([(P0, n)])
        right = ((rank + 1) % world) * 8_000_000
        theirs = crcs([(right, n)])
        t_mine = torch.tensor(mine, dtype=torch.int64, device="cuda")
        gathered = [torch.empty_like(t_mine) for _ in range(world)]
        dist.all_gather(gathered, t_mine)
        ok = gathered[(rank + 1) % world].cpu().tolist() == theirs
        flag = torch.tensor([1 if ok else 0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        assert int(flag.item()) == 1, "a rank's per-sample streams differ from its neighbour's recomputation"
        return {"ok": True, "pairs": n, "check": "CRC-32 of all %d per-sample streams of every rank's range == the same "
                                                 "range recomputed on the neighbouring GPU" % (2 * S)}


def run_e2e(args, torch, L, bcs, local_rank, rank, world, barrier):
    """Same metric through the reference-facing call with HOST buffers: every step uploads its inputs from
    pinned memory, runs the kernels and the per-sample compaction, and reads back the per-sample streams
    (compacted buffers + slice tables).  The host thread and its pinned buffers sit on the GPU's NUMA node."""
    from seqkit_b200 import Engine
    Pe, nslots = args.e2e_pairs, 3
    eng = Engine(device=local_rank, max_stream_bytes=Pe * 410 + (1 << 20), max_records=Pe, n_slots=nslots,
                 max_samples=N_SAMPLES, aux_streams=False)
    lib = eng.lib
    numa = lib.sk_bind_thread_to_device(local_rank) if os.environ.get("SK_NO_NUMA", "0") in ("", "0") else -2
    eng.set_sheet(bcs)
    n1, n2 = synth_pair(eng, Pe, rank * Pe, seed=9)

    def pinned(nbytes):  # NUMA-local, portable pinned memory from the library (a torch view over it)
        ptr = lib.sk_pinned_alloc(eng.ctx, nbytes)
        assert ptr, lib.sk_last_error(eng.ctx)
        return ptr

    h_in = [pinned(n) for n in (n1, n2)]
    for w, (ptr, n) in enumerate(zip(h_in, (n1, n2))):
        assert lib.sk_download_in(eng.ctx, 0, w, ptr, n) == 0
    cap = max(n1, n2) + Pe * 16 + (1 << 20)
    h_out = [[pinned(cap) for _ in range(2)] for _ in range(nslots)]
    h_slices = [[C.cast(pinned((N_SAMPLES + 1) * 16), C.POINTER(L.Slice)) for _ in range(2)] for _ in range(nslots)]
    opts = L.DemuxOpts(MIN_BASEQ, 0, 0, 0, 0)
    d2h = [0]
    ident = [0]

    def submit(s):
        assert lib.sk_upload(eng.ctx, s, 0, h_in[0], n1) == 0
        assert lib.sk_upload(eng.ctx, s, 1, h_in[1], n2) == 0
        assert lib.sk_demultiplex(eng.ctx, s, C.byref(opts)) == 0
        assert lib.sk_demux_compact(eng.ctx, s) == 0

    def collect(s):
        res = L.Result()
        assert lib.sk_wait(eng.ctx, s, C.byref(res)) == 0 and res.status == 0
        nb = 0
        for m in range(2):
            assert res.out_extent[m] <= cap
            assert lib.sk_download_compact(eng.ctx, s, m, h_out[s][m], res.out_extent[m]) == 0
            assert lib.sk_download_slices(eng.ctx, s, m, h_slices[s][m]) == 0
            nb += res.out_extent[m] + (N_SAMPLES + 1) * 16
        assert lib.sk_counts_accumulate(eng.ctx, s) == 0
        assert lib.sk_wait(eng.ctx, s, None) == 0  # the per-sample streams of this batch are in host memory now
        assert h_slices[s][0][N_SAMPLES].len == res.out_bytes[0]
        ident[0] = res.identified_reads
        d2h[0] = nb
        return res

    def run(k):
        inflight = []
        for i in range(k):
            s = i % nslots
            if len(inflight) == nslots:
                collect(inflight.pop(0))
            submit(s)
            inflight.append(s)
        for s in inflight:
            collect(s)

    run(3)
    steps = max(min(args.steps, 40), 6)
    barrier()
    t0 = time.perf_counter()
    run(steps)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([dt], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    eng.close()
    # the box's measured copy ceiling for this many GPUs (tools/pcie_ceiling.py, committed from the pool's 8-GPU box)
    ceiling = None
    try:
        with open(os.path.join(ROOT, "profiles", "r2_pcie_ceiling.json")) as f:
            c = json.load(f)["ceiling_gbs"].get("N=%d" % world)
        if c:
            h2d_all = (n1 + n2) * steps / dt / 1e9 * world
            d2h_all = d2h[0] * steps / dt / 1e9 * world
            ceiling = dict(c, h2d_gbs_all_gpus=h2d_all, d2h_gbs_all_gpus=d2h_all,
                           frac_of_both_at_once=max(h2d_all, d2h_all) / c["both_at_once_per_direction"],
                           source="profiles/r2_pcie_ceiling.json (plain cudaMemcpyAsync, pinned, both directions at once)")
    except Exception:
        pass
    return {"value": 2.0 * Pe * world * steps / dt, "unit": "reads/s", "h2d_bytes_per_step": int(n1 + n2), "copy_ceiling": ceiling,
            "d2h_bytes_per_step": int(d2h[0]), "pairs_per_step": Pe, "steps": steps, "slots": nslots,
            "pcie_gbs": {"h2d": (n1 + n2) * steps / dt / 1e9, "d2h": d2h[0] * steps / dt / 1e9},
            "numa_node": numa,
            "note": "pinned host buffers -> sk_upload -> sk_demultiplex -> sk_demux_compact -> sk_download_compact + "
                    "sk_download_slices (per-sample streams in host memory) + device-side run totals; gzip excluded"}


if __name__ == "__main__":
    main()
