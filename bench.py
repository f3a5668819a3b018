#!/usr/bin/env python
"""bench.py — genomic bases/sec through make_images + inference (BASELINE.json metric) on N B200s.

  python bench.py --gpus 1 --steps K --warmup W            our CUDA path (libpepper_b200 through the C-ABI)
  python bench.py --impl reference ...                     the reference's CPU algorithm on the host cores
  torchrun --nproc-per-node N ... bench.py --gpus N ...    one rank per GPU; region groups handed out over the ranks, the
                                                           network's head kernel writes 84-byte prediction records into one
                                                           gather buffer, ONE all-gather of records per step
  --config variant_ont (default, BASELINE configs[1]) | variant_hifi (configs[3] preset) | polish (configs[2])
  --scaling weak (default: per-GPU work fixed) | strong (one job of --regions regions split over the ranks, configs[4] shape)
  --schedule dynamic (default for N > 1: ranks claim groups from an atomic counter) | static (contiguous blocks)

A "step" is one pass of the hot path (pileup-summary encoder -> recurrent network) over one batch of synthetic regions, tiled
like the reference tiles a contig (pepper_variant ImageGenerationUI.py:307-316: 100 kb intervals + 100 bp halos;
pepper ImageGenerationUI.py:269-272: 1 kb regions + 100 bp overlap).

Printed JSON (one line, rank 0): `value` = whole-job genomic bases/s with the reads already resident in HBM; `e2e` = the same
metric through the public host-buffer API (pinned host reads -> H2D -> kernels -> gather -> D2H of the prediction records on
the writer rank); `roofline` for the dominant kernel (by time: the fused tcgen05 GEMMs, tensor bound) and `roofline_encoder`
for the HBM-bound pileup kernel; `rank_phase_ms` = per-rank encoder / network / wait / gather device times (min, median, max
over ranks); `verified` = sampled regions of the timed workload re-computed by the oracle AFTER the timed loops;
`cpu_baseline` = the oracle timed on one host core over that sample.  Only the verification / cpu_baseline /
--impl reference legs touch oracle/.
"""
from __future__ import annotations

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

FLOP_PER_CAND = 161.4e6          # SURVEY §8d: 92.1 M dense + 69.2 M recurrent per candidate, all batched GEMM here
FLOP_PER_IMAGE = 1.53e9          # polish: 19 windows x 100 steps (SURVEY §8d)
METRIC = "genomic bases/sec (make_images+inference)"

CONFIGS = {
    "variant_ont": dict(kind="variant", platform="ONT", coverage=30.0, regions=645, region_size=100000,
                        workload="pepper_variant make_images + run_inference, synthetic ONT R9.4.1 30x (BASELINE configs[1])"),
    "variant_hifi": dict(kind="variant", platform="HIFI", coverage=35.0, regions=645, region_size=100000,
                         workload="pepper_variant call_variant --hifi preset, synthetic PacBio-HiFi 35x (BASELINE configs[3])"),
    "polish": dict(kind="polish", platform="ONT", coverage=40.0, regions=5000, region_size=1000,
                   workload="pepper polish make_images + call_consensus, synthetic 5 Mb draft + 40x ONT (BASELINE configs[2])"),
}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_tflops_sustained=d.get("bf16_tflops_sustained"),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def host_cores() -> int:
    """Cores this process may really use: scheduler affinity, capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = max(1, min(n, int(float(q) / float(p))))
    except Exception:
        pass
    return n


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, gpu: int):
        self.gpu = gpu
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, pw, reasons = [], [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w": float(np.median(pw)) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


def encoder_algorithmic_bytes(reads, regions, n_out: int, out_bytes: int) -> int:
    """SURVEY.md §8(d): per region sum over reads of (36 + 4 n_cigar + ceil(l_seq/2) + l_seq) + L_ref + outputs
    (variant: N_cand * (33*26 + 4 + 1 + 1 + 62); polish: n_cols * (10 + 8 + 4))."""
    lseq = np.diff(reads.seq_off)
    ncig = np.diff(reads.cigar_off)
    rd = int((36 + 4 * ncig + (lseq + 1) // 2 + lseq).sum())
    ref = int(regions.col("ref_len").sum())
    return rd + ref + n_out * out_bytes


DUMP_BYTES = 60 * 10 ** 6          # the files stay under 64 MB with their headers


def dump_outputs(d: str, arrays: dict, n: int) -> None:
    """--dump-outputs: arrays with one row per output record / image, as d/<name>.npy (float32 where that is exact, else
    float64).  All n rows when they fit in DUMP_BYTES, else a sample drawn with a fixed seed (the same rows for the same n);
    sample_rows.npy holds the row indices and n_rows.npy the row count."""
    exact32 = lambda a: a.dtype == np.float32 or (a.dtype.kind in "iu" and a.dtype.itemsize <= 2)      # noqa: E731
    row_bytes = sum((4 if exact32(a) else 8) * int(np.prod(a.shape[1:])) for a in arrays.values()) + 8
    keep = DUMP_BYTES // row_bytes
    rows = np.arange(n) if n <= keep else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "sample_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(d, "n_rows.npy"), np.array([n], dtype=np.float64))
    for k, a in arrays.items():
        np.save(os.path.join(d, k + ".npy"), a[rows].astype(np.float32 if exact32(a) else np.float64))


def platform_of(cfg):
    from pepper_b200 import synth
    plat = synth.ONT if cfg["platform"] == "ONT" else synth.HIFI
    params = synth.ont_params() if cfg["platform"] == "ONT" else synth.hifi_params()
    return plat, params


def build_workload(args, cfg):
    """`--block` regions generated from scratch, tiled along the contig up to `--regions` (every rank builds the SAME block:
    the dynamic schedule hands any group to any rank)."""
    from pepper_b200 import synth
    t0 = time.time()
    plat, _ = platform_of(cfg)
    n = args.regions
    block = min(args.block, n)
    if cfg["kind"] == "variant":
        reads, regions = synth.make_variant_workload(block, args.region_size, args.coverage, plat, seed=args.seed)
    else:
        block = min(max(args.block, 250), n)
        reads, regions = synth.make_polish_workload(block, args.coverage, plat, seed=args.seed)
    reads, regions = synth.tile_workload(reads, regions, (n + block - 1) // block)
    if regions.n_regions > n:       # trim to the requested number of regions
        nr = int(regions.table[n - 1, 7])
        nb = int(reads.seq_off[nr]); nc = int(reads.cigar_off[nr])
        codes = reads.codes()[:nb]
        reads = synth.ReadBatch(reads.pos[:nr], reads.seq_off[:nr + 1], reads.cigar_off[:nr + 1], reads.flags[:nr], reads.mapq[:nr],
                                synth.pack_codes(codes), reads.qual[:nb], reads.cigar[:nc])
        if regions.ref.shape[0] > 1:
            rl = int(regions.table[n - 1, 4] + regions.table[n - 1, 5])
            regions = synth.RegionTable(regions.table[:n].copy(), regions.ref[:rl])
        else:
            regions = synth.RegionTable(regions.table[:n].copy(), regions.ref)
    return reads, regions, block, time.time() - t0


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def rank_stats(vals: dict, world: int, dev):
    """min / median / max over ranks of each per-rank figure (one small all-gather)."""
    import torch
    import torch.distributed as dist
    keys = sorted(vals)
    t = torch.tensor([float(vals[k]) for k in keys], dtype=torch.float64, device=dev)
    if world > 1:
        allt = torch.empty((world, len(keys)), dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(allt.view(-1), t)
    else:
        allt = t[None, :]
    a = allt.cpu().numpy()
    return {k: {"min": float(a[:, i].min()), "median": float(np.median(a[:, i])), "max": float(a[:, i].max())} for i, k in enumerate(keys)}, \
           {k: [float(x) for x in a[:, i]] for i, k in enumerate(keys)}


# =============================================================================================================== variant
def run_variant(args, cfg):
    import torch
    import torch.distributed as dist
    from pepper_b200 import weights, _lib
    from pepper_b200.abi import HostReads
    from pepper_b200.dist import DistributedVariantCaller, RECORD_BYTES
    from pepper_b200.pipeline import DeviceReads

    rank, world, local = dist_env()
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    _lib.require_gpu()
    dev = torch.device("cuda", local)
    peaks = load_peaks()
    plat, params = platform_of(cfg)

    reads, regions, block, gen_s = build_workload(args, cfg)
    strong = args.scaling == "strong"
    replicas = 1 if strong else world                      # weak: the job is `world` copies of the per-GPU block
    job_bases = regions.genomic_bases() * replicas
    schedule = args.schedule or ("dynamic" if world > 1 else "static")
    # per-rank record capacity: the even share of the job + head room for a rank that claims more groups than its share
    est = max(4096, int(regions.genomic_bases() * replicas / world / (45 if cfg["platform"] == "ONT" else 250)))
    cap = int(est * (1.5 if world > 1 else 1.0))
    dvc = DistributedVariantCaller(weights.random_variant_state(0), local, capacity=cap, schedule=schedule, group_regions=args.group_regions)
    dreads = DeviceReads(reads, regions, device=local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(src):
        return dvc.run(src, regions, params, seq_off=reads.seq_off, replicas=replicas)

    # ---- device-resident leg: W warm-up + K timed steps, CUDA events, max over ranks
    n_mine = 0
    for _ in range(args.warmup):
        n_mine = step(dreads)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    phases, stats = [], []
    ev0.record()
    for _ in range(args.steps):
        n_mine = step(dreads)
        phases.append(dict(dvc.phase_ms)); stats.append(dict(dvc.stats))
    ev1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        tt = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    ms_per_step = ms / args.steps
    value = job_bases / (ms_per_step / 1e3)
    mean = lambda rows, k: float(np.mean([r[k] for r in rows]))      # noqa: E731
    mine = {k: mean(phases, k) for k in ("encoder_ms", "network_ms", "wait_ms", "gather_ms", "groups")}
    mine["candidates"] = float(n_mine)
    mine["count_kernel_ms"] = mean(stats, "enc_count")
    mine["launches"] = mean(stats, "encoder_launches") + mean(stats, "network_launches")
    rstat, rall = rank_stats(mine, world, dev)
    counts = dvc.buffer.counts.cpu().numpy()
    n_job = int(counts.sum())
    if args.dump_outputs and rank == 0:                     # the last timed step's records, as the writer rank receives them
        rec = dvc.buffer.to_host()
        dump_outputs(args.dump_outputs, {"probs": rec["probs"], "position": rec["position"], "region": rec["region"], "depth": rec["depth"],
                                         "freq": rec["freq"], "key": np.ascontiguousarray(rec["key"]).view(np.uint8).reshape(-1, rec.dtype["key"].itemsize)},
                     rec.shape[0])

    # ---- end-to-end leg: pinned host reads -> H2D -> kernels -> gather -> D2H of the job's records on the writer rank
    hr = HostReads(reads, pin=True)
    e2e_steps = max(1, args.e2e_steps)
    barrier()                                               # page-locking 4 GB takes a different time on every rank
    step(hr)                                                # warm-up of the staging buffers
    if rank == 0:
        dvc.buffer.to_host()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    e0.record()
    records = None
    e2e_phases = []
    for _ in range(e2e_steps):
        step(hr)
        e2e_phases.append(dict(dvc.phase_ms))
        if rank == 0:
            records = dvc.buffer.to_host()                  # the writer reads every rank's records, genomic order restored
    e1.record()
    barrier()
    e2e_ms = max(e0.elapsed_time(e1), (time.perf_counter() - w0) * 1e3) / e2e_steps
    if world > 1:
        tt = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_ms = float(tt.item())
    # bytes over PCIe per step, whole job: every group's reads go up once; the writer rank reads all records
    h2d = int((hr.nbytes + regions.table.nbytes + regions.ref.nbytes) * replicas)
    d2h = int(n_job * RECORD_BYTES + dvc.buffer.meta.numel() * 8)
    l2_mb = dreads.nbytes / 1e6

    registered = bool(dvc.buffer.registered)
    meta_bytes = int(dvc.buffer.meta.numel() * 8)
    files_dist = None
    if (world > 1 or args.files_dist) and not args.no_files:   # north_star's input at N GPUs: every rank opens the same BAM + FASTA
        try:
            files_dist = files_leg_dist(args, cfg, local, dvc, world, rank, barrier, replicas)
        except Exception as ex:
            if world > 1:
                raise                                           # (files_leg_dist keeps the ranks in step for failures inside a pass)
            files_dist = {"error": repr(ex)[:300]}
    if records is not None:
        records = records.copy()
    dvc.close()                                             # releases the NCCL-registered buffer before the process group
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- rooflines (rank 0's launches; algorithmic work of the groups rank 0 ran)
    share = mine["candidates"] / max(1, n_job)
    alg_bytes = int(encoder_algorithmic_bytes(reads, regions, 0, 0) * replicas * (mine["groups"] / max(1.0, sum(rall["groups"])))
                    + mine["candidates"] * (33 * 26 + 4 + 1 + 1 + 62))
    count_s = mine["count_kernel_ms"] / 1e3
    net_s = mine["network_ms"] / 1e3
    sustained = peaks["bf16_tflops_sustained"] or peaks["bf16_tflops"]
    roof_enc = dict(bound="hbm", kernel="k_tile_count", achieved=alg_bytes / count_s / 1e9, peak=peaks["hbm_gbs"], unit="GB/s",
                    frac=alg_bytes / count_s / 1e9 / peaks["hbm_gbs"], traffic=int(alg_bytes * TRAFFIC_RATIO_COUNT), peak_source=peaks["source"],
                    traffic_note=TRAFFIC_NOTE_COUNT, algorithmic_bytes=alg_bytes, launches_ms=count_s * 1e3,
                    note="algorithmic bytes of the whole encoder (SURVEY 8d) for the groups this rank ran over the summed duration of "
                         "its pileup-count kernel launches (one per group)")
    tf = mine["candidates"] * FLOP_PER_CAND / net_s / 1e12
    roof_net = dict(bound="tensor", kernel="k_lstm_layer + k_tc_gemm_p (tcgen05 LSTM layers / MLP GEMMs, all launches of the step)",
                    achieved=tf, peak=sustained, unit="TFLOP/s", frac=tf / sustained,
                    traffic=int(mine["candidates"] * TRAFFIC_PER_CAND), traffic_note=TRAFFIC_NOTE_NET,
                    peak_source=peaks["source"] + ", sustained bf16", flops=mine["candidates"] * FLOP_PER_CAND, launches_ms=net_s * 1e3,
                    executed_tflops=PRODUCTS_VARIANT * tf, executed_frac=PRODUCTS_VARIANT * tf / sustained,
                    products_per_flop={k: p for k, (_, p) in VARIANT_GEMMS.items()},
                    note="achieved = fp32-equivalent algorithmic FLOPs (161.4 MFLOP per candidate) / network time of rank 0; a FLOP "
                         "runs as 2 or 3 16-bit tensor-core products (hi/lo operand split, fp32 accumulate; products_per_flop, %.2f on "
                         "average), so the tensor pipe runs at executed_frac; the step runs under the board power cap (clocks.reasons)"
                         % PRODUCTS_VARIANT)

    line = {
        "metric": METRIC, "value": value, "unit": "bases/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
        "dtype": "int32 counts / int8 images (encoder); networks f32-equivalent (%s hi/lo split, 2-3 products per GEMM on tcgen05, fp32 accumulate)" % OPERAND,
        "data": "synthetic",
        "config": {"workload": cfg["workload"], "name": args.config, "regions_per_gpu": regions.n_regions if not strong else None,
                   "job_regions": regions.n_regions * replicas, "region_size": args.region_size, "coverage": args.coverage,
                   "job_genomic_bases": job_bases, "aligned_bases_per_block": reads.n_bases, "reads_per_block": reads.n_reads,
                   "job_candidates": n_job, "schedule": schedule, "group_regions": args.group_regions,
                   "parallelism": f"region groups handed out ({schedule}) over {world} GPU(s); head kernel writes 84 B records into the "
                                  f"gather buffer; 1 all-gather of records (+1 of counts) per step",
                   "l2": "inputs larger than L2 (%.0f MB of reads resident per GPU)" % l2_mb,
                   "weights": "seeded random (no trained checkpoint offline)", "generated_block_regions": block, "gen_seconds": round(gen_s, 1),
                   "nccl_registered_buffer": registered},
        "clocks": clocks,
        "e2e": {"value": job_bases / (e2e_ms / 1e3), "unit": "bases/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms, "steps": e2e_steps,
                "kernel_ms_rank0": {"encoder": mean(e2e_phases, "encoder_ms"), "network": mean(e2e_phases, "network_ms"),
                                    "wait": mean(e2e_phases, "wait_ms"), "gather": mean(e2e_phases, "gather_ms")},
                "api": "pepper_b200.dist.DistributedVariantCaller.run(HostReads) -> pb_variant_stream_* (pinned host buffers) + "
                       "GatherBuffer.to_host() on the writer rank"},
        "gpu_launches": int(sum(rall["launches"]) * args.steps),
        "rank_phase_ms": rstat, "per_rank": rall,
        "phase_ms": {"encoder": mine["encoder_ms"], "network": mine["network_ms"], "encoder_count_kernel": mine["count_kernel_ms"],
                     "encoder_phases": {k: mean(stats, k) for k in ("enc_prefix", "enc_count", "enc_sites", "enc_alleles", "enc_windows")}},
        "roofline": roof_net, "roofline_encoder": roof_enc,
    }
    if not args.no_verify:
        line["verified"], base = verify_variant(args, cfg, reads, regions, records, replicas)
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = base
    if files_dist is not None:
        line["e2e_files"] = files_dist
    elif world == 1 and not args.no_files:
        try:
            line["e2e_files"] = files_leg(args, cfg, local)
        except Exception as ex:                                 # the headline numbers above stand on their own
            line["e2e_files"] = {"error": repr(ex)[:300]}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def files_leg(args, cfg, local):
    """north_star's input: a synthetic coordinate-sorted .bam + .bai + .fa of the SAME scale on disk -> predictions through
    VariantFromFiles.call_stream.  Inside the timed region: pread of the compressed BGZF blocks, H2D of those blocks, GPU
    inflate + record walk + parse, get_reads (trim), encoder, network, D2H of the prediction columns.  Not in it: writing the
    files (a fork pool of zlib compressors) and page-cache warm-up (one pass over the file)."""
    import shutil
    import tempfile
    import torch
    from pepper_b200 import synth, synth_files, weights
    from pepper_b200.frontend import VariantFromFiles, variant_intervals
    plat, params = platform_of(cfg)
    n_regions = args.files_regions or args.regions
    span = args.block * args.region_size
    times = -(-(n_regions * args.region_size + 200) // span)
    t0 = time.time()
    rec, genome = synth.simulate_contig_records(span, args.coverage, plat, args.seed + 7)
    d = tempfile.mkdtemp(prefix="pb_bench_files_")
    try:
        bam, fa = os.path.join(d, "s.bam"), os.path.join(d, "s.fa")
        L = synth_files.write_bam_tiled(bam, "chr20s", rec, span, times)
        synth_files.write_fasta(fa, [("chr20s", np.tile(genome[:span], times))])
        gen_s = time.time() - t0
        iv = variant_intervals(100, min(L - 100, 100 + n_regions * args.region_size), args.region_size)
        genomic = sum(e - s for s, e in iv)
        vf = VariantFromFiles(bam, fa, weights.random_variant_state(0), device=local, gpu_inflate=not args.host_inflate,
                              host_share=args.inflate_host_share)
        cap = int(genomic // (40 if cfg["platform"] == "ONT" else 250)) + 65536
        vf.call_stream("chr20s", iv[:2 * args.files_batch], params, batch=args.files_batch, capacity=cap)   # warm-up (allocations, page cache of the head)
        with open(bam, "rb") as f:                               # page cache: the file was just written, read it once anyway
            while f.read(1 << 26):
                pass
        torch.cuda.synchronize()
        steps = max(1, args.files_steps)
        t0 = time.perf_counter()
        n_cand = 0
        for _ in range(steps):
            calls = vf.call_stream("chr20s", iv, params, batch=args.files_batch, capacity=cap)
            n_cand = len(calls)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / steps
        comp, infl = vf.bam.io_stats()
        ft = vf.bam.fetch_device_timings() if not args.host_inflate else {}
        split = list(vf.inflate_split())
        stage_prof = getattr(vf, "last_profile", None)
        vf.close()
        return {"value": genomic / dt, "unit": "bases/s", "ms_per_step": dt * 1e3, "steps": steps, "regions": len(iv), "genomic_bases": genomic,
                "candidates": n_cand, "bam_bytes": os.path.getsize(bam), "records_per_block": rec.n_records, "batch_regions": args.files_batch,
                "inflate": "host zlib thread pool" if args.host_inflate else "GPU (k_bgzf_inflate, warp per BGZF block)" + (" + host pool on %.2f of the blocks" % args.inflate_host_share if args.inflate_host_share else ""),
                "inflate_blocks_host_device": split, "last_batch_fetch_ms": ft, "host_stage_ms": stage_prof, "h2d_bytes_per_step": int(os.path.getsize(bam)), "d2h_bytes_per_step": int(n_cand * 90),
                "gen_seconds": round(gen_s, 1),
                "api": "pepper_b200.frontend.VariantFromFiles.call_stream -> pb_bam_fetch_device + pb_get_reads_* + pb_variant_stream_*"}
    finally:
        shutil.rmtree(d, ignore_errors=True)


def files_leg_dist(args, cfg, local, dvc, world, rank, barrier, replicas):
    """files_leg over all ranks: rank 0 writes ONE .bam + .bai + .fa (the per-GPU block), every rank opens it
    (frontend.VariantFileSource) and claims interval groups through the same DistributedVariantCaller as the headline legs; the
    weak-scaling job is `replicas` passes over the file's intervals.  Timed (host clock around device-synchronised steps, max
    over ranks): pread + H2D of the compressed blocks of the groups each rank claimed, GPU inflate / parse / trim, encoder,
    network, the all-gather, D2H of the whole job's records on the writer rank."""
    import shutil
    import tempfile
    import torch
    import torch.distributed as dist
    from pepper_b200 import synth, synth_files
    from pepper_b200.dist import RECORD_BYTES
    from pepper_b200.frontend import VariantFileSource, variant_intervals
    plat, params = platform_of(cfg)
    n_regions = args.files_regions or args.regions
    span = args.block * args.region_size
    times = -(-(n_regions * args.region_size + 200) // span)
    box = [None, 0.0]
    if rank == 0:
        d = None
        try:
            t0 = time.time()
            rec, genome = synth.simulate_contig_records(span, args.coverage, plat, args.seed + 7)
            d = tempfile.mkdtemp(prefix="pb_bench_files_")
            synth_files.write_bam_tiled(os.path.join(d, "s.bam"), "chr20s", rec, span, times)
            synth_files.write_fasta(os.path.join(d, "s.fa"), [("chr20s", np.tile(genome[:span], times))])
            with open(os.path.join(d, "s.bam"), "rb") as f:          # page cache
                while f.read(1 << 26):
                    pass
            box = [d, time.time() - t0]
        except Exception as ex:                                      # e.g. no room in the temp dir: every rank skips the leg together
            if d is not None:
                shutil.rmtree(d, ignore_errors=True)
            box = [None, repr(ex)[:300]]
    if world > 1:
        dist.broadcast_object_list(box, src=0)
    if box[0] is None:
        return {"error": "could not write the synthetic files: %s" % box[1]}
    d, gen_s = box
    try:
        bam, fa = os.path.join(d, "s.bam"), os.path.join(d, "s.fa")
        L = times * span
        iv = variant_intervals(100, min(L - 100, 100 + n_regions * args.region_size), args.region_size)
        genomic = sum(e - s for s, e in iv) * replicas
        src = VariantFileSource(bam, fa, "chr20s", iv, int(params["min_snp_baseq"]), device=local, gpu_inflate=not args.host_inflate,
                                host_share=args.inflate_host_share)
        dev = torch.device("cuda", local)

        def step():
            """One pass; a rank whose pass fails still joins the step's two collectives (with an empty slice), so that the
            ranks stay in step and the leg is reported as failed instead of hanging the headline line."""
            err = 0
            try:
                dvc.run(src, None, params, replicas=replicas)
            except Exception as ex:
                err = 1
                print("files leg, rank %d: %r" % (rank, ex), file=sys.stderr, flush=True)
                if world > 1 and "groups were run" not in str(ex):       # (that one is raised after the collectives, on every rank)
                    dvc.buffer.gather(0, [])
            if world > 1:
                tt = torch.tensor([err], dtype=torch.int32, device=dev)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                err = int(tt.item())
            return err
        if step():                                               # warm-up: reader buffers, staging, the file's pages
            return {"error": "a rank failed in the warm-up pass (stderr has the exception)"}
        if rank == 0:
            dvc.buffer.to_host()
        torch.cuda.synchronize()
        steps = max(1, args.files_steps)
        barrier()
        t0 = time.perf_counter()
        n_cand = 0
        for _ in range(steps):
            if step():
                return {"error": "a rank failed in a timed pass (stderr has the exception)"}
            if rank == 0:
                n_cand = len(dvc.buffer.to_host())
        torch.cuda.synchronize()
        barrier()
        dt = (time.perf_counter() - t0) / steps
        if world > 1:
            tt = torch.tensor([dt], dtype=torch.float64, device=torch.device("cuda", local))
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
        phase = dict(dvc.phase_ms)
        ft = src.bam.fetch_device_timings() if not args.host_inflate else {}
        split = list(src.inflate_split())
        size = os.path.getsize(bam)
        src.close()
        barrier()
        return {"value": genomic / dt, "unit": "bases/s", "ms_per_step": dt * 1e3, "steps": steps, "regions": len(iv) * replicas,
                "genomic_bases": genomic, "candidates": n_cand, "bam_bytes": size, "batch_regions": args.group_regions,
                "inflate": "host zlib thread pool" if args.host_inflate else "GPU (k_bgzf_inflate, warp per BGZF block)" + (" + host pool on %.2f of the blocks" % args.inflate_host_share if args.inflate_host_share else ""),
                "inflate_blocks_host_device_rank0": split, "last_group_fetch_ms": ft, "rank0_phase_ms": phase, "h2d_bytes_per_step": int(size * replicas),
                "d2h_bytes_per_step": int(n_cand * RECORD_BYTES), "gen_seconds": round(gen_s, 1),
                "api": "pepper_b200.dist.DistributedVariantCaller.run(frontend.VariantFileSource) -> pb_bam_fetch_device + pb_get_reads_* + "
                       "pb_variant_stream_* per claimed group; GatherBuffer.to_host() on the writer rank"}
    finally:
        if rank == 0:
            shutil.rmtree(d, ignore_errors=True)


# figures carried over from the ncu --set full captures under profiles/ (per candidate / per algorithmic byte)
PRODUCTS = 3                      # polish network: three 16-bit products per fp32-equivalent FLOP everywhere
OPERAND = "fp16"
# variant network, FLOP per candidate by GEMM (2 directions x 33 steps; hidden 256, gates 1,024; head 16,896 -> 512 -> 4 x 512 -> 3)
# and the 16-bit tensor-core products each one executes per FLOP (handles.cuh lo_mask 0x1a): int8 images are exact in one operand,
# the recurrent GEMMs pass the parity gate with two products, the decoder's x-part and the head need three
VARIANT_GEMMS = {"encoder_x": (3.51e6, 2), "encoder_h": (34.6e6, 2), "decoder_x": (69.2e6, 3), "decoder_h": (34.6e6, 2), "head": (19.4e6, 3)}
PRODUCTS_VARIANT = sum(f * p for f, p in VARIANT_GEMMS.values()) / sum(f for f, _ in VARIANT_GEMMS.values())     # 2.55
TRAFFIC_RATIO_COUNT = 1.60
TRAFFIC_NOTE_COUNT = ("dram__bytes_read+write of k_tile_count = 1.60 x algorithmic bytes in the ncu --set full capture of one "
                      "32-region group (277.0 MB read + 102.7 MB written vs 237.6 MB, profiles/r2c_prof_k_tile_count_summary.txt: "
                      "the excess is the 8 B/op prefix arrays read beside the 4 B CIGAR words); scaled to this step")
TRAFFIC_PER_CAND = 237.36e6 / 3840 + 767.39e6 / 3840 + 678.66e6 / 9472
TRAFFIC_NOTE_NET = ("dram__bytes_read+write of the ncu --set full captures, per candidate: encoder LSTM layer (k_lstm_layer) 237.4 MB and "
                    "decoder LSTM layer 767.4 MB per launch over 3,840 candidates, linear_1 678.7 MB per launch over 9,472 "
                    "(profiles/r1_prof_lstm_*_raw.csv, r1_prof_tcp_lin1_final_raw.csv), scaled to the candidates of this step; captured "
                    "with three products in every GEMM — the shipped mask no longer reads the h_lo operand tiles of the recurrent "
                    "GEMMs, so this is an upper bound")


def verify_variant(args, cfg, reads, regions, records, replicas):
    """AFTER the timed loops: sampled regions of the timed workload are re-computed by the oracle (reference C++ encoder from
    oracle/_ref when present + PyTorch CPU network, one thread) and compared with the records the e2e leg returned.  The same
    run is the 1-core cpu_baseline.  This is the only place the product bench consults oracle/."""
    import torch
    from pepper_b200 import synth
    from oracle import oracle, nets
    torch.set_num_threads(1)
    _, params = platform_of(cfg)
    impl = "ref" if oracle.have_ref() else "port"
    from pepper_b200 import weights
    state = {k: torch.from_numpy(np.asarray(v)) for k, v in weights.random_variant_state(0).items()}     # the weights the product ran with
    n_reg = regions.n_regions
    job_regions = n_reg * replicas
    sample = sorted({0, (job_regions // 2), job_regions - 1})[:args.verify_regions]
    t_enc = t_net = 0.0
    n_chk, max_dp, ok, detail = 0, 0.0, True, []
    for j in sample:
        sub, tab = synth.region_batch(reads, regions, j % n_reg)
        t0 = time.perf_counter()
        w = oracle.variant_encode(sub, tab, params, impl)
        imgs = oracle.images_to_int8(w["images"])
        t_enc += time.perf_counter() - t0
        t0 = time.perf_counter()
        probs = nets.variant_predict(state, imgs, batch=512, threads=1)
        t_net += time.perf_counter() - t0
        got = records[records["region"] == j]
        same = (got.shape[0] == len(w["keys"]) and [k.decode() for k in got["key"]] == w["keys"]
                and np.array_equal(got["position"], w["positions"].astype(np.int32))
                and np.array_equal(got["depth"].astype(np.int32), w["depths"]) and np.array_equal(got["freq"].astype(np.int32), w["freqs"]))
        dp = float(np.abs(got["probs"] - probs).max()) if same and got.shape[0] else (0.0 if same else float("inf"))
        srt = np.sort(probs, axis=1)
        clear = (srt[:, -1] - srt[:, -2]) > 1e-4 if probs.shape[0] else np.zeros(0, bool)
        am = bool(same and np.array_equal(got["probs"].argmax(1)[clear], probs.argmax(1)[clear]))
        ok = ok and same and dp < 1e-3 and am
        max_dp = max(max_dp, dp)
        n_chk += int(got.shape[0])
        detail.append({"region": int(j), "candidates": int(got.shape[0]), "records_bit_exact": bool(same), "max_abs_dprob": dp, "argmax_exact": am})
    ver = {"ok": bool(ok), "regions": [int(j) for j in sample], "candidates": n_chk, "max_abs_dprob": max_dp,
           "oracle": ("reference C++ (oracle/_ref)" if impl == "ref" else "oracle/port_encoders.c") + " + oracle/nets.py",
           "criteria": "candidate records bit-exact; probabilities within 1e-3; class index exact outside a 1e-4 margin", "detail": detail}
    bases = len(sample) * int(regions.table[0, 3] - regions.table[0, 2])
    base = {"value": bases / (t_enc + t_net), "unit": "bases/s", "cores": 1, "kind": "reference" if impl == "ref" else "port",
            "sample": "%d region(s) x %d kb of the timed workload (%d candidates) on one host thread: encoder %.2fs, network (PyTorch CPU, "
                      "bit-identical to the reference nn.Module) %.2fs" % (len(sample), args.region_size // 1000, n_chk, t_enc, t_net),
            "encoder_s": t_enc, "network_s": t_net}
    return ver, base


# ================================================================================================================ polish
def run_polish(args, cfg):
    import torch
    import torch.distributed as dist
    from pepper_b200 import weights, _lib
    from pepper_b200.abi import HostReads
    from pepper_b200.pipeline import PolishCaller, DeviceReads

    rank, world, local = dist_env()
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    _lib.require_gpu()
    dev = torch.device("cuda", local)
    peaks = load_peaks()
    reads, regions, block, gen_s = build_workload(args, cfg)
    genomic = int((regions.col("cand_end") - regions.col("cand_start")).sum())
    pc = PolishCaller(weights.random_polish_state(0), local)
    d = DeviceReads(reads, regions, device=local)
    cap = 3 * regions.n_regions + 16
    out = dict(bases=torch.empty((cap, 1000), dtype=torch.uint8, device=dev), phred=torch.empty((cap, 1000), dtype=torch.uint8, device=dev),
               position=torch.empty((cap, 1000), dtype=torch.int64, device=dev), index=torch.empty((cap, 1000), dtype=torch.int32, device=dev),
               image_region=torch.empty(cap, dtype=torch.int32, device=dev), chunk_id=torch.empty(cap, dtype=torch.int32, device=dev))
    gathered = torch.empty((world, cap, 2000), dtype=torch.uint8, device=dev) if world > 1 else None

    def gather(n_img):
        """north_star: one all-gather of the per-region predictions (bases + phred, 2,000 B per image, fixed capacity)."""
        if world > 1:
            mine = gathered[rank]
            mine[:n_img, :1000] = out["bases"][:n_img]; mine[:n_img, 1000:] = out["phred"][:n_img]
            dist.all_gather_into_tensor(gathered.view(-1), mine.view(-1))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    n_img = 0
    for _ in range(args.warmup):
        n_img = pc.call_device(d, out); gather(n_img)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    enc, net, cnt = [], [], []
    e0.record()
    for _ in range(args.steps):
        n_img = pc.call_device(d, out); gather(n_img)
        t = pc.timings(); enc.append(t["encode_ms"]); net.append(t["network_ms"]); cnt.append(t["enc_count"])
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:                     # what the last timed step wrote into `out`
        dump_outputs(args.dump_outputs, {k: v[:n_img].cpu().numpy() for k, v in out.items()}, n_img)
    ms = e0.elapsed_time(e1)
    if world > 1:
        tt = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    ms_per_step = ms / args.steps
    launches = pc.net.launches()
    rstat, rall = rank_stats({"encoder_ms": float(np.mean(enc)), "network_ms": float(np.mean(net))}, world, dev)

    hr = HostReads(reads, pin=True)
    calls = pc.call_prepared(hr, regions, reuse_buffers=True)
    barrier()
    e2e_steps = max(1, args.e2e_steps)
    w0 = time.perf_counter()
    for _ in range(e2e_steps):
        calls = pc.call_prepared(hr, regions, reuse_buffers=True)
        gather(calls.bases.shape[0])
    barrier()
    e2e_ms = (time.perf_counter() - w0) * 1e3 / e2e_steps
    if world > 1:
        tt = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_ms = float(tt.item())
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    n_cols = int((calls.position >= 0).sum())
    alg = encoder_algorithmic_bytes(reads, regions, n_cols, 10 + 8 + 4)
    sustained = peaks["bf16_tflops_sustained"] or peaks["bf16_tflops"]
    tf = n_img * FLOP_PER_IMAGE / (float(np.mean(net)) / 1e3) / 1e12
    line = {"metric": "genomic bases/sec (make_images+call_consensus)", "value": world * genomic / (ms_per_step / 1e3), "unit": "bases/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "int32 counts / uint8 images (encoder, fp64 normalisation); network f32-equivalent (%s hi/lo split x%d on tcgen05)" % (OPERAND, PRODUCTS),
            "data": "synthetic",
            "config": {"workload": cfg["workload"], "name": args.config, "regions_per_gpu": regions.n_regions, "genomic_bases_per_gpu": genomic,
                       "aligned_bases_per_gpu": reads.n_bases, "images_per_gpu": n_img, "coverage": args.coverage,
                       "parallelism": f"regions sharded over {world} GPU(s), 1 all-gather of bases+phred",
                       "l2": "inputs larger than L2 (%.0f MB of reads resident per GPU)" % (d.nbytes / 1e6), "gen_seconds": round(gen_s, 1),
                       "generated_block_regions": block, "weights": "seeded random"},
            "clocks": clocks,
            "e2e": {"value": world * genomic / (e2e_ms / 1e3), "unit": "bases/s", "ms_per_step": e2e_ms, "steps": e2e_steps,
                    "h2d_bytes_per_step": int(hr.nbytes + regions.table.nbytes), "d2h_bytes_per_step": int(calls.bases.shape[0] * (2000 + 12000 + 8)),
                    "api": "pepper_b200.pipeline.PolishCaller.call -> pb_polish_call_host (pinned host buffers)"},
            "gpu_launches": int((launches + 6) * args.steps * world), "rank_phase_ms": rstat,
            "phase_ms": {"encoder": float(np.mean(enc)), "network": float(np.mean(net)), "encoder_count_kernel": float(np.mean(cnt))},
            "roofline": dict(bound="tensor", kernel="k_gru_layer (tcgen05 bi-GRU window layers, 38 launches per chunk of 9,472 images)", achieved=tf,
                             peak=sustained, unit="TFLOP/s", frac=tf / sustained, traffic=None, executed_tflops=PRODUCTS * 1.25 * tf,
                             executed_frac=PRODUCTS * 1.25 * tf / sustained, peak_source=peaks["source"] + ", sustained bf16",
                             note="1.53 GFLOP per image (SURVEY 8d) / network time; executed = x%d products x1.25 (zero blocks of the split n gate)" % PRODUCTS),
            "roofline_encoder": dict(bound="hbm", kernel="k_polish_count", achieved=alg / (float(np.mean(cnt)) / 1e3) / 1e9, peak=peaks["hbm_gbs"],
                                     unit="GB/s", frac=alg / (float(np.mean(cnt)) / 1e3) / 1e9 / peaks["hbm_gbs"], traffic=None,
                                     algorithmic_bytes=alg, launch_ms=float(np.mean(cnt)), peak_source=peaks["source"])}
    if not args.no_verify:
        line["verified"], base = verify_polish(args, reads, regions, calls)
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = base
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def verify_polish(args, reads, regions, calls):
    import torch
    from pepper_b200 import synth, weights
    from oracle import oracle, nets, chunk_images as och
    torch.set_num_threads(1)
    impl = "ref" if oracle.have_ref() else "port"
    state = {k: torch.from_numpy(np.asarray(v)) for k, v in weights.random_polish_state(0).items()}
    n_reg = regions.n_regions
    sample = sorted({0, n_reg // 2, n_reg - 1})[:args.verify_regions]
    t_enc = t_net = 0.0
    ok, n_img, detail = True, 0, []
    for r in sample:
        sub, tab = synth.region_batch(reads, regions, r)
        t0 = time.perf_counter()
        w = oracle.polish_encode(sub, tab, impl)
        imgs, pos, idx, cids, regs = och.chunk_images(w["image"], w["pos"], w["idx"], w["col_off"])
        t_enc += time.perf_counter() - t0
        t0 = time.perf_counter()
        wb, wp, wh, wa = nets.polish_predict(state, imgs, threads=1)
        t_net += time.perf_counter() - t0
        sel = np.flatnonzero(calls.image_region == r)
        same = sel.shape[0] == imgs.shape[0] and np.array_equal(calls.position[sel], pos) and np.array_equal(calls.index[sel].astype(np.int64), idx)
        srt = np.sort(wa, axis=2)
        clear = (srt[:, :, -1] - srt[:, :, -2]) > 1e-4
        bases_ok = bool(same and np.array_equal(calls.bases[sel][clear], wb[clear]))
        ok = ok and same and bases_ok
        n_img += int(sel.shape[0])
        detail.append({"region": int(r), "images": int(sel.shape[0]), "columns_bit_exact": bool(same), "bases_exact_outside_margin": bases_ok})
    ver = {"ok": bool(ok), "regions": [int(r) for r in sample], "images": n_img, "detail": detail,
           "oracle": ("reference C++ (oracle/_ref)" if impl == "ref" else "oracle/port_encoders.c") + " + oracle/chunk_images.py + oracle/nets.py"}
    bases = len(sample) * 1000
    base = {"value": bases / (t_enc + t_net), "unit": "bases/s", "cores": 1, "kind": "reference" if impl == "ref" else "port",
            "sample": "%d region(s) x 1 kb of the timed workload (%d images) on one host thread: encoder %.2fs, network %.2fs" % (len(sample), n_img, t_enc, t_net),
            "encoder_s": t_enc, "network_s": t_net}
    return ver, base


# ---------------------------------------------------------------------------------------------------------------
# --impl reference: the reference's CPU algorithm on the host cores, organised the way the reference organises its CPU run —
# P single-threaded worker processes over regions for make_images (pepper_variant ImageGenerationUI.py:326) and over
# candidate / image slices for inference with 1 intra-op thread per caller (predict_distributed_cpu.py:47-57).  One region
# per worker per step at least (VERDICT r1: an under-fed pool made the arm unstable).
# ---------------------------------------------------------------------------------------------------------------
_W = {}


def _worker_init(kind, platform):
    import torch
    torch.set_num_threads(1)
    from oracle import oracle, nets
    from pepper_b200 import synth, weights
    oracle.lib("port")
    _W["impl"] = "ref" if oracle.have_ref() else "port"
    if _W["impl"] == "ref":
        oracle.lib("ref_variant" if kind == "variant" else "ref_polish")
    st = weights.random_variant_state(0) if kind == "variant" else weights.random_polish_state(0)
    _W["state"] = {k: torch.from_numpy(np.asarray(v)) for k, v in st.items()}
    _W["oracle"], _W["nets"], _W["kind"] = oracle, nets, kind
    _W["params"] = synth.ont_params() if platform == "ONT" else synth.hifi_params()


def _worker_encode(task):
    sub, tab = task
    if _W["kind"] == "variant":
        c = _W["oracle"].variant_encode(sub, tab, _W["params"], _W["impl"])
        return _W["oracle"].images_to_int8(c["images"])
    from oracle import chunk_images as och
    w = _W["oracle"].polish_encode(sub, tab, _W["impl"])
    return och.chunk_images(w["image"], w["pos"], w["idx"], w["col_off"])[0]


def _worker_net(images):
    if _W["kind"] == "variant":
        return _W["nets"].variant_predict(_W["state"], images, batch=512, threads=1)
    return _W["nets"].polish_predict(_W["state"], images, threads=1)[0]


def _worker_ready(_):
    return _W["impl"]


class CpuReference:
    def __init__(self, args, cfg, procs: int):
        from pepper_b200 import synth
        self.procs, self.kind = procs, cfg["kind"]
        per_worker = 1 if self.kind == "variant" else 8           # polish regions are 100 x smaller
        self.nreg = max(1, procs * per_worker)
        a = argparse.Namespace(**vars(args))
        a.regions = self.nreg
        reads, regions, _, _ = build_workload(a, cfg)
        self.tasks = [synth.region_batch(reads, regions, r) for r in range(self.nreg)]
        self.genomic_bases = int((regions.col("cand_end") - regions.col("cand_start")).sum())
        import multiprocessing as mp
        self.pool = mp.get_context("spawn").Pool(procs, initializer=_worker_init, initargs=(self.kind, cfg["platform"]))
        self.impl = self.pool.map(_worker_ready, range(procs))[0]

    def step(self):
        t0 = time.perf_counter()
        parts = self.pool.map(_worker_encode, self.tasks, chunksize=1)
        images = np.concatenate(parts)
        t_enc = time.perf_counter() - t0
        t0 = time.perf_counter()
        per = max(1, -(-images.shape[0] // self.procs))
        self.pool.map(_worker_net, [images[i:i + per] for i in range(0, images.shape[0], per)], chunksize=1)
        t_net = time.perf_counter() - t0
        return t_enc, t_net, images.shape[0]

    def close(self):
        self.pool.close()
        self.pool.join()

    def describe(self, t_enc, t_net, n):
        enc = "reference C++ compiled into oracle/_ref" if self.impl == "ref" else "oracle/port_encoders.c"
        return (f"{self.nreg} region(s) of the same workload ({n} {'candidates' if self.kind == 'variant' else 'images'}) per step over "
                f"{self.procs} single-threaded worker process(es): encoder = {enc} {t_enc:.2f}s, network = oracle/nets.py (PyTorch CPU, "
                f"bit-identical to the reference nn.Module) {t_net:.2f}s")


def run_reference(args, cfg):
    """The reference's CPU implementation of the path on all host cores this process may use."""
    rank, world, _ = dist_env()
    if rank != 0:
        return
    procs = host_cores()
    ref = CpuReference(args, cfg, procs)
    tot_t, last = 0.0, None
    for i in range(args.warmup + args.steps):
        t_enc, t_net, n = ref.step()
        if i >= args.warmup:
            tot_t += t_enc + t_net
        last = (t_enc, t_net, n)
    ref.close()
    value = ref.genomic_bases * args.steps / tot_t
    line = {"impl": "reference", "metric": METRIC if cfg["kind"] == "variant" else "genomic bases/sec (make_images+call_consensus)",
            "value": value, "unit": "bases/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * tot_t / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int32/f64 (encoder), f32 (network)", "data": "synthetic",
            "config": {"workload": cfg["workload"], "name": args.config, "region_size": args.region_size, "coverage": args.coverage,
                       "sample_regions_per_step": ref.nreg},
            "cpu_baseline": {"value": value, "unit": "bases/s", "cores": procs, "kind": "reference" if ref.impl == "ref" else "port",
                             "sample": ref.describe(*last)},
            "e2e": {"value": value, "unit": "bases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=os.environ.get("PB_BENCH_CONFIG", "variant_ont"), choices=sorted(CONFIGS))
    ap.add_argument("--regions", type=int, default=None, help="regions per GPU per step (weak) / in the job (strong); chr20 = 645 x 100 kb")
    ap.add_argument("--region-size", type=int, default=None)
    ap.add_argument("--coverage", type=float, default=None)
    ap.add_argument("--block", type=int, default=8, help="regions generated from scratch; tiled up to --regions")
    ap.add_argument("--seed", type=int, default=2)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--schedule", default=None, choices=["static", "dynamic"])
    ap.add_argument("--group-regions", type=int, default=32, help="regions per hand-out group")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--verify-regions", type=int, default=2)
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-files", action="store_true", help="skip the from-files leg (writes a chr20-scale BAM to a temp dir)")
    ap.add_argument("--files-regions", type=int, default=0, help="regions of the from-files leg (default: --regions)")
    ap.add_argument("--files-steps", type=int, default=2)
    ap.add_argument("--files-batch", type=int, default=32, help="regions per batch of the from-files streaming session")
    ap.add_argument("--files-dist", action="store_true", help="N=1: run the from-files leg through DistributedVariantCaller + VariantFileSource "
                                                             "(the N>1 path) instead of VariantFromFiles.call_stream")
    ap.add_argument("--inflate-host-share", type=float, default=None,
                    help="from-files leg: share of the BGZF blocks inflated by the host pool beside the kernel (default 0: all on the GPU)")
    ap.add_argument("--host-inflate", action="store_true", help="from-files leg with the host zlib pool instead of the GPU inflate")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (float32 / float64, at most 64 MB: a seeded "
                         "sample of the rows of a larger output)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    cfg = CONFIGS[args.config]
    if args.regions is None:
        args.regions = int(os.environ.get("PB_BENCH_REGIONS", cfg["regions"]))
    if args.region_size is None:
        args.region_size = cfg["region_size"]
    if args.coverage is None:
        args.coverage = cfg["coverage"]
    if args.impl == "reference":
        run_reference(args, cfg)
    elif cfg["kind"] == "variant":
        run_variant(args, cfg)
    else:
        run_polish(args, cfg)


if __name__ == "__main__":
    main()
