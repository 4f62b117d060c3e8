#!/usr/bin/env python3
"""Headline benchmark: candidate sites/sec (pileup tensor generation + network inference).

Workload (BASELINE.json configs[1]): ont_r10_dorado_cdna on a synthetic chr20-sized
transcriptome at 30x, one contig per GPU (weak scaling: rank r gets its own contig of
the same size, no data-path collective).  A "step" is one pass of the hot path over the
whole contig.

  value        sites/s with the flat reads already resident in HBM (c3r_rerun_resident: one pass at a time)
  e2e          sites/s through the public API (Engine.submit / wait, three tickets in flight) from pinned host
               arrays, H2D and D2H of every step inside the timed region
  roofline     the network kernels (tensor bound); roofline_count / _k1 / _k3 / _k4: the integer stages (HBM bound)
  shard_cfg5   BASELINE.json configs[4]: the whole synthetic genome (24 contigs, 631 chunks) read from a BAM + FASTA,
               sharded by (contig, chunk) over the ranks through run_chunks (strong scaling, host limiter reported)
  cpu_baseline the oracle port of the reference CPU pipeline on a bounded sample

`--impl reference` times the oracle port (the reference is Python + samtools + TensorFlow,
none of which can run on the GPU box) with all host cores on bounded samples.

`--dump-outputs DIR` writes what the last timed end-to-end step returned to its caller as DIR/<name>.npy
(see dump_outputs), so that two builds can be compared output for output on the same seeded inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_SITE = {18: 47.786e6, 30: 48.597e6}       # SURVEY.md §8(d), BASELINE.md §3


E2E_DEPTH = int(os.environ.get("C3R_E2E_DEPTH", "2"))        # submits queued ahead of the one being waited for in the end-to-end leg (three tickets in flight)
# Generated inputs are cached between runs outside the source tree, which may be read-only.  One directory per user:
# a directory that another account left in a shared /tmp can be neither written to nor trusted.
CACHE_DIR = os.path.join(tempfile.gettempdir(), "c3r_bench_cache_%d" % os.getuid())
DUMP_LIMIT = 64 * 10 ** 6                                      # bytes written by --dump-outputs at most

def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        z = json.load(open(p))
        return dict(hbm=z["hbm_gbs"], tf_burst=z["bf16_tflops"], tf_sus=z["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sus=1400.0, src="fallback")


def measured_traffic(workload_name):
    """DRAM bytes per pass and stage from the newest committed `ncu --set full` capture (profiles/rN*_traffic.json,
    written by tools/make_profile_md.py), when it is of this workload: ({stage: bytes}, file name) or ({}, None)"""
    import glob
    for p in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")), reverse=True):
        z = json.load(open(p))
        if z.get("workload") == workload_name and "dram_bytes_per_stage" in z:
            return z["dram_bytes_per_stage"], os.path.relpath(p, ROOT)
    return {}, None


def dataset(cfg_idx, scale, contig_slot, cache_dir=CACHE_DIR):
    """reads + reference of one contig; `contig_slot` varies the seed per rank."""
    import dataclasses
    from clair3_rna_b200 import synth
    from clair3_rna_b200.reads import ReadBatch
    cfg = synth.config(cfg_idx, scale=scale)
    cfg = dataclasses.replace(cfg, seed=cfg.seed + 1000 * contig_slot, contigs=cfg.contigs[:1])
    os.makedirs(cache_dir, exist_ok=True)
    key = "%s_s%g_r%d" % (cfg.name, scale, contig_slot)
    path = os.path.join(cache_dir, key + ".npz")
    ref = synth.Reference(cfg)
    if os.path.exists(path):
        batch = ReadBatch.load(path)
    else:
        batch = synth.make_contig_reads(cfg, 0, ref)
        batch.save(path)
    return cfg, batch, ref


class ClockSampler(threading.Thread):
    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop_flag = gpu, [], False
        self.paused, self.lock = False, threading.Lock()

    def sample(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q,
                                  "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout
            row = [x.strip() for x in out.strip().split(",")]
            if len(row) >= 7:
                self.rows.append(row)
        except Exception:
            pass

    def run(self):
        while not self.stop_flag:
            if not self.paused:
                with self.lock:
                    self.sample()
            time.sleep(0.2)

    def pause(self):
        """nvidia-smi takes driver locks that stall CUDA API calls: the wall-clock (end-to-end) leg runs without it,
        the device-timed leg (CUDA events around each pass) is sampled throughout"""
        self.paused = True
        with self.lock:                      # a query in flight has returned
            pass

    def summary(self):
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons)}


# ------------------------------------------------------------------ CPU oracle legs
# The reference pipeline on the host cores, stage by stage (SURVEY.md 8d): mpileup text -> generate_tensor windows
# (producer, oracle/pileup_oracle.py), then batches of 200 through the fp32 network (oracle/model.py, one torch
# thread like call_variants.py:200-206) and every candidate through the decoder (output_with restated in
# clair3_rna_b200/decoder.py:vcf_row) - the consumer.  The reference itself (Python + samtools + TensorFlow) cannot
# travel to the GPU box, so this is the port (kind "port").
_W = {}


def _cpu_init(w):
    import torch
    torch.set_num_threads(1)                 # call_variants.py:200-206
    _W["w"] = w                              # weights once per worker, not once per job


def _cpu_worker(args):
    """one job = one region: -> (candidates, producer seconds, consumer seconds)"""
    from oracle import pileup_oracle, model
    from clair3_rna_b200 import decoder
    batch, ref_seq, ref_start1, s1, e1, contig, phased, padding = args
    t0 = time.time()
    out = pileup_oracle.run_region(batch, ref_seq, ref_start1, s1, e1, phased=phased, padding=padding)
    t1 = time.time()
    n = len(out["pos"])
    for i in range(0, n, 200):               # predictBatchSize, param_p.py:51
        p = model.forward(_W["w"], out["tensor"][i:i + 200])
        for k in range(p.shape[0]):
            decoder.vcf_row(contig, int(out["pos"][i + k]), out["ref33"][i + k], out["alt_info"][i + k], p[k])
    return n, t1 - t0, time.time() - t1


def cpu_jobs(cfg, batch, ref, n_jobs, span=4000):
    """n_jobs regions of about equal cost: the first `span` bp of the read clusters of the contig's genes, largest
    first (the pool hands them out one at a time, so the workers finish together)"""
    from clair3_rna_b200 import synth
    genes = synth.make_genes(cfg, 0, ref)
    contig = cfg.contigs[0][0]
    jobs = []
    for g in genes:
        s1 = max(1, g.exons[0][0] - 100)
        e1 = min(g.exons[-1][1] + 100, s1 + span)
        sub = batch.fetch(s1, e1)
        if sub.n_reads < 8:
            continue
        rs1 = max(1, s1 - 1000)
        jobs.append((sub, ref.fetch_str(contig, rs1 - 1, e1 + 1000), rs1, s1, e1, contig, cfg.phased, cfg.padding))
        if len(jobs) >= n_jobs:
            break
    jobs.sort(key=lambda j: -j[0].n_reads)
    return jobs


class CpuPipeline:
    """persistent pool of worker processes over a fixed job list"""

    def __init__(self, cfg, batch, ref, w, cores, n_jobs):
        import multiprocessing as mp
        self.jobs = cpu_jobs(cfg, batch, ref, n_jobs)
        self.cores = cores
        self.w = w
        self.pool = mp.get_context("fork").Pool(cores, initializer=_cpu_init, initargs=(w,)) if cores > 1 else None
        if self.pool is None:
            _cpu_init(w)

    def step(self):
        t0 = time.time()
        if self.pool is not None:
            out = list(self.pool.imap_unordered(_cpu_worker, self.jobs, chunksize=1))
        else:
            out = [_cpu_worker(j) for j in self.jobs]
        dt = time.time() - t0
        return sum(o[0] for o in out), dt, sum(o[1] for o in out), sum(o[2] for o in out)

    def close(self):
        if self.pool is not None:
            self.pool.close()
            self.pool.join()


def run_cpu(cfg, batch, ref, w, C, cores, n_jobs):
    cp = CpuPipeline(cfg, batch, ref, w, cores, n_jobs)
    try:
        return cp.step()
    finally:
        cp.close()


# ------------------------------------------------------------------ config 5: the sharded whole-genome leg
# BASELINE.json configs[4]: 24 contigs with GRCh38 lengths, ont_dorado_drna004, partitioned by (contig, 5 Mb chunk)
# exactly like the reference's CHUNK_LIST (run_clair3_rna:441-449, 681-706); rank r takes its greedy-LPT share
# (sharder.assign), reads its chunks from a real BAM + FASTA (native BGZF/BAI reader), runs them through
# Engine.submit / wait with one ticket ahead, decodes VCF rows natively and leaves them to rank 0, which merges with
# sort_vcf semantics.  Strong scaling: the genome is fixed, the ranks share it.
def _cfg5_make_contig(args):
    scale, ci, path = args
    from clair3_rna_b200 import synth
    cfg = synth.config(5, scale=scale)
    b = synth.make_contig_reads(cfg, ci, synth.Reference(cfg))
    b.save(path)
    return ci


def cfg5_dataset(scale, rank, world, cores, barrier, cache_dir=CACHE_DIR):
    """reads.bam (+ .bai), genome.fa (+ .fai), weights.npz of the config-5 genome at `scale`, made once per box:
    the ranks generate the contigs between them (process pools), rank 0 then writes the BAM, the last rank the FASTA"""
    import multiprocessing as mp
    from clair3_rna_b200 import synth, weights
    from clair3_rna_b200.reads import ReadBatch
    from clair3_rna_b200.bam import write_bam
    cfg = synth.config(5, scale=scale)
    d = os.path.join(cache_dir, "cfg5_s%g" % scale)
    os.makedirs(d, exist_ok=True)
    bam, fa, wnpz = os.path.join(d, "reads.bam"), os.path.join(d, "genome.fa"), os.path.join(d, "weights.npz")
    done = os.path.join(d, "done")
    t0 = time.time()
    if not os.path.exists(done):
        mine = [(scale, ci, os.path.join(d, "c%d.npz" % ci)) for ci in range(len(cfg.contigs))
                if ci % world == rank and not os.path.exists(os.path.join(d, "c%d.npz" % ci))]
        if mine:
            # largest contigs first; the pool is sized to this rank's share of the host cores
            with mp.get_context("fork").Pool(max(1, min(len(mine), cores // world))) as pool:
                list(pool.imap_unordered(_cfg5_make_contig, sorted(mine, key=lambda a: -cfg.contigs[a[1]][1]), chunksize=1))
        barrier()
        if rank == 0:
            batches = {cfg.contigs[ci][0]: ReadBatch.load(os.path.join(d, "c%d.npz" % ci)) for ci in range(len(cfg.contigs))}
            write_bam(bam, cfg.contigs, batches, level=1)
            weights.save(wnpz, weights.synthetic(18, sharpen=8.0))
        if rank == world - 1:
            ref = synth.Reference(cfg)
            off = 0
            with open(fa, "wb") as fp, open(fa + ".fai", "w") as fi:
                for name, length in cfg.contigs:
                    hdr = (">%s\n" % name).encode()
                    fp.write(hdr)
                    off += len(hdr)
                    fi.write("%s\t%d\t%d\t60\t61\n" % (name, length, off))
                    for s0 in range(0, length, 60 * (1 << 16)):
                        a = ref.fetch(name, s0, min(length, s0 + 60 * (1 << 16)))
                        full = (a.size // 60) * 60
                        lines = np.empty((full // 60, 61), np.uint8)
                        lines[:, :60] = a[:full].reshape(-1, 60)
                        lines[:, 60] = 10
                        fp.write(lines.tobytes())
                        off += lines.size
                        if a.size > full:
                            fp.write(a[full:].tobytes() + b"\n")
                            off += a.size - full + 1
        barrier()
        if rank == 0:
            open(done, "w").write("ok\n")
    barrier()
    return cfg, bam, fa, wnpz, time.time() - t0


def shard_cfg5_leg(scale, rank, world, local_rank, cores, barrier, gloo, eng):
    """-> dict for the bench line (rank 0) or None"""
    import pickle
    import torch.distributed as dist
    from clair3_rna_b200 import run_chunks
    cfg, bam, fa, wnpz, prep_s = cfg5_dataset(scale, rank, world, cores, barrier)
    tmp = os.path.join(os.path.dirname(bam), "rows_w%d" % world)
    os.makedirs(tmp, exist_ok=True)

    def gather(rows_of):
        # per-shard VCF rows are left on the node's file system, like the reference's tmp/pileup_output/*.vcf
        with open(os.path.join(tmp, "rank%d.pkl" % rank), "wb") as fp:
            pickle.dump(rows_of, fp, protocol=4)
        barrier()
        if rank != 0:
            return None
        return [pickle.load(open(os.path.join(tmp, "rank%d.pkl" % r), "rb")) for r in range(world)]

    cold = {}
    barrier()
    n_loaders, n_native = max(1, min(4, cores // (2 * world))), max(1, cores // (2 * world))
    # first pass: cold (BAM handles and their indexes opened, file cache and buffers touched for the first time)
    run_chunks.run(bam, fa, wnpz, None, device=local_rank, rank=rank, world=world, merge=False, stats=cold,
                   engine=eng, loader_threads=n_loaders, native_threads=n_native)
    # two warm passes (a 1-2 s loop over 631 chunks is exposed to a single host hiccup): the better one is reported,
    # both times are listed; the second one also gathers and merges the rows
    warm1 = {}
    barrier()
    run_chunks.run(bam, fa, wnpz, None, device=local_rank, rank=rank, world=world, merge=False, stats=warm1,
                   engine=eng, loader_threads=n_loaders, native_threads=n_native)
    stats = {}
    barrier()
    t0 = time.time()
    merged = run_chunks.run(bam, fa, wnpz, os.path.join(tmp, "merged.vcf") if rank == 0 else None, device=local_rank,
                            rank=rank, world=world, gather=gather if world > 1 else None, stats=stats, engine=eng,
                            loader_threads=n_loaders, native_threads=n_native)
    t_all = time.time() - t0
    mine = dict(rank=rank, shards=stats["shards"], candidates=stats["candidates"], loop_s=stats["seconds"], cold_loop_s=cold["seconds"],
                host_s=stats["host_seconds"], cost=stats["cost"], total_s=t_all,
                warm1_loop_s=warm1["seconds"], warm1_host_s=warm1["host_seconds"])
    if world > 1:
        allst = [None] * world
        dist.all_gather_object(allst, mine, group=gloo)
    else:
        allst = [mine]
    if rank != 0:
        return None
    pass_times = [max(a["warm1_loop_s"] for a in allst), max(a["loop_s"] for a in allst)]
    if pass_times[0] < pass_times[1]:                    # the first warm pass was the better one: report its loop
        for a in allst:
            a["loop_s"], a["host_s"] = a["warm1_loop_s"], a["warm1_host_s"]
    n = sum(a["candidates"] for a in allst)
    t_max = max(a["loop_s"] for a in allst)
    t_mean = sum(a["loop_s"] for a in allst) / world
    cost = [a["cost"] for a in allst]
    return {
        "workload": "%s at scale %g: %d contigs, %d bp, %d (contig, chunk) shards, %d reads in one BAM" % (
            cfg.name, scale, len(cfg.contigs), sum(l for _, l in cfg.contigs), stats["total_shards"],
            int(sum(c for c in cost))),
        "scaling": "strong", "n_gpus": world,
        "value": n / t_max if t_max > 0 else 0.0, "unit": "sites/s",
        "note": "candidates of the whole genome / slowest rank's loop (BAM fetch -> submit -> wait -> native decode, one "
                "ticket ahead, loader and decoder threads beside the submitting thread), the better of two warm passes over the "
                "genome in the same process (the first, cold pass is reported beside them); the rank-0 merge (Python "
                "sort_vcf restatement) is timed apart",
        "candidates": n, "merged_rows": len(merged) if merged is not None else None,
        "slowest_rank_s": t_max, "mean_rank_s": t_mean, "imbalance": t_max / t_mean if t_mean > 0 else None,
        "cold_pass_slowest_rank_s": max(a["cold_loop_s"] for a in allst),
        "warm_passes_slowest_rank_s": pass_times,
        "lpt_cost_imbalance": max(cost) / (sum(cost) / world) if sum(cost) > 0 else None,
        "merge_and_write_s": t_all - stats["seconds"],
        "per_rank": [{"rank": a["rank"], "shards": a["shards"], "candidates": a["candidates"], "loop_s": round(a["loop_s"], 3),
                      "host_s": {k: round(v, 3) for k, v in a["host_s"].items()}} for a in allst],
        "host_feed": "host seconds of the slowest rank: " + ", ".join(
            "%s %.2f" % (k, v) for k, v in max(allst, key=lambda a: a["loop_s"])["host_s"].items()),
        "host": (lambda a: {
            "cores": cores, "ranks": world, "loader_threads_per_rank": n_loaders, "native_threads_per_call": n_native,
            # share of the slowest rank's loop each host thread group is busy: the largest one is what bounds the loop
            "busy": {"decoder threads (2; c3r_decode_vcf + row strings), each": round(a["host_s"]["decode"] / 2 / a["loop_s"], 3),
                     "loader threads (BAM fetch + inflate, FASTA window), each": round((a["host_s"]["fetch"] + a["host_s"]["ref"]) / n_loaders / a["loop_s"], 3),
                     "submitting thread: submit + wait for the device": round((a["host_s"]["submit"] + a["host_s"]["wait"]) / a["loop_s"], 3),
                     "submitting thread: waiting for the decoder": round(a["host_s"]["decode_wait"] / a["loop_s"], 3),
                     "submitting thread: waiting for a loader": round(a["host_s"]["load_wait"] / a["loop_s"], 3)},
            "cpu_seconds_per_genome": round(sum(x["host_s"][k] for x in allst for k in ("fetch", "ref", "submit", "decode")), 2),
        })(max(allst, key=lambda a: a["loop_s"])),
        "dataset_prep_s": prep_s,
    }


# ------------------------------------------------------------------ outputs of the timed path
def dump_outputs(out_dir, r, seed=0):
    """Writes the arrays of a ChunkResult as the caller of Engine.wait receives them, one .npy each: pos, depth,
    alt_off, alt_n (int, stored as float64, which holds them exactly), probs (float32) and alt_<field> for the fields
    of the allele table.  The allele table holds each candidate's alt_n entries in candidate order (the slots between
    two candidates' entries are never written, so they are left out).  When all of it would exceed DUMP_LIMIT bytes,
    a fixed, seeded sample of the candidates is written, in ascending order.  -> (candidates written, candidates)"""
    n = r.n_cand
    alt_n = r.alt_n.astype(np.int64)
    cost = 4 * 8 + 24 * 4 + 8 * len(r.alt.dtype.names) * alt_n          # bytes written per candidate
    budget = DUMP_LIMIT - 4096                                           # less the .npy headers
    keep = np.arange(n)
    if cost.sum() > budget:
        order = np.random.default_rng(seed).permutation(n)
        keep = np.sort(order[np.cumsum(cost[order]) <= budget])
    k_n = alt_n[keep]
    first = np.repeat(r.alt_off[keep], k_n)
    within = np.arange(int(k_n.sum())) - np.repeat(np.cumsum(k_n) - k_n, k_n)
    alt = r.alt[first + within]
    arrays = {"pos": r.pos[keep], "depth": r.depth[keep], "probs": r.probs[keep], "alt_off": r.alt_off[keep],
              "alt_n": r.alt_n[keep]}
    arrays.update(("alt_" + f, alt[f]) for f in alt.dtype.names)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32 if a.dtype == np.float32 else np.float64))
    return keep.size, n


# ------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--nn_impl", type=int, default=1)
    ap.add_argument("--no_cpu_baseline", action="store_true")
    ap.add_argument("--cfg5_scale", type=float, default=1.0,
                    help="genome scale of the sharded config-5 leg (1.0 = GRCh38 lengths, 631 chunks; 0 = skip the leg)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed end-to-end step returned (rank 0) as DIR/<name>.npy, "
                         "float32 / float64, at most 64 MB")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    from clair3_rna_b200 import weights, params as P
    cfg, batch, ref = dataset(args.config, args.scale, rank)
    contig, clen = cfg.contigs[0]
    C = 30 if cfg.phased else 18
    w = weights.synthetic(C, sharpen=8.0)
    workload = "%s: %s, 1 contig %s of %d bp per GPU, %d reads, %.1fM aligned bases" % (
        cfg.name, cfg.platform, contig, clen, batch.n_reads, batch.n_aligned_bases() / 1e6)
    cores = len(os.sched_getaffinity(0))

    if args.impl == "reference":
        if rank != 0:
            return
        # a bounded sample per step (the same >= 4 jobs per worker every step) so that W+K steps end within minutes
        n_jobs = 4 * cores
        cp = CpuPipeline(cfg, batch, ref, w, cores, n_jobs)
        vals = []
        for i in range(args.warmup + args.steps):
            r = cp.step()
            if i >= args.warmup:
                vals.append(r)
        cp.close()
        one = CpuPipeline(cfg, batch, ref, w, 1, max(4, n_jobs // cores))       # the same pipeline in one process
        n1, dt1, _, _ = one.step()
        n = sum(v[0] for v in vals)
        dt = sum(v[1] for v in vals)
        prod, cons = sum(v[2] for v in vals), sum(v[3] for v in vals)
        v = n / dt if dt > 0 else 0.0
        v1 = n1 / dt1 if dt1 > 0 else 0.0
        sample = ("%d regions of <= 4 kb around the first exons of the workload's genes per step (%d candidate sites/step), "
                  "oracle port: mpileup text -> generate_tensor -> fp32 network (batch 200, 1 torch thread) -> VCF row decode; "
                  "%d persistent worker processes, jobs handed out largest first; the full workload is %d reads - a sample, "
                  "hence not the same config as the GPU arm" % (len(cp.jobs), vals[0][0] if vals else 0, cores, batch.n_reads))
        print(json.dumps({
            "impl": "reference", "metric": "candidate sites/sec (tensor+inference)", "value": v, "unit": "sites/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / max(1, len(vals)), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32+f32", "data": "synthetic",
            "config": {"workload": workload, "sample": sample},
            "cpu_baseline": {"value": v, "unit": "sites/s", "cores": cores, "kind": "port", "sample": sample,
                             "sites_per_s_per_core": v / cores, "one_process_sites_per_s": v1,
                             "parallel_speedup": (v / v1) if v1 > 0 else None,
                             "producer_share": prod / (prod + cons) if prod + cons > 0 else None,
                             "consumer_share": cons / (prod + cons) if prod + cons > 0 else None},
            "e2e": {"value": v, "unit": "sites/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import torch
    import torch.distributed as dist
    gloo = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        gloo = dist.new_group(backend="gloo")           # python objects (per-rank statistics) travel over gloo
    torch.cuda.set_device(local_rank)
    from clair3_rna_b200.engine import Engine
    eng = Engine(local_rank, C, enable_padding=cfg.padding, nn_impl=args.nn_impl)
    eng.set_weights(w)
    # one chunk = the whole contig (all 5 Mb reference chunks batched into one submit)
    region = (1, clen + P.NO_OF_POSITIONS)
    ref_arr = ref.fetch(contig, 0, clen)
    # pinned host staging for the e2e leg
    pin = {}
    for k in ("pos", "flag", "mapq", "hp", "cigar_off", "cigar", "seq_off", "seq"):
        a = getattr(batch, k)
        tsr = torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).copy()).pin_memory()
        pin[k] = tsr.numpy().view(a.dtype)
    from clair3_rna_b200.reads import ReadBatch
    pbatch = ReadBatch(batch.contig, **pin)
    pref = torch.from_numpy(ref_arr.copy()).pin_memory().numpy()
    eng.set_reference(pref, 1)                # the contig's reference stays resident, like the weights
    h2d = sum(v.nbytes for v in pin.values())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident leg
    ticket = eng.submit(pbatch, None, 1, region[0], region[1])
    res0 = eng.wait(ticket, release=False)
    n_cand, n_rows = res0.n_cand, res0.n_rows
    first_pos = int(res0.pos[0]) if n_cand else -1
    d2h = res0.pos.nbytes + res0.depth.nbytes + res0.probs.nbytes + res0.alt_off.nbytes + res0.alt_n.nbytes + res0.alt.nbytes
    sampler = ClockSampler(local_rank)        # samples nvidia-smi through the warm-up, the timed steps and the e2e leg
    sampler.start()
    for _ in range(args.warmup):
        flush.fill_(1)
        eng.rerun_resident(ticket)
    barrier()
    tot_ms, stage_acc, launches = 0.0, np.zeros(8), 0
    t_wall0 = time.time()
    for _ in range(args.steps):
        flush.fill_(1)                       # L2 flush between timed iterations
        torch.cuda.synchronize()
        ms, st, nl = eng.rerun_resident(ticket)
        tot_ms += ms
        stage_acc += np.array(st)
        launches += nl
    barrier()
    eng.release(ticket)
    t_dev = torch.tensor([tot_ms], dtype=torch.float64, device="cuda")
    n_all = torch.tensor([float(n_cand)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t_dev, op=dist.ReduceOp.MAX)
        dist.all_reduce(n_all, op=dist.ReduceOp.SUM)
    value = float(n_all.item()) * args.steps / (float(t_dev.item()) / 1e3)

    # ---- end-to-end leg: public API, host arrays in, host results out
    for _ in range(min(args.warmup, 2)):              # warm the tickets' buffers
        ts = [eng.submit(pbatch, None, 1, region[0], region[1]) for _ in range(E2E_DEPTH + 1)]
        for t in ts:
            eng.wait(t)
    # E2E_DEPTH + 1 = 3 tickets in flight: while the GPU runs step i's network, step i+2's H2D copies and position /
    # row stages run on the SMs it leaves idle, and step i+1's window / allele / network stages are already queued
    # (c3r_wait queues them as soon as the candidate count is in) - so LSTM1 of step i+1 runs beside the remainder
    # round of step i's LSTM2 (tc_forward).  The pipeline is primed with untimed submits (like warm-up steps) and
    # drained after the timed region: each of the K timed steps is one submit (its H2D inside) + one wait (its D2H
    # inside).
    sampler.pause()
    barrier()
    from collections import deque
    inflight = deque(eng.submit(pbatch, None, 1, region[0], region[1]) for _ in range(E2E_DEPTH))
    t0 = time.time()
    for i in range(args.steps):
        inflight.append(eng.submit(pbatch, None, 1, region[0], region[1]))
        tk = inflight.popleft()
        r = eng.wait(tk, copy=False)                   # results as numpy arrays over the library's pinned buffers
        assert r.n_cand == n_cand and r.probs.shape == (n_cand, 24) and (n_cand == 0 or r.pos[0] == first_pos)
        if i + 1 < args.steps:
            eng.release(tk)
    e2e_wall = time.time() - t0
    # the last timed step's results against the first (sequential) call of this run: same inputs, same outputs
    # (the alt table is not compared as a block: the slots between two candidates' entries are never written)
    assert np.array_equal(r.pos, res0.pos) and np.array_equal(r.probs, res0.probs) and np.array_equal(r.alt_n, res0.alt_n)
    if args.dump_outputs and rank == 0:
        print("--dump-outputs: %d of %d candidates written to %s" % (dump_outputs(args.dump_outputs, r) + (args.dump_outputs,)),
              file=sys.stderr)
    eng.release(tk)
    while inflight:
        eng.wait(inflight.popleft())                   # drain (untimed)
    barrier()
    e2e_t = torch.tensor([e2e_wall], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e = float(n_all.item()) * args.steps / float(e2e_t.item())
    if not sampler.rows:                     # very short runs: take one sample with the GPU still busy
        tk = eng.submit(pbatch, None, 1, region[0], region[1])
        sampler.sample()
        eng.wait(tk)
    sampler.stop_flag = True
    shard5 = None
    if args.cfg5_scale > 0 and C == 18 and not cfg.padding:
        # the same engine (its buffers are warm, like in a process that has been running for a while)
        shard5 = shard_cfg5_leg(args.cfg5_scale, rank, world, local_rank, cores, barrier, gloo, eng)
    eng.close()

    if rank == 0:
        pk = peaks()
        st = stage_acc / args.steps                              # ms per step per stage
        k5_ms, k2_ms = float(st[6]), float(st[2]) + float(st[3])    # K2 = compare/event pass + row pass
        tr, tr_src = measured_traffic(cfg.name) if args.scale == 1.0 else ({}, None)
        flops = FLOP_PER_SITE[C] * n_cand
        ach_tf = flops / (k5_ms * 1e-3) / 1e12 if k5_ms > 0 else 0.0
        # algorithmic bytes per unit (DESIGN.md section 4 / SURVEY.md 8d)
        NW = (clen + P.NO_OF_POSITIONS + 31) // 32
        KX = 48 if C == 18 else 64
        alg = {
            # K1: 4 B read + 12 B written per op, ~30 B per read; 8 B (covA, covE) + 4 B (rowR) + 4 B read again + 4 B
            # (word_base) per 32 positions; 4 B (row_pos) + 24 B of zeroed accumulators per row
            "k1": 16.0 * batch.n_ops + 30.0 * batch.n_reads + 20.0 * NW + 28.0 * n_rows,
            "k2": 0.5 * batch.n_aligned_bases() + 16.0 * batch.n_ops + (4 * C + 8) * n_rows,  # bases, ops, count rows
            "k3": 9.0 * n_rows + 12.0 * n_cand,                                              # flag + bitmap per row, list entry
            "k4": (33 * 4 * C + 33 * KX * 2) * float(n_cand),                                # window read, operand image written
        }

        def hbm_roofline(kernel, key, ms):
            gbs = alg[key] / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
            return {"kernel": kernel, "bound": "hbm", "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": gbs / pk["hbm"],
                    "traffic": tr.get(key), "algorithmic_bytes": alg[key], "ms": ms, "peak_source": pk["src"], "traffic_source": tr_src}
        line = {
            "metric": "candidate sites/sec (tensor+inference)", "value": value, "unit": "sites/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": float(t_dev.item()) / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32 pileup + fp16/fp32-accumulate network" if args.nn_impl == 1 else "int32+f32",
            "data": "synthetic",
            "config": {"workload": workload, "candidates_per_gpu": n_cand, "rows_per_gpu": n_rows, "channels": C,
                       "l2_flush": "256 MiB write between timed steps", "reference": "resident in HBM (c3r_set_reference), not part of h2d", "nn_impl": args.nn_impl,
                       "timed_region": "value: the CUDA-event times of the K passes summed (%.1f ms in all, one pass per step, L2 flushed in "
                                       "between); e2e: wall clock over K submit + wait pairs with %d tickets in flight (%.1f ms)" % (
                                           float(t_dev.item()), E2E_DEPTH + 1, 1e3 * float(e2e_t.item()))},
            "e2e": {"value": e2e, "unit": "sites/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "tickets_in_flight": E2E_DEPTH + 1},
            "gpu_launches": int(launches),
            "clocks": sampler.summary(),
            "stage_ms": {"memset": float(st[0]), "k1_scan_rows": float(st[1]), "k2_compare_events": float(st[2]), "k2_rows": float(st[3]),
                         "k3_filter": float(st[4]), "k4_window_alt": float(st[5]), "k5_network": k5_ms},
            "roofline": {"kernel": "K5 network (k_lstm_tc<4>, k_lstm2_fused, k_gemm_tc L4 + L5, k_l4_finish, k_heads_out)", "bound": "tensor",
                         "achieved": ach_tf, "peak": pk["tf_sus"], "unit": "TFLOP/s", "frac": ach_tf / pk["tf_sus"],
                         "traffic": tr.get("k5"), "traffic_source": tr_src,
                         "peak_source": pk["src"] + " bf16 sustained",
                         "hbm_gbs_of_traffic": (tr["k5"] / (k5_ms * 1e-3) / 1e9) if (tr.get("k5") and k5_ms > 0) else None,
                         "note": "useful flops (47.786 MFLOP/site) over the CUDA-event time of the network kernels of a pass; "
                                 "traffic = h1 and h2 (hi + lo) written once and read once, nothing else of size leaves the SMs "
                                 "(profiles/, newest rN summary)"},
            "roofline_count": hbm_roofline("K2 count path (k_cmp, event scan, k_scatter, k_rows)", "k2", k2_ms),
            "roofline_k1": hbm_roofline("K1 CIGAR geometry, coverage bitmaps, row bits and ranks (k_cigar, k_row_bits, k_row_rank)", "k1", float(st[1])),
            "roofline_k3": hbm_roofline("K3 candidate list (k_cand_emit; the window test runs inside k_rows)", "k3", float(st[4])),
            "roofline_k4": hbm_roofline("K4 window assembly into LSTM1's operand images + alt table", "k4", float(st[5])),
        }
        if not args.no_cpu_baseline:
            n, dt, prod, cons = run_cpu(cfg, batch, ref, w, C, 1, 12)
            line["cpu_baseline"] = {"value": n / dt if dt > 0 else 0.0, "unit": "sites/s", "cores": 1, "kind": "port",
                                    "sample": "12 regions of <= 4 kb of the workload (%d candidate sites, %.1f s), oracle port "
                                              "(mpileup text -> generate_tensor -> fp32 network, batch 200 -> VCF row decode), "
                                              "1 process; producer %.0f %% / consumer %.0f %% of the time" % (
                                                  n, dt, 100 * prod / max(prod + cons, 1e-9), 100 * cons / max(prod + cons, 1e-9))}
        if shard5 is not None:
            line["shard_cfg5"] = shard5
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
