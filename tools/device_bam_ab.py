"""Config 5 (the whole-genome leg of bench.py) through run_chunks with host and device BAM reading, alternating.

    python tools/device_bam_ab.py [--scale 1.0] [--runs 3] [--out DIR]

Two host budgets: all cores (bench.py's thread counts for one rank), and native_threads=2, loader_threads=1, which
stands in for one of 8 ranks on a 16-core host.  Before the timed runs it checks once per budget that the merged VCF
text of both modes is identical.  Per run: the loop's seconds, the host seconds of each stage of the loop (summed
over the threads that run it), and for device reading the summed device time of the parse stages (inflate, record
boundaries, parse + offsets + write, from c3r_wait_reads_stages).  The data set is bench.py's cfg5_dataset (made once
in its cache directory), the GPU's name and power limit are read (read-only) with nvidia-smi in the same run.  One
JSON line per run, then a summary line per budget."""
import argparse
import ctypes as C
import json
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools.device_calls_ab import gpu_info  # noqa: E402


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--scale", type=float, default=1.0, help="config-5 scale (bench.py --cfg5_scale)")
    ap.add_argument("--runs", type=int, default=3, help="timed runs of each mode per budget")
    ap.add_argument("--out", default=None, help="directory for the JSON lines (and nothing else)")
    a = ap.parse_args(argv)
    import bench
    from clair3_rna_b200 import run_chunks, weights
    from clair3_rna_b200.engine import Engine

    print("gpu:", gpu_info(), flush=True)
    cores = len(os.sched_getaffinity(0))
    cfg, bam, fa, wnpz, prep_s = bench.cfg5_dataset(a.scale, 0, 1, cores, lambda: None)
    print("config 5 at scale %g: %d contigs, data set ready in %.1f s" % (a.scale, len(cfg.contigs), prep_s), flush=True)
    eng = Engine(0, 18)
    eng.set_weights(weights.load(wnpz))
    # the parse stages' device time, split: sum c3r_wait_reads_stages over the tickets a run waits for
    split = [0.0, 0.0, 0.0]
    orig_wait = eng.wait

    def wait(ticket, release=True, copy=True):
        bam = ticket in eng._bam_of
        res = orig_wait(ticket, release=release and not bam, copy=copy)
        if bam:
            ms = (C.c_float * 3)()
            if eng.lib.c3r_wait_reads_stages(eng.ctx, ticket, ms) == 0:
                for k in range(3):
                    split[k] += ms[k]
            if release and copy:
                eng.release(ticket)
        return res
    eng.wait = wait
    budgets = {"all_cores": dict(loader_threads=max(1, min(4, cores // 2)), native_threads=max(1, cores // 2)),
               "rank_of_8_on_16_cores": dict(loader_threads=1, native_threads=2)}
    lines, summary = [], {}
    for bname, bkw in budgets.items():
        kw = dict(engine=eng, **bkw)
        with tempfile.TemporaryDirectory() as tmp:
            texts = []
            for dev in (False, True):                # also the warm-up of both modes
                out = os.path.join(tmp, "merged_%d.vcf" % dev)
                run_chunks.run(bam, fa, wnpz, out, device_bam=dev, **kw)
                texts.append(open(out, "rb").read())
            same = texts[0] == texts[1]
            print("%s: merged VCF identical with host and device BAM reading: %s (%d bytes, %d lines)" % (
                bname, same, len(texts[0]), texts[0].count(b"\n")), flush=True)
            if not same:
                return 1
        for k in range(2 * a.runs):
            dev = bool(k % 2)
            st = {}
            split[:] = [0.0, 0.0, 0.0]
            run_chunks.run(bam, fa, wnpz, None, merge=False, stats=st, device_bam=dev, **kw)
            hs = st["host_seconds"]
            rec = dict(budget=bname, device_bam=dev, loop_s=round(st["seconds"], 4), shards=st["shards"],
                       candidates=st["candidates"], host_s={k2: round(v, 4) for k2, v in hs.items()},
                       bam_device_ms=round(st["bam_device_ms"], 3),
                       inflate_ms=round(split[0], 3), boundaries_ms=round(split[1], 3), parse_write_ms=round(split[2], 3))
            lines.append(rec)
            print(json.dumps(rec), flush=True)
        med = lambda xs: sorted(xs)[len(xs) // 2]
        for dev in (False, True):
            rs = [r for r in lines if r["budget"] == bname and r["device_bam"] == dev]
            summary["%s/%s" % (bname, "device" if dev else "host")] = dict(
                loop_s=med([r["loop_s"] for r in rs]), fetch_s=med([r["host_s"]["fetch"] for r in rs]),
                load_wait_s=med([r["host_s"]["load_wait"] for r in rs]), wait_s=med([r["host_s"]["wait"] for r in rs]),
                bam_device_ms=med([r["bam_device_ms"] for r in rs]), inflate_ms=med([r["inflate_ms"] for r in rs]),
                boundaries_ms=med([r["boundaries_ms"] for r in rs]), parse_write_ms=med([r["parse_write_ms"] for r in rs]))
    eng.close()
    summary.update(gpu=gpu_info(), scale=a.scale, time=time.strftime("%Y-%m-%d %H:%M:%S"))
    print(json.dumps(summary), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "device_bam_ab.jsonl"), "w") as fp:
            fp.write("\n".join(json.dumps(r) for r in lines + [summary]) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
