"""Config 5 (the whole-genome leg of bench.py) through run_chunks in three modes, alternating: host decode (the
default), --device_calls (decisions on the GPU, rows printed on the host) and --device_vcf (rows printed on the GPU).

    python tools/device_vcf_ab.py [--scale 1.0] [--runs 3] [--out DIR]

Two host budgets: all cores (bench.py's thread counts for one rank), and native_threads=2, loader_threads=1, which
stands in for one of 8 ranks on a 16-core host.  Before the timed runs it checks once per budget that the merged VCF
text of the three modes is identical.  Per run: the loop's seconds, the decoder workers' host seconds (summed over
the two), the submitting thread's wait for them, the device time of the text kernels and the bytes their copies move
to the host (each ticket's bound: candidates times the row bound of its contig).  The data set is bench.py's
cfg5_dataset (made once in its cache directory), the GPU's name and power limit are read (read-only) with nvidia-smi
in the same run.  One JSON line per run, then a summary line per budget."""
import argparse
import json
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools.device_calls_ab import gpu_info  # noqa: E402

MODES = {"host": {}, "device_calls": dict(device_calls=True), "device_vcf": dict(device_vcf=True)}


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
    budgets = {"all_cores": dict(loader_threads=max(1, min(4, cores // 2)), native_threads=max(1, cores // 2)),
               "2_cores": dict(loader_threads=1, native_threads=2)}
    lines, summary = [], []
    for budget, threads in budgets.items():
        kw = dict(engine=eng, **threads)
        with tempfile.TemporaryDirectory() as tmp:
            texts = {}
            for mode, opt in MODES.items():              # also the warm-up of every mode
                out = os.path.join(tmp, "merged_%s.vcf" % mode)
                run_chunks.run(bam, fa, wnpz, out, **opt, **kw)
                texts[mode] = open(out, "rb").read()
            same = len(set(texts.values())) == 1
            print("%s: merged VCF identical in all modes: %s (%d bytes, %d lines)" % (
                budget, same, len(texts["host"]), texts["host"].count(b"\n")), flush=True)
            if not same:
                return 1
        mine = []
        for k in range(a.runs):
            for mode, opt in MODES.items():
                st = {}
                run_chunks.run(bam, fa, wnpz, None, merge=False, stats=st, **opt, **kw)
                hs = st["host_seconds"]
                rec = dict(budget=budget, mode=mode, loop_s=round(st["seconds"], 4), candidates=st["candidates"],
                           decode_host_s=round(hs["decode"], 4), decode_wait_s=round(hs["decode_wait"], 4),
                           load_wait_s=round(hs["load_wait"], 4), vcf_device_ms=round(st["vcf_device_ms"], 3),
                           call_device_ms=round(st["call_device_ms"], 3), vcf_d2h_bytes=st["vcf_d2h_bytes"])
                mine.append(rec)
                print(json.dumps(rec), flush=True)
        lines += mine
        med = lambda xs: sorted(xs)[len(xs) // 2]
        s = dict(budget=budget, identical_vcf=same)
        for mode in MODES:
            rs = [r for r in mine if r["mode"] == mode]
            s[mode] = {k: med([r[k] for r in rs]) for k in ("loop_s", "decode_host_s", "decode_wait_s", "load_wait_s",
                                                            "vcf_device_ms", "vcf_d2h_bytes")}
            s[mode]["loop_s_range"] = [min(r["loop_s"] for r in rs), max(r["loop_s"] for r in rs)]
        summary.append(s)
        print(json.dumps(s), flush=True)
    eng.close()
    tail = dict(gpu=gpu_info(), scale=a.scale, time=time.strftime("%Y-%m-%d %H:%M:%S"))
    print(json.dumps(tail), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "device_vcf_ab.jsonl"), "w") as fp:
            fp.write("\n".join(json.dumps(r) for r in lines + summary + [tail]) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
