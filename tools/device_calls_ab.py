"""Config 5 (the whole-genome leg of bench.py) through run_chunks with call records off and on, alternating.

    python tools/device_calls_ab.py [--scale 1.0] [--runs 3] [--out DIR]

Per run: the loop's seconds, the decoder workers' host seconds (summed over the two) and the share of the loop a
worker is busy, the submitting thread's wait for the decoder, and the summed device time of k_call with its share
of the loop.  Before the timed runs it checks once that the merged VCF text of both
modes is identical.  The data set is bench.py's cfg5_dataset (made once in its cache directory), the GPU's name and
power limit are read (read-only) with nvidia-smi in the same run.  One JSON line per run, then a summary line."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=60).stdout
        return out.strip().splitlines()[0]
    except Exception as e:                           # the measurement stands without it, but says so
        return "unknown (%s)" % e


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--scale", type=float, default=1.0, help="config-5 scale (bench.py --cfg5_scale)")
    ap.add_argument("--runs", type=int, default=3, help="timed runs of each mode")
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
    # bench.py's thread counts for one rank
    kw = dict(engine=eng, loader_threads=max(1, min(4, cores // 2)), native_threads=max(1, cores // 2))
    with tempfile.TemporaryDirectory() as tmp:
        texts = []
        for on in (False, True):                     # also the warm-up of both modes
            out = os.path.join(tmp, "merged_%d.vcf" % on)
            run_chunks.run(bam, fa, wnpz, out, device_calls=on, **kw)
            texts.append(open(out, "rb").read())
        same = texts[0] == texts[1]
        print("merged VCF identical with records off and on: %s (%d bytes, %d lines)" % (
            same, len(texts[0]), texts[0].count(b"\n")), flush=True)
        if not same:
            return 1
    lines = []
    for k in range(2 * a.runs):
        on = bool(k % 2)
        st = {}
        run_chunks.run(bam, fa, wnpz, None, merge=False, stats=st, device_calls=on, **kw)
        loop = st["seconds"]
        rec = dict(device_calls=on, loop_s=round(loop, 4), candidates=st["candidates"], shards=st["shards"],
                   decode_host_s=round(st["host_seconds"]["decode"], 4),
                   # run_chunks decodes on two worker threads: the share of the loop one of them is busy
                   decoder_busy=round(st["host_seconds"]["decode"] / (2 * loop), 4),
                   decode_wait_s=round(st["host_seconds"]["decode_wait"], 4),
                   k_call_ms=round(st["call_device_ms"], 3), k_call_share=round(st["call_device_ms"] / 1e3 / loop, 5))
        lines.append(rec)
        print(json.dumps(rec), flush=True)
    eng.close()
    med = lambda xs: sorted(xs)[len(xs) // 2]
    summary = {}
    for on in (False, True):
        rs = [r for r in lines if r["device_calls"] == on]
        summary["on" if on else "off"] = {k: med([r[k] for r in rs]) for k in ("loop_s", "decode_host_s", "decoder_busy",
                                                                              "decode_wait_s", "k_call_ms")}
    summary.update(gpu=gpu_info(), scale=a.scale, identical_vcf=same, time=time.strftime("%Y-%m-%d %H:%M:%S"))
    print(json.dumps(summary), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "device_calls_ab.jsonl"), "w") as fp:
            fp.write("\n".join(json.dumps(r) for r in lines + [summary]) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
