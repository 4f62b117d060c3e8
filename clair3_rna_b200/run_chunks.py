"""Pileup calling of a whole BAM on one or more GPUs: the CHUNK_LIST loop of the reference's workflow
(`parallel -j THREADS ... call_var_bam :::: CHUNK_LIST` then `sort_vcf`, /root/reference/run_clair3_rna:
378-381, 441-449, 681-706, 868-889) as one process per GPU.

    python -m clair3_rna_b200.run_chunks --bam_fn x.bam --ref_fn ref.fa --chkpnt_fn w.npz --output out.vcf
    python -m torch.distributed.run --nproc-per-node 8 -m clair3_rna_b200.run_chunks ...        # 8 GPUs

Shards = (contig, chunk) with the reference's geometry (chunk_num = ceil(len / 5 Mb)); they are independent, so
ranks share nothing on the data path: each rank owns one GPU, takes its shards by greedy LPT on the per-contig
mapped-read counts of the BAM index (what `samtools idxstats` gives run_clair3_rna:187), and only VCF rows are
gathered on rank 0 (gloo/nccl `gather_object`), merged with sort_vcf semantics (sharder.merge_rows).

Inside a rank the stages of consecutive shards overlap: while the GPU runs shard i (c3r_submit_chunk returns
once the work is queued), the host fetches + inflates the BAM blocks of shard i+1 and decodes the rows of
shard i-1 (c3r_decode_vcf, all host cores).

Region modes (`--bed_fn`, `--genotyping_mode_vcf_fn`, run_clair3_rna:319-345, 434-435): contigs are intersected
with those of the BED / VCF, the per-contig "split BED" (rows widened by 33 bp) becomes the pileup filter of
every chunk of the contig, and the chunk geometry follows the BED span / the site count (regions.plan_chunk).
"""
from __future__ import annotations

import argparse
import os
import sys
import time

from . import params as P
from . import decoder, fasta, regions, sharder, weights as W


def build_shards(contigs, mapped, chunk_size=P.CHUNK_SIZE):
    """contigs [(name, len)], mapped {name: reads} -> ([(name, len, chunk_id1, chunk_num)], [cost])"""
    shards, costs = [], []
    for name, length in contigs:
        n = mapped.get(name, 0)
        if n <= 0:
            continue
        num = max(1, -(-length // chunk_size))
        for i in range(num):
            shards.append((name, length, i + 1, num))
            costs.append(n / num)
    return shards, costs


def chunk_size_bytes():
    """bytes of the largest reference window of a chunk: the chunk, its reference flanks and the 33-column window"""
    return P.CHUNK_SIZE + 2 * P.EXPAND_REFERENCE_REGION + 4 * P.NO_OF_POSITIONS + 64


BAM_BUFFER_BYTES = 64 << 20                         # page-locked buffer of a chunk's compressed BAM bytes (device_bam)


def run(bam_fn, ref_fn, chkpnt_fn, output, *, contigs=None, device=0, rank=0, world=1, phased=False, padding=False,
        snp_min_af=P.SNP_MIN_AF, indel_min_af=P.INDEL_MIN_AF, min_coverage=P.MIN_COVERAGE, min_mq=P.MIN_MQ,
        qual=P.QUAL_CUT_OFF, sample_name="SAMPLE", gather=None, stats=None, bed_fn=None, vcf_fn=None, head_tail=False,
        merge_qual=None, show_ref=True, rediportal_fn=None, rediportal_tags=None, output_no_tagging=None,
        compress_vcf=False, engine=None, loader_threads=2, native_threads=0, merge=True, cmdline=None,
        device_calls=False, device_bam=False, device_vcf=False):
    """merge_qual / show_ref / rediportal_*: the options of the merge stage (sharder.sort_vcf = sort_vcf_from of the
    reference); the defaults keep every row as the chunks produced it.  engine: an Engine to reuse (its parameters and
    weights are then the caller's business); loader_threads: BAM / FASTA readers working ahead of the GPU;
    native_threads: threads of each BGZF inflate and of the row decoder (0 = all cores - give every rank its share
    when several ranks run on one host).  device_calls: decide the genotypes on the GPU (call records, k_call) and
    leave only the formatting to the decoder threads (c3r_format_vcf); the rows are the same.  A caller's engine
    gets its own device_calls setting back when the run ends.  device_bam: the loader threads only read the compressed
    BAM blocks of a chunk (BamFile.fetch_raw, into page-locked buffers) and the GPU inflates and parses them
    (Engine.submit_bam); the rows are the same.  device_vcf: the GPU also prints each chunk's rows (Engine.set_device_vcf,
    which implies the decisions on the GPU) and the decoder threads only split its text; the rows are the same, and a
    caller's engine gets its own setting back when the run ends."""
    from .bam import BamFile
    from .engine import Engine, PinnedPool, decode_vcf_rows, device_vcf_rows, format_vcf_rows
    fai = fasta.read_fai(ref_fn)
    bf = BamFile(bam_fn)
    idx = {n: m for n, _, m, _ in bf.idxstats()}
    conf_rows = regions.read_bed_rows(bed_fn) if bed_fn else None          # {contig: rows}
    known_pos = regions.read_known_positions(vcf_fn) if vcf_fn else None    # {contig: sites}
    ctgs = [(n, l) for n, l in zip(bf.references, bf.lengths) if n in fai and (contigs is None or n in contigs)
            and (conf_rows is None or n in conf_rows) and (known_pos is None or n in known_pos)]
    shards, costs = build_shards(ctgs, idx)
    owner = sharder.assign(costs, world)
    mine = [i for i in range(len(shards)) if owner[i] == rank]
    C = P.CHANNEL_SIZE + (P.PHASED_CHANNEL_SIZE if phased else 0)
    eng = engine
    calls_before = eng.device_calls if eng is not None else None
    vcf_before = eng._vcf_opts if eng is not None else None
    if eng is None:
        eng = Engine(device, C, snp_min_af=snp_min_af, indel_min_af=indel_min_af, min_coverage=min_coverage,
                     min_mq=min_mq, enable_padding=padding, enable_head_tail=head_tail, device_calls=device_calls)
        eng.set_weights(W.load(chkpnt_fn))
    elif eng.device_calls != bool(device_calls):
        eng.set_device_calls(device_calls)
    if device_vcf or eng.device_vcf:
        eng.set_device_vcf(device_vcf, qual=qual, show_ref=True)
    t0 = time.time()
    rows_of = {}
    n_cand = 0
    # host seconds per stage of this rank's loop (the GPU works under all of them but `wait`)
    tm = dict(fetch=0.0, ref=0.0, submit=0.0, wait=0.0, decode=0.0)
    call_ms = 0.0                                    # device time of k_call (device_calls)
    vcf_ms = 0.0                                     # device time of the text kernels (device_vcf)
    vcf_d2h = 0                                      # bytes of the text copies: each ticket's bound (device_vcf)
    bam_ms = 0.0                                     # device time of the BAM parse stages (device_bam)

    import threading
    tls = threading.local()
    readers = []
    # reference windows in page-locked buffers: tickets in flight (2) + being decoded (2) + loaded ahead; the pool
    # lives with the engine (page-locking 70 MB costs tens of milliseconds: once per process, not once per run)
    pool = getattr(eng, "_ref_pool", None)
    if pool is None or pool.n_bytes < chunk_size_bytes() or len(pool.ptrs) < 6 + 2 * max(1, loader_threads):
        if pool is not None:
            pool.close()
        pool = eng._ref_pool = PinnedPool(6 + 2 * max(1, loader_threads), chunk_size_bytes())
    # compressed BAM bytes of a chunk (device_bam): tickets in flight (2) + loaded ahead; a larger chunk is read into
    # ordinary memory
    bam_pool = None
    if device_bam:
        bam_pool = getattr(eng, "_bam_pool", None)
        if bam_pool is None or len(bam_pool.ptrs) < 4 + max(1, loader_threads):
            if bam_pool is not None:
                bam_pool.close()
            bam_pool = eng._bam_pool = PinnedPool(4 + max(1, loader_threads), BAM_BUFFER_BYTES)

    def reader():
        # one BAM handle per loader thread (a handle serves one fetch at a time)
        if getattr(tls, "bf", None) is None:
            tls.bf = BamFile(bam_fn, threads=native_threads)
            readers.append(tls.bf)
        return tls.bf

    def load(i):
        name, length, cid, num = shards[i]
        conf = conf_rows.get(name) if conf_rows is not None else None
        known = known_pos.get(name) if known_pos is not None else None
        # the split BED of the contig (run_clair3_rna:231-289): the VCF one is written first, the BED one over it
        ext = regions.extend_bed_rows(conf) if conf is not None else \
            regions.extend_known_rows(known) if known is not None else None
        plan = regions.plan_chunk(length, chunk_id=cid, chunk_num=num, extend_rows=ext, confident_rows=conf,
                                  known_positions=known)
        if plan is None:
            return None
        t = time.time()
        bbuf = None
        if device_bam:
            bbuf = bam_pool.get(0)
            batch = reader().fetch_raw(name, plan.start1, plan.end1, buf=bbuf)
            if batch.data is not bbuf:               # larger than the pool's buffers: read into ordinary memory
                bam_pool.put(bbuf)
                bbuf = None
        else:
            batch = reader().fetch(name, plan.start1, plan.end1)
        tm["fetch"] += time.time() - t
        t = time.time()
        pbuf = pool.get(plan.ref_end1 - plan.ref_start1 + 1)
        if pbuf is not None:
            ref = fasta.fetch_into(ref_fn, fai, name, plan.ref_start1, plan.ref_end1, pbuf)
        else:
            ref = fasta.fetch(ref_fn, fai, name, plan.ref_start1, plan.ref_end1)
        tm["ref"] += time.time() - t
        return name, batch, ref, plan, (pbuf, bbuf)

    # Three host stages run side by side (the native calls release the GIL): a loader thread fetches + inflates the
    # BAM blocks and reads the reference of the shards ahead, this thread submits shard i+1 and waits for shard i,
    # decoder threads turn finished results into VCF rows.  Tickets: one running, one queued, two being decoded.
    from collections import deque
    from concurrent.futures import ThreadPoolExecutor
    # two decoder workers (the two tickets being decoded proceed side by side), each with half of the native threads
    loader, dec = ThreadPoolExecutor(max(1, loader_threads)), ThreadPoolExecutor(2)
    dec_threads = max(1, (native_threads if native_threads > 0 else len(os.sched_getaffinity(0))) // 2)
    tm.update(load_wait=0.0, decode_wait=0.0, release=0.0)
    submit_ms = []
    it = iter(mine)
    loads, decoding = deque(), deque()               # (shard, future) / (shard, ticket, future)

    def prefetch():
        i = next(it, None)
        if i is not None:
            loads.append((i, loader.submit(load, i)))

    def decode(res, pbatch, pref, prs1, pname, pbuf):
        t = time.time()
        if device_vcf:
            rows = device_vcf_rows(res)
        else:
            rows = (format_vcf_rows if device_calls else decode_vcf_rows)(res, pbatch, pref, prs1, pname, qual=qual,
                                                                          threads=dec_threads)
        tm["decode"] += time.time() - t
        pool.put(pbuf[0])                            # the reference window is free again
        return rows

    def retire(block):
        while decoding and (block or decoding[0][2].done()):
            j, tk, f = decoding.popleft()
            t = time.time()
            rows_of[j] = f.result()
            tm["decode_wait"] += time.time() - t
            t = time.time()
            eng.release(tk)
            tm["release"] += time.time() - t
            block = False

    for _ in range(2 + max(1, loader_threads)):
        prefetch()
    pending = None                                   # (shard index, ticket, name, batch, ref, rs1)
    while loads or pending is not None:
        nxt = None
        if loads:
            i, fut = loads.popleft()
            prefetch()
            t = time.time()
            got = fut.result()
            tm["load_wait"] += time.time() - t
            if got is None:                          # genotyping chunk without sites
                rows_of[i] = []
            else:
                name, batch, ref, plan, pbuf = got
                retire(len(decoding) >= 2)           # keep a ticket free for this submit
                t = time.time()
                sub = eng.submit_bam if device_bam else eng.submit
                nxt = (i, sub(batch, ref, plan.ref_start1, plan.start1, plan.end1, plan.site_filter()),
                       name, batch, ref, plan.ref_start1, pbuf)
                tm["submit"] += time.time() - t
                submit_ms.append(1e3 * (time.time() - t))
        if pending is not None:
            j, ticket, pname, pbatch, pref, prs1, ppbuf = pending
            t = time.time()
            res = eng.wait(ticket, copy=False)       # arrays over the library's pinned buffers, no copies
            tm["wait"] += time.time() - t
            n_cand += res.n_cand
            call_ms += res.call_ms
            vcf_ms += res.vcf_ms
            if device_vcf:
                vcf_d2h += res.n_cand * eng.lib.c3r_vcf_row_max(len(pname.encode()))
            if device_bam:                           # the compressed bytes are on the device: the buffer is free
                bam_ms += res.bam_ms
                bam_pool.put(ppbuf[1])
                pbatch = res.reads                   # the records the GPU parsed, valid until release
            decoding.append((j, ticket, dec.submit(decode, res, pbatch, pref, prs1, pname, ppbuf)))
        retire(False)
        pending = nxt
    while decoding:
        retire(True)
    loader.shutdown()
    dec.shutdown()
    if engine is None:
        pool.close()
        eng._ref_pool = None
        if bam_pool is not None:
            bam_pool.close()
            eng._bam_pool = None
        eng.close()
    else:
        if eng.device_calls != calls_before:
            eng.set_device_calls(calls_before)
        if eng._vcf_opts != vcf_before:
            eng.set_device_vcf(vcf_before is not None, *(vcf_before or ()))
    bf.close()
    for r in readers:
        r.close()
    if stats is not None:
        stats.update(shards=len(mine), candidates=n_cand, seconds=time.time() - t0, host_seconds=tm, submit_ms=submit_ms,
                     cost=sum(costs[i] for i in mine), total_shards=len(shards), call_device_ms=call_ms,
                     bam_device_ms=bam_ms, vcf_device_ms=vcf_ms, vcf_d2h_bytes=vcf_d2h)
    if not merge:                                    # the caller only wants this rank's loop (timing passes)
        return None
    if world > 1:
        if gather is None:
            import torch.distributed as dist

            def gather(obj):
                out = [None] * world if rank == 0 else None
                dist.gather_object(obj, out, dst=0)
                return out
        parts = gather(rows_of)
        if rank != 0 or parts is None:
            return None
        rows_of = {}
        for p in parts:
            rows_of.update(p)
    names = [n for n, _ in ctgs]
    redi = sharder.read_rediportal(rediportal_fn, names, rediportal_tags) if rediportal_fn else None
    merged, untagged = sharder.sort_vcf([rows_of[i] for i in range(len(shards))], names, qual=merge_qual,
                                        show_ref=show_ref, rediportal=redi)
    for path, rows in ((output, merged), (output_no_tagging, untagged)):
        if path is None or rows is None:
            continue
        if os.path.exists(path):
            os.remove(path)
        for stale in (path + ".gz", path + ".gz.tbi"):
            if os.path.exists(stale):
                os.remove(stale)
        if not rows:
            # sort_vcf_from always opens output_fn for writing: without a record it leaves an EMPTY file (and its
            # bgzip'ed twin under --compress_vcf) for the steps that follow (sort_vcf.py:123-292)
            open(path, "w").close()
            if compress_vcf:                         # `bgzip -f` of an empty file: the 28-byte BGZF end-of-file block
                with open(path + ".gz", "wb") as fp:
                    fp.write(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))
            continue
        header = decoder.vcf_header([(n, fai[n][0]) for n in fai], sample_name, ref_fn, cmdline=cmdline)
        if compress_vcf:                             # bgzip -f + tabix -p vcf (sort_vcf.py:70-76): path.gz, path.gz.tbi
            from . import vcf_io
            vcf_io.write_vcf_gz(path + ".gz", header, rows)
            continue
        with open(path, "w") as fp:
            fp.write(header + "\n")
            fp.write("\n".join(rows) + "\n")
    return merged


def main(argv=None):
    ap = argparse.ArgumentParser(description="pileup calling of a whole BAM on the GPU(s) of one node")
    ap.add_argument("--bam_fn", required=True)
    ap.add_argument("--ref_fn", required=True)
    ap.add_argument("--chkpnt_fn", required=True)
    ap.add_argument("--output", required=True)
    ap.add_argument("--ctgName", default=None, help="comma separated contigs")
    ap.add_argument("--include_all_ctgs", action="store_true",
                    help="call every contig with mapped reads; default like run_clair3_rna:331-334: chr{1..22,X,Y} and {1..22,X,Y}")
    ap.add_argument("--bed_fn", default=None, help="call only in these regions (BED, plain or gzip)")
    ap.add_argument("--genotyping_mode_vcf_fn", default=None, help="call exactly the sites of this VCF (plain or gzip)")
    ap.add_argument("--sampleName", default="SAMPLE")
    ap.add_argument("--snp_min_af", type=float, default=P.SNP_MIN_AF)
    ap.add_argument("--indel_min_af", type=float, default=P.INDEL_MIN_AF)
    ap.add_argument("--minCoverage", type=int, default=P.MIN_COVERAGE)
    ap.add_argument("--minMQ", type=int, default=P.MIN_MQ)
    ap.add_argument("--platform", default="ont", help="ont* / hifi*: sets the default of --qual like run_clair3_rna:535-539")
    ap.add_argument("--qual", type=int, default=None, help="variants with QUAL <= qual are marked LowQual at the merge")
    ap.add_argument("--print_ref_calls", action="store_true", help="keep reference calls in the merged VCF")
    ap.add_argument("--tag_variant_using_readiportal", action="store_true")
    ap.add_argument("--readiportal_source_fn", default=None, help="REDIportal TABLE1 (plain or gzip)")
    ap.add_argument("--readiportal_database_filter_tag", default="A,D:A,R:A,R,D")
    ap.add_argument("--output_no_tagging_fn", default=None)
    ap.add_argument("--compress_vcf", action="store_true", help="write <output>.gz (BGZF) and <output>.gz.tbi instead of plain text")
    ap.add_argument("--enable_phasing_model", action="store_true")
    ap.add_argument("--enable_padding_in_splice_junction_regions", action="store_true")
    ap.add_argument("--enable_variant_calling_at_sequence_head_and_tail", action="store_true")
    ap.add_argument("--device_calls", action="store_true",
                    help="decide the genotypes on the GPU and only format the rows on the host (same output)")
    ap.add_argument("--device_bam", action="store_true",
                    help="inflate and parse the BAM blocks of each chunk on the GPU (same output)")
    ap.add_argument("--device_vcf", action="store_true",
                    help="decide the genotypes and print the VCF rows on the GPU (same output)")
    a = ap.parse_args(argv)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("gloo")              # only VCF rows travel: no device collective on the data path
    merge_qual = a.qual                              # param_p.py: qual_cut_off 2, min_thred_qual {ont: 8, hifi: 2}
    if merge_qual is None:
        merge_qual = 8 if a.platform.startswith("ont") else 2
    stats = {}
    # run_clair3_rna:364-368: without --ctg_name / --bed_fn / a genotyping VCF only the major contigs are called
    restrict = not (a.include_all_ctgs or a.ctgName or a.bed_fn or a.genotyping_mode_vcf_fn)
    contigs = a.ctgName.split(",") if a.ctgName else (list(sharder.MAJOR_CONTIGS) if restrict else None)
    run(a.bam_fn, a.ref_fn, a.chkpnt_fn, a.output, contigs=contigs, device=local,
        rank=rank, world=world, phased=a.enable_phasing_model, padding=a.enable_padding_in_splice_junction_regions,
        snp_min_af=a.snp_min_af, indel_min_af=a.indel_min_af, min_coverage=a.minCoverage, min_mq=a.minMQ,
        merge_qual=merge_qual, show_ref=a.print_ref_calls,
        rediportal_fn=a.readiportal_source_fn if a.tag_variant_using_readiportal else None,
        rediportal_tags=a.readiportal_database_filter_tag, output_no_tagging=a.output_no_tagging_fn,
        compress_vcf=a.compress_vcf,
        cmdline=" ".join(sys.argv) if argv is None else " ".join(["run_chunks"] + list(argv)),
        sample_name=a.sampleName, stats=stats, bed_fn=a.bed_fn, vcf_fn=a.genotyping_mode_vcf_fn,
        head_tail=a.enable_variant_calling_at_sequence_head_and_tail, device_calls=a.device_calls,
        device_bam=a.device_bam, device_vcf=a.device_vcf)
    print("[rank %d] %d shards, %d candidates in %.2f s" % (rank, stats["shards"], stats["candidates"], stats["seconds"]),
          file=sys.stderr)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
