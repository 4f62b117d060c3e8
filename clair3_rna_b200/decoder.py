"""Probabilities + alt_info -> VCF record (host side of the path, A7 in SURVEY.md §8a).

Restates the pileup-mode behaviour of the reference's consumer
(/root/reference/clair3_rna/call_variants.py):

    possible_outcome_probabilites_from   :518-667   (add_indel_length=False branch)
    find_alt_base                        :670-681
    insertion_/deletion_bases_using_alt_info_from   :112-196
    output_from                          :684-1020  (retry loop over outcome families)
    output_with                          :1117-1392 (AD / AF / QUAL / FILTER / row text)
    quality_score_from                   :383-389

with the options `call_var_bam` always passes: --pileup --showRef, --add_indel_length
False, --qual 2 (clair3_rna/call_var_bam.py:247-272).  Products of probabilities are
float32 like the reference's numpy scalars; QUAL is computed in float64 from the float32
product (NumPy-1 promotion, SURVEY.md §8c).
"""
from __future__ import annotations

import math

import numpy as np

from . import params as P

ACGT = "ACGT"
GT21 = {lab: i for i, lab in enumerate(P.GT21_LABELS)}
HOMO_SNP = ("AA", "CC", "GG", "TT")
HETERO_SNP = ("AC", "AG", "AT", "CG", "CT", "GT")
BASE2ACGT = dict(zip("ACGTURYSWKMBDHVN", "ACGTTACCAGACAAAA"))       # shared/utils.py:41-44
PHRED_TRANS = -10 * math.log(math.e, 10)                             # call_variants.py:58
MAX_INDEL = P.MAX_VARIANT_LENGTH


def parse_alt_info(alt_info: str):
    """'12-XT 3 IAG 2 RA 7' -> (12, [('XT',3), ('IAG',2), ('RA',7)])   (call_variants.py:1150-1154)"""
    parts = alt_info.rstrip().split('-')
    depth = int(parts[0])
    toks = (parts[1] if len(parts) > 1 else '').split(' ')
    items = {}
    for k, v in zip(toks[::2], toks[1::2]):
        items[k] = int(v)
    return depth, items


def _snp_alts(alt: dict, want=None):
    """find_alt_base: X alleles by descending count (stable); falls back to the best supported
    base when `want` is absent or trails it by >= 9 reads."""
    ranked = sorted(((k[1], c) for k, c in alt.items() if k[0] == 'X'), key=lambda kv: kv[1], reverse=True)
    if not ranked:
        return [], None
    mine = [c for b, c in ranked if b == want]
    if not mine or ranked[0][1] - mine[0] >= 9:
        want = ranked[0][0]
    return [b for b, _ in ranked], want


def _indel_keys(alt: dict, kind: str):
    return {k[1:]: c for k, c in alt.items() if k[0] == kind and 1 <= len(k) - 1 <= MAX_INDEL}


def _best_indel(alt: dict, kind: str) -> str:
    d = _indel_keys(alt, kind)
    return max(d, key=d.get) if d else ""


def _two_indels(alt: dict, kind: str):
    d = _indel_keys(alt, kind)
    ranked = [k for k, _ in sorted(d.items(), key=lambda kv: kv[1])][::-1]
    if kind == 'I':
        return ranked[:2]
    if len(ranked) <= 1:
        return []
    a, b = ranked[0], ranked[1]
    return [a, b] if len(a) > len(b) else [b, a]


FAMILIES = ("ref", "homo_snp", "het_snp", "homo_ins", "het_acgt_ins", "het_insins",
            "homo_del", "het_acgt_del", "het_deldel", "insdel")


def decide(ref33: str, probs, alt: dict):
    """output_from: -> (flags dict, reference_base, alternate_base, probability)"""
    center = ref33[P.FLANK] if len(ref33) > 1 else ref33[0]
    ref_acgt = BASE2ACGT[center]
    gt21 = np.asarray(probs[:21], dtype=np.float32)
    gen = np.asarray(probs[21:24], dtype=np.float32)
    p00, p11, p01 = gen[0], gen[1], gen[2]
    rr = gt21[GT21[ref_acgt + ref_acgt]]
    p_ref = p00 * rr
    flags = dict.fromkeys(FAMILIES, False)
    if p00 >= 0.5 and rr >= 0.5:
        flags["ref"] = True
        return flags, ref_acgt, ref_acgt, p_ref
    fam = {
        "homo_snp": [p11 * gt21[GT21[l]] for l in HOMO_SNP],
        "het_snp": [p01 * gt21[GT21[l]] for l in HETERO_SNP],
        "homo_ins": [p11 * gt21[GT21["InsIns"]]],
        "het_insins": [p01 * gt21[GT21["InsIns"]]],
        "het_acgt_ins": [gt21[GT21[b + "Ins"]] * p01 for b in ACGT],
        "homo_del": [p11 * gt21[GT21["DelDel"]]],
        "het_deldel": [p01 * gt21[GT21["DelDel"]]],
        "het_acgt_del": [gt21[GT21[b + "Del"]] * p01 for b in ACGT],
        "insdel": [p01 * gt21[GT21["InsDel"]]],
    }
    ref_base = alt_base = None
    best = 0.0
    # A failed family zeroes its probability and `continue`s WITHOUT clearing ref_base/alt_base,
    # exactly like the reference: the loop ends as soon as both happen to be set.
    while ref_base is None or alt_base is None:
        best = max([p_ref] + [max(v) for v in fam.values()])
        if best == p_ref:
            flags = dict.fromkeys(FAMILIES, False)
            flags["ref"] = True
            return flags, ref_acgt, ref_acgt, best
        flags = {k: (best in v) for k, v in fam.items()}
        flags["ref"] = False
        if flags["homo_snp"]:
            v = fam["homo_snp"]
            ref_base = center
            i = v.index(best)
            lab = HOMO_SNP[int(np.argmax(v))]
            _, alt_base = _snp_alts(alt, lab[0] if lab[0] != ref_base else lab[1])
            if alt_base is None or alt_base == ref_base:
                v[i] = 0
                continue
        elif flags["het_snp"]:
            v = fam["het_snp"]
            lab = HETERO_SNP[int(np.argmax(v))]
            i = v.index(best)
            ref_base = center
            if lab[0] != ref_base and lab[1] != ref_base:
                ranked, _ = _snp_alts(alt)
                if len(ranked) < 2:
                    v[i] = 0
                    continue
                alt_base = ','.join(ranked[:2])
            else:
                _, alt_base = _snp_alts(alt, lab[0] if lab[0] != ref_base else lab[1])
                if alt_base is None or alt_base == ref_base:
                    v[i] = 0
                    continue
        elif flags["homo_ins"]:
            v = fam["homo_ins"]
            i = v.index(best)
            ins = _best_indel(alt, 'I')
            if not ins:
                v[i] = 0
                continue
            ref_base, alt_base = center, ins
        elif flags["het_acgt_ins"]:
            v = fam["het_acgt_ins"]
            i = v.index(best)
            ins = _best_indel(alt, 'I')
            if not ins:
                v[i] = 0
                continue
            ref_base, alt_base = center, ins
            if ACGT[i] != ref_base:
                ranked, _ = _snp_alts(alt)
                if not ranked:
                    v[i] = 0
                    continue
                alt_base = "%s,%s" % (ranked[0], alt_base)
        elif flags["het_insins"]:
            v = fam["het_insins"]
            i = v.index(best)
            two = _two_indels(alt, 'I')
            if len(two) < 2:
                v[i] = 0
                continue
            ref_base, alt_base = center, two[0]
            if two[1] != two[0]:
                alt_base = "%s,%s" % (two[1], two[0])
            else:
                v[i] = 0
                continue
        elif flags["homo_del"]:
            v = fam["homo_del"]
            i = v.index(best)
            dele = _best_indel(alt, 'D')
            if not dele:
                v[i] = 0
                continue
            ref_base = center + dele
            alt_base = ref_base[0]
        elif flags["het_acgt_del"]:
            v = fam["het_acgt_del"]
            i = v.index(best)
            dele = _best_indel(alt, 'D')
            if not dele:
                v[i] = 0
                continue
            ref_base = center + dele
            alt_base = ref_base[0]
            if ACGT[i] != ref_base[0]:
                alt_base = "%s,%s" % (alt_base, ACGT[i] + ref_base[1:])
        elif flags["het_deldel"]:
            v = fam["het_deldel"]
            i = v.index(best)
            two = _two_indels(alt, 'D')
            if len(two) < 2:
                v[i] = 0
                continue
            longer, other = two
            ref_base = center + longer
            alt_base = ref_base[0]
            a1, a2 = alt_base, ref_base[0] + ref_base[len(other) + 1:]
            if a1 != a2 and ref_base != a1 and ref_base != a2:
                alt_base = "%s,%s" % (a1, a2)
            else:
                v[i] = 0
                continue
        elif flags["insdel"]:
            v = fam["insdel"]
            i = v.index(best)
            ins, dele = _best_indel(alt, 'I'), _best_indel(alt, 'D')
            if not ins or not dele:
                v[i] = 0
                continue
            ref_base = center + dele
            alt_base = "%s,%s" % (ref_base[0], ins + ref_base[1:])
    return flags, ref_base, alt_base, best


def quality_score(p) -> float:
    p = float(p)
    return float(round(max(PHRED_TRANS * math.log(((1.0 - p) + 1e-10) / (p + 1e-10)) + 10, 0), 2))


def _iupac_to_n(s: str) -> str:
    if s == ".":
        return s
    return ''.join(c if c.upper() in "ACGTN,." else 'N' for c in s)


def vcf_row(contig: str, pos: int, ref33: str, alt_info: str, probs, qual_for_pass=P.QUAL_CUT_OFF, show_ref=True):
    """output_with: one VCF data line, or None when the reference prints nothing."""
    depth, alt = parse_alt_info(alt_info)
    return vcf_row_from(contig, pos, ref33, depth, alt, probs, qual_for_pass, show_ref)


def vcf_row_from(contig: str, pos: int, ref33: str, depth: int, alt: dict, probs, qual_for_pass=P.QUAL_CUT_OFF,
                 show_ref=True):
    """vcf_row on the parsed alt_info: depth and the {key: count} dict"""
    f, ref_base, alt_base, prob = decide(ref33, probs, alt)
    is_ref = f["ref"]
    if (not show_ref and is_ref) or (not is_ref and ref_base == alt_base):
        return None
    if ref_base is None or alt_base is None:
        return None
    multi = ',' in str(alt_base)
    gt = None
    if is_ref:
        gt = "0/0"
    elif f["homo_snp"] or f["homo_ins"] or f["homo_del"]:
        gt = "1/1"
    elif f["het_snp"] or f["het_acgt_ins"] or f["het_insins"] or f["het_acgt_del"] or f["het_deldel"]:
        gt = "0/1"
    if multi:
        gt = "1/2"
    snp = {k[1]: c for k, c in alt.items() if k[0] == 'X'}
    ins = {k[1:]: c for k, c in alt.items() if k[0] == 'I'}
    dele = {k[1:]: c for k, c in alt.items() if k[0] == 'D'}
    ref_count = 0
    for k, c in alt.items():
        if k[0] == 'R':
            ref_count = c
    ref_count = max(0, ref_count)
    support, counts = 0, []
    if is_ref:
        support = ref_count
        alt_base = "."
    elif f["homo_snp"] or f["het_snp"]:
        for b in str(alt_base):
            if b == ',':
                continue
            support += snp.get(b, 0)
            counts.append(support)                   # cumulative, as the reference does
    elif f["homo_ins"] or f["het_insins"]:
        for s in alt_base.split(','):
            c = ins.get(s, 0)
            support += c
            counts.append(c)
    elif f["het_acgt_ins"]:
        snp_b = alt_base.split(",")[0][0] if multi else None
        ins_b = alt_base.split(",")[1] if multi else alt_base
        c_snp = snp.get(snp_b, 0) if multi else 0
        c_ins = ins.get(ins_b, 0)
        support = c_ins + c_snp
        if snp_b:
            counts.append(c_snp)
        counts.append(c_ins)
    elif f["homo_del"] or f["het_deldel"]:
        if dele:
            if f["homo_del"]:
                db = ref_base[1:] if len(ref_base) > 1 else None
                support = dele.get(db, 0)
                counts.append(support)
            elif f["het_deldel"] and len(dele) > 1:
                for s in alt_base.split(','):
                    ln = len(ref_base) - len(s)
                    hit = [c for k, c in dele.items() if len(k) == ln]
                    c = hit[0] if hit else 0
                    counts.append(c)
                    support += c
    elif f["het_acgt_del"]:
        parts = alt_base.split(",")
        snp_b = (parts[1][0] if len(parts) > 1 else None) if multi else None
        c_snp = snp.get(snp_b, 0) if multi else 0
        db = ref_base[1:] if len(ref_base) > 1 else None
        c_del = dele.get(db, 0)
        support = c_del + c_snp
        if snp_b:
            counts.append(c_snp)
        counts.append(c_del)
    elif f["insdel"]:
        for s in alt_base.split(','):
            ln = len(ref_base) - len(s)
            if ln < 0:
                ib = s[:-(len(ref_base) - 1)] if len(ref_base) > 1 else s
                c = ins.get(ib, 0)
            else:
                hit = [c2 for k, c2 in dele.items() if len(k) == ln]
                c = hit[0] if hit else 0
            counts.append(c)
            support += c
    af = (support + 0.0) / depth if depth != 0 else 0.0
    if af > 1:
        af = 1
    qual = quality_score(prob)
    filt = "RefCall" if is_ref else ("PASS" if qual_for_pass is None or qual >= qual_for_pass else "LowQual")
    ref_base = _iupac_to_n(ref_base)
    alt_base = _iupac_to_n(alt_base)
    ad = str(ref_count) + ((',' + ','.join(str(c) for c in counts)) if counts else "")
    afs = "%.4f" % af if len(counts) <= 1 else ','.join("%.4f" % min(1.0, 1.0 * c / depth) for c in counts)
    return "%s\t%d\t.\t%s\t%s\t%.2f\t%s\t%s\tGT:GQ:DP:AD:AF\t%s:%d:%d:%s:%s" % (
        contig, pos, ref_base, alt_base, qual, filt, ".", gt, qual, depth, ad, afs)


def vcf_header(fai_rows, sample_name="SAMPLE", reference_path=None, cmdline=None) -> str:
    """get_header (shared/utils.py:261-316); fai_rows = [(contig, length)]."""
    lines = ["##fileformat=VCFv4.2", "##source=Clair3-RNA", "##clair3_rna_version=%s" % P.VERSION,
             '##FILTER=<ID=PASS,Description="All filters passed">',
             '##FILTER=<ID=LowQual,Description="Low quality variant">',
             '##FILTER=<ID=RefCall,Description="Reference call">',
             '##FILTER=<ID=RNAEditing,Description="RNA editing site tagged by REDIportal dataset">',
             '##INFO=<ID=A,Number=0,Type=Flag,Description="RNA editing site from ATLAS dataset in REDIportal">',
             '##INFO=<ID=R,Number=0,Type=Flag,Description="RNA editing site from RADAR dataset in REDIportal">',
             '##INFO=<ID=D,Number=0,Type=Flag,Description="RNA editing site from DARNED dataset in REDIportal">',
             '##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">',
             '##FORMAT=<ID=GQ,Number=1,Type=Integer,Description="Genotype Quality">',
             '##FORMAT=<ID=DP,Number=1,Type=Integer,Description="Approximate read depth (reads with MQ<5 or selected by \'samtools view -F 2316\' are filtered)">',
             '##FORMAT=<ID=AD,Number=R,Type=Integer,Description="Allelic depths for the ref and alt alleles in the order listed">',
             '##FORMAT=<ID=AF,Number=1,Type=Float,Description="Observed allele frequency in reads, for each ALT allele, in the same order as listed, or the REF allele for a RefCall">']
    if reference_path:
        lines.insert(3, "##reference=%s" % reference_path)
    if cmdline:
        lines.insert(3, "##cmdline=%s" % cmdline)
    for name, length in fai_rows:
        lines.append("##contig=<ID=%s,length=%s>" % (name, length))
    return "\n".join(lines) + "\n" + "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t%s" % sample_name
