"""Output writers with the reference's API (TrueConsense/Outputs.py): consensus FASTA, the
VCF-like variant list and the corrected GFF.

Pure host formatting around the GPU path: ``WriteOutputs`` needs the consensus with and without
insertions plus the insertion list (Outputs.py:94-105 runs BuildConsensus twice and ListInserts a
third time); here the count table is ranked once per (mincov, ambiguity) setting by the call kernel
and the insertion columns are piled up once per BAM handle (Events.ListInserts caches them), so
the three passes cost one.  Every quirk of the VCF writer (SURVEY.md Appendix D item 10) is kept:
records are produced from the same comparisons in the same order.
"""
from __future__ import annotations

import sys
from datetime import date

import numpy as np

from .Coverage import GetCoverage
from .Events import ListInserts
from .indexing import Readbam
from .Sequences import BuildConsensus

GFF_COLUMNS = ["seqid", "source", "type", "start", "end", "score", "strand", "phase", "attributes"]


def _first_fasta_record(path):
    """(id, list of residues) of the first record — what Outputs.py:107-113 keeps of SeqIO.parse."""
    rec_id, chunks, seen = None, [], False
    with open(path) as fh:
        for line in fh:
            if line.startswith(">"):
                if seen:
                    break
                seen = True
                words = line[1:].split(None, 1)
                rec_id = words[0] if words else ""
            elif seen:
                chunks.append("".join(line.split()))
    if not seen:
        raise UnboundLocalError("cannot access local variable 'reflist' where it is not associated with a value")
    return rec_id, list("".join(chunks))


def _fasta_records(path):
    """{id: list of residues} of every record, the first of an id winning — _first_fasta_record for each reference."""
    out: dict[str, list] = {}
    rec_id, chunks = None, []

    def close():
        if rec_id is not None and rec_id not in out:
            out[rec_id] = list("".join(chunks))

    with open(path) as fh:
        for line in fh:
            if line.startswith(">"):
                close()
                words = line[1:].split(None, 1)
                rec_id, chunks = (words[0] if words else ""), []
            elif rec_id is not None:
                chunks.append("".join(line.split()))
    close()
    return out


def _gff_line(feature: dict) -> str:
    """One output line for a feature dict (Outputs.py:31-57): the eight fixed columns keep their
    value, everything else — including the parsed ``attributes`` string — is folded into the
    attributes column as key=value pairs (later keys overwrite earlier ones)."""
    fixed = GFF_COLUMNS[:-1]
    cleaned: dict[str, str] = {}
    extra: dict[str, str] = {}
    for key, value in feature.items():
        low = str(key).lower()
        if low in fixed:
            cleaned[low] = str(value)
        else:
            extra[low] = str(value)
    merged: dict[str, str] = {}
    for key, value in extra.items():
        if key != "attributes":
            merged[key] = value
            continue
        for item in value.split(";"):
            if item == "":
                continue
            k, v = item.split("=")           # ValueError for 'a=b=c' or a bare word, like the reference
            merged[k] = v
    cleaned["attributes"] = ";".join(f"{k}={v}" for k, v in merged.items())
    assert list(cleaned.keys()) == GFF_COLUMNS
    return "\t".join(cleaned.values()) + "\n"


def WriteGFF(gffheader, gffdict, output_gff, name):
    """Outputs.py:13-71."""
    with open(output_gff, "w") as out:
        out.write(gffheader.raw_text)
        for feature in gffdict.values():
            out.write(_gff_line(feature))


VCF_HEADER = ("##fileformat=VCFv4.3\n"
              "##fileDate={today}\n"
              "##source='TrueConsense {argv}'\n"
              "##reference='{ref}'\n"
              "##contig=<ID={contig}>\n"
              '##INFO=<ID=DP,Number=1,Type=Integer,Description="Read Depth">\n'
              '##INFO=<ID=INDEL,Number=0,Type=Flag,Description="Indicates that the variant is an INDEL.">\n'
              "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n")


def vcf_header(ref, contigs) -> str:
    """The VCF header with one ``##contig`` line per reference."""
    head = VCF_HEADER.format(today=date.today().strftime("%Y%m%d"), argv=" ".join(sys.argv[1:]), ref=ref, contig="\0")
    return head.replace("##contig=<ID=\0>\n", "".join(f"##contig=<ID={c}>\n" for c in contigs))


def _vcf_records(contig, reference, called, index, mincov, inserts):
    """The reference's variant records (Outputs.py:131-180), one text line at a time and in its order, from the reference
    residues, the upper-cased consensus without insertions and ListInserts' result.  Its coordinate quirks are part of the
    format (SURVEY.md Appendix D item 10) and kept: a deletion is reported on the 0-based index of its first column with the
    base before it; a substitution on index + 1 with the depth of position max(index, 1) + 1; an insertion where the 0-based
    index equals the 1-based insertion position, i.e. one column late."""
    has_inserts, by_position = inserts
    covered_by_deletion = set()
    for i, ref_base in enumerate(reference):
        if i in covered_by_deletion:
            continue
        base = called[i]
        if base != ref_base:
            if base == "-":
                j = i
                deleted = []
                while called[j] == "-":         # (runs off the end like the reference: IndexError on a trailing deletion)
                    deleted.append(reference[j])
                    covered_by_deletion.add(j)
                    j += 1
                yield (f"{contig}\t{i}\t.\t{reference[i - 1] + ''.join(deleted)}\t{called[i - 1]}\t.\tPASS\t"
                       f"DP={GetCoverage(index, i + 1)};INDEL\n")
            else:
                depth_at = (1 if i < 2 else i) + 1
                yield f"{contig}\t{i + 1}\t.\t{ref_base}\t{base}\t.\tPASS\tDP={GetCoverage(index, depth_at)}\n"
        if has_inserts is True and i in by_position:
            depth = GetCoverage(index, i + 1)
            if depth > mincov:
                for inserted in by_position[i].values():
                    yield f"{contig}\t{i}\t.\t{ref_base}\t{called[i]}{inserted}\t.\tPASS\tDP={depth};INDEL\n"


def WriteOutputs(mincov, iDict, uGffDict, inputbam, IncludeAmbig, output_vcf, name, ref, output_gff, gffheader,
                 output_consensus):
    """Outputs.py:74-183: corrected GFF, variant list, consensus FASTA — in that order, each file written as soon as its
    content exists, so a failure part-way leaves what the reference leaves."""
    bam = Readbam(inputbam)
    with_inserts, corrected_gff = BuildConsensus(mincov, iDict, uGffDict, IncludeAmbig, bam, True)
    without_inserts = BuildConsensus(mincov, iDict, uGffDict, IncludeAmbig, bam, False)[0]    # same call table, second walk

    if output_gff is not None:
        WriteGFF(gffheader, corrected_gff, output_gff, name)

    if output_vcf is not None:
        inserts = ListInserts(iDict, mincov, bam)
        contig, reference = _first_fasta_record(ref)
        with open(output_vcf, "w") as out:
            out.write(VCF_HEADER.format(today=date.today().strftime("%Y%m%d"), argv=" ".join(sys.argv[1:]), ref=ref, contig=contig))
            for line in _vcf_records(contig, reference, list(without_inserts.upper()), iDict, mincov, inserts):
                out.write(line)         # streamed: records up to a failure stay in the file

    with open(output_consensus, "w") as out:
        out.write(f">{name} mincov={mincov}\n{with_inserts}\n")
    return None, None


def WriteOutputsContigs(mincov, indexes, gffdicts, inputbam, IncludeAmbig, output_vcf, name, ref, output_gff, gffheader,
                        output_consensus):
    """``WriteOutputs`` for every reference of the BAM (``indexes`` / ``gffdicts``: ``{reference: index dict}`` and
    ``{reference: that reference's GFF rows as a dict}``, header order).  Both walks of every reference are computed first —
    one segmented call table and one insertion pass for all of them — then the files are written in the usual order:
    the GFF header once and each reference's corrected features; one VCF header with a ``##contig`` line per reference
    and each reference's records with CHROM = the reference; one FASTA record ``>{name}_{reference}`` per reference.  An
    exception of any reference aborts the run before a file is written (the VCF writer's own, part-way, as usual); the
    FASTA then does not exist."""
    from . import gpu
    from .Events import ListInsertsContigs, _counts_from_index
    from .Sequences import complement_index, consensus_from_inserts

    bam = Readbam(inputbam)
    names = list(bam.references)
    for n in names:
        complement_index(indexes[n], gffdicts[n], [])
    inserts = ListInsertsContigs(indexes, mincov, bam)
    parts = [_counts_from_index(indexes[n]) for n in names]
    start = np.concatenate(([0], np.cumsum([c.shape[1] for c in parts]))).astype(np.int64)
    table = gpu.default_context().call_contigs(np.concatenate(parts, axis=1), start, mincov, IncludeAmbig is True)
    walks = {}
    for k, n in enumerate(names):
        t = table.slice(int(start[k]), int(start[k + 1]))
        with_inserts, corrected_gff = consensus_from_inserts(mincov, parts[k], gffdicts[n], IncludeAmbig, inserts[n], True, table=t)
        without_inserts = consensus_from_inserts(mincov, parts[k], gffdicts[n], IncludeAmbig, inserts[n], False, table=t)[0]
        walks[n] = (with_inserts, corrected_gff, without_inserts)

    if output_gff is not None:
        with open(output_gff, "w") as out:
            out.write(gffheader.raw_text)
            for n in names:
                for feature in walks[n][1].values():
                    out.write(_gff_line(feature))

    if output_vcf is not None:
        residues = _fasta_records(ref)
        with open(output_vcf, "w") as out:
            out.write(vcf_header(ref, names))
            for n in names:
                for line in _vcf_records(n, residues[n], list(walks[n][2].upper()), indexes[n], mincov, inserts[n]):
                    out.write(line)

    with open(output_consensus, "w") as out:
        for n in names:
            out.write(f">{name}_{n} mincov={mincov}\n{walks[n][0]}\n")
    return None, None
