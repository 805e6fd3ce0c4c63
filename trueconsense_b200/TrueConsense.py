"""Command line with the reference's surface (TrueConsense/TrueConsense.py): same flags, same
validators and exit behaviour, same order of work — on top of the GPU hot path.

    python -m trueconsense_b200.TrueConsense -i x.bam -ref ref.fasta -gff f.gff -cov 30 -name S -o cons.fasta
    python -m trueconsense_b200.TrueConsense --all-contigs -i flu.bam -ref flu.fasta -gff flu.gff -cov 30 -name S -o S.fasta
    python -m trueconsense_b200.TrueConsense --sort-input -i aligner_out.bam -ref ref.fasta -gff f.gff -cov 30 -name S -o S.fasta

    minimap2 -a ref.fa r.fq > s.sam
    python -m trueconsense_b200.TrueConsense --sort-input -i s.sam -ref ref.fa -gff f.gff -cov 30 -name S -o S.fasta
    python -m trueconsense_b200.TrueConsense --primers scheme.primer.bed --primer-both-ends -i s.sam -ref ref.fa -gff f.gff \
        -cov 30 -name S -o S.fasta

``main(args)`` is the console-script entry point of the reference (pyproject.toml:38-40).
"""
from __future__ import annotations

import argparse
import concurrent.futures as cf
import multiprocessing
import os
import pathlib
import sys

from .Coverage import BuildCoverage, BuildCoverageContigs
from .func import MyHelpFormatter, color
from .indexing import (BuildIndex, BuildIndexContigs, Gffindex, Override_index_positions, Readbam, gff_by_contig,
                       read_override_index)
from .Outputs import WriteOutputs, WriteOutputsContigs
from .primers import read_bed
from .version import __version__


def _not_a_file(fname, code):
    print(f'"{fname}" is not a file. Exiting...')
    sys.exit(code)


def GetArgs(givenargs):
    """TrueConsense.py:25-209.  Validators: a missing file exits (-1 for the BAM, 1 otherwise), a
    wrong extension is an argparse error."""
    parser = argparse.ArgumentParser(
        prog="TrueConsense",
        usage="%(prog)s [required options] [optional arguments]",
        description="TrueConsense: Creating biologically valid consensus sequences from reference-based alignments",
        formatter_class=MyHelpFormatter,
        add_help=False,
    )

    def with_suffix(kind, allowed, exit_code, label):
        def check(fname):
            if not os.path.isfile(fname):
                _not_a_file(fname, exit_code)
            if pathlib.Path(fname).suffix not in allowed:
                parser.error(f"{label} {color.YELLOW}({fname}){color.END} doesn't seem to be a {kind}.")
            return fname
        return check

    def check_index_override(fname):
        if not os.path.isfile(fname):
            _not_a_file(fname, 1)
        ext = "".join(pathlib.Path(fname).suffixes)
        if ".csv" not in ext or ".gz" not in ext:
            parser.error(f"Given file {color.YELLOW}({fname}){color.END} doesn't seem to be a compressed csv file.")
        return fname

    req = parser.add_argument_group("Required arguments")
    req.add_argument("--input", "-i", type=with_suffix("BAM or SAM file", (".bam", ".sam"), -1, "Input file"), metavar="File",
                     help="Input file in BAM or SAM format (SAM: the aligner's text output, converted on the GPU)", required=True)
    req.add_argument("--output", "-o", type=str, default=os.getcwd() + "consensus.fasta", metavar="File",
                     help="Output consensus fasta", required=True)
    req.add_argument("--reference", "-ref", type=with_suffix("Fasta-file", (".fasta", ".fa"), 1, "Reference file"),
                     metavar="File", help="Reference Fasta file", required=True)
    req.add_argument("--features", "-gff", type=with_suffix("GFF file", (".gff",), 1, "Given file"), metavar="File",
                     help="File with genome features (GFF)", required=True)
    req.add_argument("--coverage-level", "-cov", type=int, default=30, metavar="100",
                     help="The minimum coverage level of the consensus and variant calls", required=True)
    req.add_argument("--samplename", "-name", metavar="Text",
                     help="Name of the sample that is being processed, will be used to create the fasta header", required=True)

    opt = parser.add_argument_group("Optional arguments")
    opt.add_argument("--variants", "-vcf", type=str, metavar="File", help="Output VCF file")
    opt.add_argument("--depth-of-coverage", "-doc", type=str, metavar="File",
                     help="Output TSV file listing the coverage per position")
    opt.add_argument("--output-gff", "-ogff", type=str, metavar="File", help="Ouput location a corrected GFF file")
    opt.add_argument("--threads", "-t", default=min(multiprocessing.cpu_count(), 128), metavar="N", type=int,
                     help="Number of threads that can be used by TrueConsense")
    opt.add_argument("--noambiguity", "-noambig", action="store_true",
                     help="Turn off ambiguity nucleotides in the generated consensus sequence")
    opt.add_argument("--index-override", type=check_index_override, metavar="File",
                     help="Override the positional index of certain genome positions with 'known' information if the given "
                          "alignment is not sufficient for these positions\nMust be a compressed csv.\nPlease use with caution "
                          "as this will overwrite the generated index at the given positions!\n")
    opt.add_argument("--all-contigs", action="store_true",
                     help="Call every reference of a multi-contig BAM (a segmented genome, a panel of references) in one "
                          "pass: one FASTA record '{samplename}_{reference}' per reference, the GFF rows matched by seqid, "
                          "one VCF and one depth file for all references")
    opt.add_argument("--sort-input", action="store_true",
                     help="Accept a BAM or SAM whose records are not coordinate-sorted (e.g. straight from the aligner); they "
                          "are put in samtools' coordinate order on the GPU. A sorted file is used as written")
    opt.add_argument("--primers", type=with_suffix("BED file", (".bed",), 1, "Primer file"), metavar="File",
                     help="Amplicon primer scheme (BED: chrom, 0-based start, end). The primers are soft-clipped off the "
                          "aligned reads on the GPU, as samtools ampliconclip --soft-clip does; implies --sort-input")
    opt.add_argument("--primer-tolerance", type=int, default=None, metavar="N",
                     help="Bases a read end may lie in front of a primer's start or behind its end and still match it "
                          "(default 5; needs --primers)")
    opt.add_argument("--primer-both-ends", action="store_true",
                     help="Clip primers at both ends of every read (nanopore reads span the whole amplicon), not only at "
                          "the 5' end (needs --primers)")
    opt.add_argument("--version", "-v", action="version", version=__version__,
                     help="Show the TrueConsense version and exit")
    opt.add_argument("--help", "-h", action="help", default=argparse.SUPPRESS, help="Show this help message and exit")
    opts = parser.parse_args(givenargs)
    if opts.all_contigs and opts.index_override:
        parser.error("--index-override cannot be combined with --all-contigs: its positions name no reference")
    if opts.primers is None and (opts.primer_tolerance is not None or opts.primer_both_ends):
        parser.error("--primer-tolerance and --primer-both-ends need --primers")
    if opts.primer_tolerance is None:
        opts.primer_tolerance = 5
    elif opts.primer_tolerance < 0:
        parser.error("--primer-tolerance must be 0 or more")
    return opts


def _index_and_features(opts, bam):
    """The count table and the GFF, read side by side like TrueConsense.py:225-230 (BuildIndex runs on a pool thread: the
    C-ABI sets its device per call), then the optional override of single positions (:232-235)."""
    with cf.ThreadPoolExecutor(max_workers=opts.threads) as pool:
        jobs = (pool.submit(BuildIndex, bam, opts.reference), pool.submit(Gffindex, opts.features))
        frame, gff = (j.result() for j in jobs)
    if opts.index_override:
        frame = Override_index_positions(frame, read_override_index(opts.index_override))
    return frame, gff


def _main_all_contigs(opts, bam):
    """--all-contigs: every reference of the BAM header through one device pass, the outputs assembled per reference."""
    with cf.ThreadPoolExecutor(max_workers=opts.threads) as pool:
        jobs = (pool.submit(BuildIndexContigs, bam, opts.reference), pool.submit(Gffindex, opts.features))
        frames, gff = (j.result() for j in jobs)
    indexes = {n: f.to_dict("index") for n, f in frames.items()}
    gffdicts = {}
    for n, rows in gff_by_contig(gff.df, list(frames)).items():
        rows["seqid"] = f"{opts.samplename}_{n}"
        gffdicts[n] = rows.to_dict("index")
    if opts.depth_of_coverage is not None:
        with cf.ThreadPoolExecutor(max_workers=opts.threads) as pool:
            pool.submit(BuildCoverageContigs, indexes, opts.depth_of_coverage)
    WriteOutputsContigs(opts.coverage_level, indexes, gffdicts, bam, opts.noambiguity is False, opts.variants, opts.samplename,
                        opts.reference, opts.output_gff, gff.header, opts.output)


def main(args: list[str] | None = None):
    """The reference's command line (TrueConsense.py:212-264): same flags, same files."""
    argv = args or sys.argv[1:]
    if not argv:
        print("TrueConsense was called but no arguments were given, please try again.\n"
              "Use 'TrueConsense -h' to see the help document")
        sys.exit(1)
    opts = GetArgs(argv)
    primers = None if opts.primers is None else read_bed(opts.primers, opts.primer_tolerance, opts.primer_both_ends)
    # one decoded copy of the BAM serves the index and the insertion columns
    bam = Readbam(opts.input, sort=opts.sort_input, primers=primers)
    if opts.all_contigs:
        return _main_all_contigs(opts, bam)
    frame, gff = _index_and_features(opts, bam)
    index = frame.to_dict("index")
    features = gff.df
    features["seqid"] = opts.samplename
    if opts.depth_of_coverage is not None:
        # fire and forget on a pool thread, its outcome never looked at (:243-245)
        with cf.ThreadPoolExecutor(max_workers=opts.threads) as pool:
            pool.submit(BuildCoverage, index, opts.depth_of_coverage)
    WriteOutputs(opts.coverage_level, index, features.to_dict("index"), bam, opts.noambiguity is False, opts.variants,
                 opts.samplename, opts.reference, opts.output_gff, gff.header, opts.output)


if __name__ == "__main__":
    main()
