#!/usr/bin/env python3
"""Non-interactive tag counting: the option surface of the reference's
tagdigger_script.py (/root/reference/tagdigger_script.py:10-35) on the GPU path.

    python -m tagdigger_b200.tagdigger_script -e PstI --MergedTags tags.csv -b key.csv -o counts.csv [-g geno.csv]
    torchrun --nproc-per-node 8 -m tagdigger_b200.tagdigger_script ...      # files dealt to 8 GPUs, one all-reduce
    python -m tagdigger_b200.tagdigger_script -e PstI --MergedTags tags.csv -b key.csv -o counts.csv --adapter PstI-MspI-Hall

With --adapter the key lists the raw library files (File, Barcode, Sample): every file is split by
barcode and trimmed as barcode_splitter_script -a would, and the trimmed reads are counted with a blank
barcode -- the two-stage run in one pass on the GPU, without the split files.

The flow is the reference's (:37-133): resolve the cut site, change directory,
read the tags in exactly one format, sanitise them, read the key file, sniff
every FASTQ file, count, merge by sample name, write the count CSV and the
optional genotype CSV.  The outputs are byte-identical to the reference's.
"""

import argparse
import os
import sys

from . import tagdigger_fun as tdf

TAG_OPTIONS = ("UNEAKtags", "MergedTags", "ColumnTags", "RowTags", "StacksTags", "StacksSnps",
               "StacksAlleles", "TASSELSAM", "pyRADalleles")


def build_parser():
    p = argparse.ArgumentParser(description="TagDigger tag counting on B200 GPUs (options of tagdigger_script.py)")
    p.add_argument("-e", "--enzyme", help="Restriction enzyme name", choices=sorted(tdf.enzymes.keys()))
    p.add_argument("-c", "--cutsite", help="Restriction cut site sequence expected in sequencing reads")
    p.add_argument("-w", "--directory", help="Working directory")
    p.add_argument("--UNEAKtags", help="File name for tags in UNEAK format")
    p.add_argument("--MergedTags", help="File name for tags in merged format")
    p.add_argument("--ColumnTags", help="File name for tags in column format")
    p.add_argument("--RowTags", help="File name for tags in row format.")
    p.add_argument("--StacksTags", help="File name for Stacks tags.tsv file.")
    p.add_argument("--StacksSnps", help="File name for Stacks snps.tsv file.")
    p.add_argument("--StacksAlleles", help="File name for Stacks alleles.tsv file.")
    p.add_argument("--TASSELSAM", help="File name for TASSEL SAM file")
    p.add_argument("--pyRADalleles", help="File name for pyRAD .alleles file.")
    p.add_argument("-k", "--tokeep", help="File name listing tags to keep")
    p.add_argument("--binaryOnly", help="'T' to retain only binary markers; 'F' to retain all markers.",
                   default="F", choices=["T", "F"])
    p.add_argument("--TASSELkeyFile", help="File name to output for key to TASSEL SNP names")
    p.add_argument("-b", "--barcodefile", help="Name of barcode key file", required=True)
    p.add_argument("-o", "--outputcounts", help="Output file name for read counts", required=True)
    p.add_argument("-g", "--outputgen", help="Output file name for numeric genotypes")
    p.add_argument("--adapter", help="Name of an adapter set: split and trim every FASTQ file by barcode as "
                   "barcode_splitter_script -a would (its cut site from the set's enzyme) and count the trimmed reads, "
                   "without writing the split files", choices=sorted(tdf.adapters.keys()))
    return p


def resolve_cutsite(enzyme, cutsite):
    """tagdigger_script.py:37-49."""
    if enzyme is None and cutsite is None:
        raise Exception("Need either restriction enzyme name or cutsite sequence.  "
                        "Use '-e None' if no restriction site is present in reads.")
    if enzyme is not None and cutsite is not None:
        if cutsite.upper() != tdf.enzymes[enzyme]:
            raise Exception("Restriction enzyme name and cutsite do not match.  "
                            "Note that only one of these two arguments is required.")
        return cutsite.upper()
    if enzyme is not None:
        return tdf.enzymes[enzyme]
    site = cutsite.upper()
    if not set(site) <= set("ACGTRYSWKMBDHVN"):
        raise Exception("Cut site contains unexpected characters.")
    return site


def read_tags(args, to_keep):
    """Exactly one tag format (tagdigger_script.py:57-102)."""
    given = {name: getattr(args, name) is not None for name in TAG_OPTIONS}
    stacks = [given["StacksTags"], given["StacksSnps"], given["StacksAlleles"]]
    if any(stacks) and not all(stacks):
        raise Exception("Need all three files for Stacks format.")
    formats = [given["UNEAKtags"], given["MergedTags"], given["ColumnTags"], given["RowTags"],
               given["StacksTags"], given["TASSELSAM"], given["pyRADalleles"]]
    if sum(formats) != 1:
        raise Exception("Exactly one tag format required.")
    binary = args.binaryOnly == "T"
    if given["UNEAKtags"]:
        return tdf.readTags_UNEAK_FASTA(args.UNEAKtags, toKeep=to_keep)
    if given["MergedTags"]:
        return tdf.readTags_Merged(args.MergedTags, toKeep=to_keep)
    if given["ColumnTags"]:
        return tdf.readTags_Columns(args.ColumnTags, toKeep=to_keep)
    if given["RowTags"]:
        return tdf.readTags_Rows(args.RowTags, toKeep=to_keep)
    if given["StacksTags"]:
        return tdf.readTags_Stacks(args.StacksTags, args.StacksSnps, args.StacksAlleles, toKeep=to_keep,
                                   binaryOnly=binary)
    if given["TASSELSAM"]:
        return tdf.readTags_TASSELSAM(args.TASSELSAM, toKeep=to_keep, binaryOnly=binary,
                                      writeMarkerKey=args.TASSELkeyFile is not None,
                                      keyfilename=args.TASSELkeyFile)
    return tdf.readTags_pyRAD(args.pyRADalleles, toKeep=to_keep, binaryOnly=binary)


def main(argv=None):
    args = build_parser().parse_args(argv)
    cutsite = resolve_cutsite(args.enzyme, args.cutsite)
    if args.directory is not None:
        if not os.path.isdir(args.directory):
            raise Exception("Directory {} not found".format(args.directory))
        os.chdir(args.directory)
    to_keep = None
    if args.tokeep is not None:
        to_keep = tdf.readMarkerNames(args.tokeep)
        if to_keep is None:
            raise Exception("Problem reading marker names to keep.")
    tags = read_tags(args, to_keep)
    if tags is None:
        raise Exception("Problem reading tags.")
    tags = tdf.sanitizeTags(tags)
    bckeys = tdf.readBarcodeKeyfile(args.barcodefile)
    if bckeys is None:
        raise Exception("Problem reading barcode file.")
    fqfiles = sorted(bckeys.keys())
    fqok = [tdf.isFastq(f) for f in fqfiles]
    if not all(fqok):
        print("Cannot read the following as FASTQ files:")
        print([f for f, ok in zip(fqfiles, fqok) if not ok])
        raise Exception("Cannot read all FASTQ files.")
    if args.outputgen is not None and set(t[-1] for t in tags[0]) != {"0", "1"}:
        raise Exception("Cannot output numeric genotypes for non-binary markers.")

    # one process per GPU under torchrun; a single process otherwise
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    reduce = gather = None
    if world > 1:
        import torch
        import torch.distributed as dist
        from .counting import dist_gather, engine_reduce, get_engine, init_comm
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl")
        init_comm(get_engine(), rank, world)       # the library's own communicator (tdg_comm_init)
        reduce = engine_reduce                      # one ncclAllReduce on the counting stream
        gather = dist_gather
    samples, counts = tdf.count_files(bckeys, tags[1], cutsite=cutsite, rank=rank, world=world, reduce=reduce,
                                      gather=gather, as_array=True, adapter=args.adapter)
    if rank == 0:
        tdf.writeCounts(args.outputcounts, counts, samples, tags[0])
        if args.outputgen is not None:
            tdf.writeDiploidGeno(args.outputgen, counts, samples, tags[0])
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
