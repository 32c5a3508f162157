#!/usr/bin/env python3
"""Non-interactive barcode splitting: the options of the reference's
barcode_splitter_script.py (/root/reference/barcode_splitter_script.py:8-36).

    python -m tagdigger_b200.barcode_splitter_script -b key.csv -a PstI-MspI-Hall
    torchrun --nproc_per_node=8 -m tagdigger_b200.barcode_splitter_script -b key.csv -a PstI-MspI-Hall

The key file has the columns Input File, Barcode, Output File; the enzyme (and with it
the cut site) is the first part of the adapter-set name.  Under torchrun the input files are
shared out among the GPUs, and one large library file is split by all of them together; the output
files are those of a single process.
"""

import argparse
import os
import sys

from . import hostio, splitter


def build_parser():
    p = argparse.ArgumentParser(description="TagDigger barcode splitter on B200 GPUs (options of barcode_splitter_script.py)")
    p.add_argument("-b", "--barcodefile", help="Name of barcode key file", required=True)
    p.add_argument("-a", "--adapter", help="Name of the adapter set", required=True,
                   choices=sorted(hostio.adapters.keys()))
    p.add_argument("--bgzf", action="store_true",
                   help="Write the output files BGZF-compressed (bgzip's format; their names must end in 'gz')")
    return p


def main(argv=None):
    args = build_parser().parse_args(argv)
    bckeys = hostio.readBarcodeKeyfile(args.barcodefile, forSplitter=True)
    if bckeys is None:
        raise Exception("Problem reading barcode file.")
    adapter = hostio.adapters[args.adapter]
    cutsite = hostio.enzymes[args.adapter[:args.adapter.find("-")]]
    fqfiles = sorted(bckeys.keys())
    fqok = [hostio.isFastq(f) for f in fqfiles]
    if not all(fqok):
        print("Cannot read the following as FASTQ files:")
        print([f for f, ok in zip(fqfiles, fqok) if not ok])
        raise Exception("Cannot read all FASTQ files.")
    # one process per GPU under torchrun; a single process otherwise
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    gather = None
    if world > 1:
        import torch
        import torch.distributed as dist
        from .counting import dist_gather
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("gloo")            # only small host lists are exchanged
        gather = dist_gather
    try:
        splitter.split_files(bckeys, cutsite, adapter, bgzf=args.bgzf, rank=rank, world=world, gather=gather)
    finally:
        if world > 1:
            dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
