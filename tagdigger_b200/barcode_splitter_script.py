#!/usr/bin/env python3
"""Non-interactive barcode splitting: the options of the reference's
barcode_splitter_script.py (/root/reference/barcode_splitter_script.py:8-36).

    python -m tagdigger_b200.barcode_splitter_script -b key.csv -a PstI-MspI-Hall

The key file has the columns Input File, Barcode, Output File; the enzyme (and with it
the cut site) is the first part of the adapter-set name.
"""

import argparse
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
    for f in fqfiles:
        splitter.barcodeSplitter(f, bckeys[f][0], bckeys[f][1], cutsite=cutsite, adapter=adapter, bgzf=args.bgzf)
    return 0


if __name__ == "__main__":
    sys.exit(main())
