"""CROPSR.py-compatible command line (/root/reference/CROPSR.py:24-51, :333-336)."""
import argparse
import sys

__version__ = "1.11b-b200"


def build_parser():
    # the usage line is spelled out: with the reference's empty metavars argparse cannot wrap a usage
    # line of this length (its own consistency assertion fails), and --help would crash
    p = argparse.ArgumentParser(prog="CROPSR.py", usage="CROPSR.py [-h] -f FASTA [-g GFF] [-p TXT] [-o CSV] [-l 20] [-L 200] --cas9 [-v]\n"
                                "                 [--device N | --devices 0-7] [--side-output TSV] [--offtargets TSV] [--offtarget-sites TSV]\n"
                                "                 [--offtarget-scores TSV] [--offtarget-pams NAG,NGA] [--mismatches K] [--max-sites N]\n"
                                "                 [--blas-threads N]")
    p.add_argument("-f", "--fasta", metavar="", required=True, dest="f",
                   help="[required] path to input file in FASTA format")
    p.add_argument("-g", "--gff", metavar="", dest="g", help="path to input file in GFF format")
    p.add_argument("-p", "--phytozome", metavar="", dest="p", default=None,
                   help="path to input annotation info file in TXT format, default = None")
    p.add_argument("-o", "--output", metavar="", dest="o", default="data.csv",
                   help="path to output file, default = data.csv")
    p.add_argument("-l", "--length", metavar="", dest="l", type=int, default=20,
                   help="length of the gRNA sequence, default = 20")
    p.add_argument("-L", "--flanking", metavar="", dest="L", type=int, default=200,
                   help="length of flanking region for verification, default = 200")
    p.add_argument("--cas9", action="store_true",
                   help="specifies that design will be made for the Cas9 CRISPR system")
    p.add_argument("-v", "--verbose", action="store_true",
                   help="prints visual indicators for each iteration")
    # additions (defaults reproduce the reference)
    p.add_argument("--device", type=int, default=0, help="CUDA device ordinal, default = 0")
    p.add_argument("--devices", metavar="", default=None,
                   help="several CUDA devices, e.g. 0-7 or 0,2,4: the genome is cut into one contiguous shard per "
                        "device (one process each), candidate counts are exchanged by one NCCL all-gather and the "
                        "CSV is written in the same order as on one device")
    p.add_argument("--side-output", metavar="", default=None,
                   help="also write a tab-separated table of opt-in per-candidate side outputs (GC, poly-T, "
                        "homopolymer, +-L flank window, GFF feature under the cut site); the CSV is unaffected")
    p.add_argument("--offtargets", metavar="", default=None,
                   help="also write a tab-separated table of off-target counts: per candidate its protospacer and the "
                        "number of other NGG sites of the genome (both strands, any case) at exactly 0 .. K mismatches; "
                        "-l 20 on one GPU only; the CSV is unaffected")
    p.add_argument("--offtarget-sites", metavar="", default=None,
                   help="also write a tab-separated table of off-target sites: one row per candidate and other NGG site "
                        "of the genome within K mismatches, with the site's chromosome, strand, position and protospacer "
                        "(differing bases in lower case); candidates with more than --max-sites such sites are left out "
                        "(their counts are in --offtargets); -l 20 on one GPU only; the CSV is unaffected")
    p.add_argument("--offtarget-scores", metavar="", default=None,
                   help="also write a tab-separated table of off-target scores: per candidate its protospacer, the sum "
                        "of the MIT hit scores (Hsu et al. 2013, as CRISPOR computes them) of the other NGG sites of the "
                        "genome within K mismatches, and the MIT specificity 100 / (100 + sum) * 100; CRISPOR also "
                        "counts 4-mismatch sites, and NAG/NGA sites unless --offtarget-pams NAG,NGA is given, so its "
                        "numbers differ; -l 20 on one GPU only; the CSV is unaffected")
    p.add_argument("--offtarget-pams", metavar="", default=None,
                   help="PAM patterns whose sites the off-target tables also read, besides NGG, e.g. NAG,NGA: N and "
                        "two IUPAC letters (ACGTRYSWKMBDHV), disjoint from NGG and from each other.  --offtargets "
                        "gains PAM_mm0 .. PAM_mmK per pattern, --offtarget-sites a site_pam column (the cap counts "
                        "every pattern), --offtarget-scores PAM_mit_hit_sum per pattern and all_mit_specificity over "
                        "all of them")
    p.add_argument("--mismatches", metavar="", type=int, default=3,
                   help="K of --offtargets, --offtarget-sites and --offtarget-scores: 0 to 3, default = 3")
    p.add_argument("--max-sites", metavar="", type=int, default=1000,
                   help="--offtarget-sites lists the candidates with at most this many other sites within K "
                        "mismatches: at least 1, default = 1000")
    p.add_argument("--blas-threads", type=int, default=1,
                   help="emulate the float summation order of the reference running with this many "
                        "OpenBLAS threads (default 1 = OPENBLAS_NUM_THREADS=1)")
    return p


def banner(args):
    from multiprocessing import cpu_count
    return f"""
        CROPSR (B200) -- genome-wide CRISPR gRNA candidate scan

        You are currently utilizing the following settings:

        CROPSR version:                                 {__version__}
        Path to genome file in FASTA format:            {args.f}
        Path to output file:                            {args.o}
        Length of the gRNA sequence:                    {args.l}
        Length of flanking region for verification:     {args.L}
        Number of available CPUs:                       {cpu_count()}
        Path to annotation file in GFF format:          {args.g}
        Path to annotation_info file in TXT format:     {args.p}
        Designing for CRISPR system:
            Streptococcus pyogenes Cas9                 {args.cas9}
        """


def parse_devices(text):
    """'0-3' / '0,2,5' / '1' -> [ordinals]"""
    out = []
    for part in text.split(","):
        a, _, b = part.strip().partition("-")
        out += list(range(int(a), int(b or a) + 1))
    if not out or len(set(out)) != len(out):
        raise ValueError(f"bad --devices value {text!r}")
    return out


def main(argv=None):
    args = build_parser().parse_args(argv)
    if not args.cas9:
        sys.exit("Please select at least one CRISPR system: Cas9")     # CROPSR.py:335-336
    if args.verbose:
        print(banner(args))
    devices = parse_devices(args.devices) if args.devices else [args.device]
    pams = args.offtarget_pams.split(",") if args.offtarget_pams is not None else []
    if args.offtargets is not None or args.offtarget_sites is not None or args.offtarget_scores is not None:
        from .pipeline import check_offtarget_args
        try:
            check_offtarget_args(args.l, devices, args.mismatches,
                                 args.max_sites if args.offtarget_sites is not None else None, pams)
        except ValueError as e:
            flag = ("--offtarget-sites" if args.offtarget_sites is not None else
                    "--offtargets" if args.offtargets is not None else "--offtarget-scores")
            sys.exit(f"CROPSR.py: error: {flag}: {e}")
    elif args.offtarget_pams is not None:
        sys.exit("CROPSR.py: error: --offtarget-pams: no off-target table asked for (--offtargets, --offtarget-sites, "
                 "--offtarget-scores)")
    if args.side_output is not None:
        from .pipeline import check_side_output_args
        try:
            check_side_output_args(args.L)
        except ValueError as e:
            sys.exit(f"CROPSR.py: error: --side-output: {e}")
    from . import engine, pipeline
    engine.init(devices[0])
    pipeline.run_cas9(args.f, args.g, args.o, args.l, args.verbose, args.blas_threads,
                      side_output=args.side_output, flank=args.L, annotation_info=args.p, devices=devices,
                      offtargets=args.offtargets, max_mismatches=args.mismatches,
                      offtarget_sites=args.offtarget_sites, max_sites=args.max_sites,
                      offtarget_scores=args.offtarget_scores, offtarget_pams=pams)
    return 0
