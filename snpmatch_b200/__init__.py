"""
snpmatch_b200 — B200-native genotype-matching hot path behind SNPmatch's `inbred` / `cross` interface.

The command line mirrors the reference's `snpmatch/__init__.py` for the two sub-commands on the
matching path (`inbred`, `cross`: flags of __init__.py:44-63), `parser` (:80-84) and the callers next to the
path that work on the resident panel (SURVEY.md 8(f)-3/4: `pairsnp` :86-92, `simulate` :101-111, `genotype_cross`
:65-78 without its HMM mode, `makedb` :94-99 without bcftools / HDF5); the other
sub-commands of the reference are outside this package's scope (SURVEY.md section 8).
"""
import argparse
import logging
import os
import os.path
import sys

__version__ = '0.1.0'
__reference_version__ = '5.0.1'


def setLog(logDebug):
    log = logging.getLogger()
    level = logging.DEBUG if logDebug else logging.ERROR
    handler = logging.StreamHandler()
    handler.setLevel(level)
    handler.setFormatter(logging.Formatter("%(asctime)s - %(name)s - %(levelname)s - %(message)s"))
    log.setLevel(level)
    log.addHandler(handler)


def die(msg):
    sys.stderr.write('Error: ' + msg + '\n')
    sys.exit(1)


def check_file(inFile):
    if not inFile:
        die("file: %s not specified" % inFile)
    if not os.path.isfile(inFile):
        die("input file does not exist: " + inFile)


def snpmatch_inbred(args):
    if args.get('samples'):
        samples = read_sample_list(args['samples'], args['outFile'])
        from .core import snpmatch
        snpmatch.potatoGenotyperMany(args, samples)
        return
    check_file(args['inFile'])
    from .core import snpmatch
    snpmatch.potatoGenotyper(args)


def snpmatch_cross(args):
    if args.get('samples'):
        samples = read_sample_list(args['samples'], args['outFile'])
        from .core import csmatch
        csmatch.potatoCrossIdentifierMany(args, samples)
        return
    check_file(args['inFile'])
    from .core import csmatch
    csmatch.potatoCrossIdentifier(args)


def read_sample_list(list_file, out_prefix, default_name=None):
    """`inbred --samples` / `cross --samples`: one sample file per line, optionally a tab and the sample's output prefix (default
    <out_prefix>.<file name up to its first '.'>).  Blank lines are skipped.  Returns [(path, prefix)]; dies on a missing
    file, an empty list or two samples with the same prefix.  `pairsnp --samples` reads the second column as the sample's
    label: default_name(path) gives it when the line has none."""
    check_file(list_file)
    samples = []
    with open(list_file) as fh:
        for line in fh:
            line = line.rstrip("\r\n")
            if not line.strip():
                continue
            cols = line.split("\t")
            path = cols[0].strip()
            if len(cols) > 1 and cols[1].strip():
                prefix = cols[1].strip()
            else:
                prefix = default_name(path) if default_name else out_prefix + "." + os.path.basename(path).split(".")[0]
            samples.append((path, prefix))
    if not samples:
        die("sample list is empty: " + list_file)
    for path, _ in samples:
        check_file(path)
    seen = {}
    for path, prefix in samples:
        if prefix in seen:
            die("samples %s and %s have the same %s %s" % (seen[prefix], path, "label" if default_name else "output prefix", prefix))
        seen[prefix] = path
    return samples


def snpmatch_parser(args):
    check_file(args['inFile'])
    if not args['outFile'] and os.path.isfile(args['inFile'] + ".snpmatch.npz"):
        os.remove(args['inFile'] + ".snpmatch.npz")
    from .core import parsers
    parsers.potatoParser(inFile=args['inFile'], logDebug=args['logDebug'], outFile=args['outFile'])


def snpmatch_paircomparions(args):
    if args.get('samples'):
        if args['inFile_1'] or args['inFile_2']:
            die("--samples compares every pair of the list; it cannot be combined with -i / -j")
        samples = read_sample_list(args['samples'], args['outFile'], default_name=os.path.basename)
        from .core import snpmatch
        snpmatch.pairwiseScoreMany(args, samples)
        return
    check_file(args['inFile_1'])
    check_file(args['inFile_2'])
    from .core import snpmatch
    snpmatch.pairwiseScore(args['inFile_1'], args['inFile_2'], args['logDebug'], args['outFile'], args['hdf5File'])


def makedb_vcf_to_db(args):
    check_file(args['inFile'])
    from .core import makedb
    makedb.makedb_from_vcf(args)


def simulate_snps(args):
    from .core import simulate
    simulate.potatoSimulate(args)


def genotype_cross(args):
    if not args['parents']:
        die("parents not specified")
    from .core import genotype_cross as gtm
    gtm.potatoCrossGenotyper(args)


def get_options(description, version_message):
    p = argparse.ArgumentParser(description=description)
    p.add_argument('-V', '--version', action='version', version=version_message)
    sub = p.add_subparsers(title='commands', description='one of', help='what each does')
    db_help = "Path to the SNP database: the reference's row-chunked hdf5 file (needs h5py) or a packed .npz written by Genotype.save_packed"
    inbred = sub.add_parser('inbred', help="identify the accession an inbred sample comes from")
    inbred_in = inbred.add_mutually_exclusive_group()
    inbred_in.add_argument("-i", "--input_file", dest="inFile", help="sample variants: VCF (GT, optional PL), BED (chr, pos, GT) or a parser .npz")
    inbred_in.add_argument("--samples", dest="samples", default=None,
                           help="text file listing many samples, one path per line (VCF/BED/npz), optionally a tab and that sample's output "
                                "prefix (default <-o>.<file name up to its first '.'>); all samples are scored together on the GPU; exit "
                                "status 1 when --refine finds a sample without top hits")
    inbred.add_argument("-d", "--hdf5_file", default=None, dest="hdf5File", help=db_help)
    inbred.add_argument("-e", "--hdf5_acc_file", default=None, dest="hdf5accFile", help="Column-chunked hdf5 file of the reference (accepted for compatibility; one resident copy serves both)")
    inbred.add_argument("--refine", action="store_true", dest="refine", default=False, help="re-score the accessions that cannot be told apart on the SNPs that segregate among them")
    inbred.add_argument("--skip_db_hets", action="store_true", dest="skip_db_hets", default=False, help="treat heterozygous database calls as missing")
    inbred.add_argument("-v", "--verbose", action="store_true", dest="logDebug", default=False, help="log at DEBUG level")
    inbred.add_argument("-o", "--output", dest="outFile", default="identify_inbred", help="output prefix (<prefix>.scores.txt, <prefix>.matches.json)")
    inbred.set_defaults(func=snpmatch_inbred)

    cross = sub.add_parser('cross', help="identify the parents of a cross (F2, F3): window scores and simulated F1s")
    cross_in = cross.add_mutually_exclusive_group()
    cross_in.add_argument("-i", "--input_file", dest="inFile", help="sample variants: VCF (GT, optional PL), BED (chr, pos, GT) or a parser .npz")
    cross_in.add_argument("--samples", dest="samples", default=None,
                          help="text file listing many samples, one path per line (VCF/BED/npz), optionally a tab and that sample's output "
                               "prefix (default <-o>.<file name up to its first '.'>); all samples are scored together on the GPU")
    cross.add_argument("-d", "--hdf5_file", default=None, dest="hdf5File", help=db_help)
    cross.add_argument("-e", "--hdf5_acc_file", default=None, dest="hdf5accFile", help="Column-chunked hdf5 file of the reference (accepted for compatibility)")
    cross.add_argument("-b", "--binLength", dest="binLen", help="window length in bp", default=300000, type=int)
    cross.add_argument("--genome", dest="genome", default="athaliana_tair10", help="bundled genome id or path to a genome JSON (chromosome names and lengths)")
    cross.add_argument("--skip_db_hets", action="store_true", dest="skip_db_hets", default=False, help="treat heterozygous database calls as missing")
    cross.add_argument("-v", "--verbose", action="store_true", dest="logDebug", default=False, help="log at DEBUG level")
    cross.add_argument("-o", "--output", dest="outFile", default="identify_cross", help="output prefix (<prefix>.scores.txt, <prefix>.windowscore.txt, <prefix>.scores.txt.matches.json)")
    cross.set_defaults(func=snpmatch_cross)

    parser = sub.add_parser('parser', help="parse a VCF/BED file into the .npz the other commands load")
    parser.add_argument("-i", "--input_file", dest="inFile", help="sample variants: VCF (GT, optional PL), BED (chr, pos, GT) or a parser .npz")
    parser.add_argument("-v", "--verbose", action="store_true", dest="logDebug", default=False, help="log at DEBUG level")
    parser.add_argument("-o", "--output", dest="outFile", help="prefix of the parser dump (<prefix>.npz)")
    parser.set_defaults(func=snpmatch_parser)

    gc = sub.add_parser('genotype_cross', help="call parent 1 / het / parent 2 per window for every sample of a multi-sample VCF")
    gc.add_argument("-i", "--input_file", dest="inFile", help="multi-sample VCF of the cross")
    gc.add_argument("-d", "--hdf5_file", default=None, dest="hdf5File", help=db_help)
    gc.add_argument("-e", "--hdf5_acc_file", default=None, dest="hdf5accFile", help="Column-chunked hdf5 file of the reference (accepted for compatibility)")
    gc.add_argument("-p", "--parents", dest="parents", help="the two parents as database accession ids, e.g. 6091x6191 (or the file of parent 1 with -q)")
    gc.add_argument("-q", "--father", dest="father", help="VCF/BED file of parent 2 when the parents are given as files (then -p is the file of parent 1)")
    gc.add_argument("-b", "--binLength", dest="binLen", help="window length in bp", type=int, default=200000)
    gc.add_argument("--good_samples", dest="good_samples", help="accepted for compatibility (unused by the reference's window genotyper)", default=None)
    gc.add_argument("--lr_thres", dest="lr_thres", default=1.5, type=float, help="second-best likelihood ratio a homozygous call needs")
    gc.add_argument("--hmm", dest="hmm", action="store_true", help="HMM Viterbi genotyper of the reference: not part of this package")
    gc.add_argument("--genome", dest="genome", default="athaliana_tair10", help="bundled genome id or path to a genome JSON (chromosome names and lengths)")
    gc.add_argument("-o", "--output", dest="outFile", default="genotype_cross", help="output CSV (R/qtl layout)")
    gc.add_argument("-v", "--verbose", action="store_true", dest="logDebug", default=False, help="log at DEBUG level")
    gc.set_defaults(func=genotype_cross)

    pair = sub.add_parser('pairsnp', help="agreement of the genotype calls two samples (or every pair of many samples) share")
    pair.add_argument("-i", "--input_file_1", dest="inFile_1", help="first sample (VCF/BED/npz)")
    pair.add_argument("-j", "--input_file_2", dest="inFile_2", help="second sample (VCF/BED/npz)")
    pair.add_argument("--samples", dest="samples", default=None,
                      help="text file listing many samples, one path per line (VCF/BED/npz), optionally a tab and that sample's label "
                           "(default: the file name); every pair is compared in one GPU pass: <-o>.identity.tsv, <-o>.common.tsv")
    pair.add_argument("--pairs_json", action="store_true", dest="pairs_json", default=False,
                      help="with --samples: also <-o>.pairs.jsonl, one line per pair with the statistics -i/-j writes to .matches.json")
    pair.add_argument("-d", "--hdf5_file", dest="hdf5File", default=None, help=db_help)
    pair.add_argument("-v", "--verbose", action="store_true", dest="logDebug", default=False, help="log at DEBUG level")
    pair.add_argument("-o", "--output", dest="outFile", default="pairsnp", help="output prefix (<prefix>.matches.json)")
    pair.set_defaults(func=snpmatch_paircomparions)

    mk = sub.add_parser('makedb', help="build the packed database (<id>.npz) and the genome JSON from a multi-sample VCF of the known strains, or from the intermediate CSV of the reference")
    mk.add_argument("-i", "--input_vcf", dest="inFile", help="VCF of the known strains (biallelic SNPs), or a CSV with the columns Chromosome,Position,<accession>...")
    mk.add_argument("-p", "--bcftools_path", dest="bcfpath", default='', help="accepted for compatibility: the VCF is read directly, bcftools is not needed")
    mk.add_argument("-o", "--out_db_id", dest="db_id", help="output id: <id>.npz, <id>.json (and <id>.csv for VCF input)")
    mk.add_argument("-v", "--verbose", action="store_true", dest="logDebug", default=False, help="log at DEBUG level")
    mk.set_defaults(func=makedb_vcf_to_db)

    sim = sub.add_parser('simulate', help="draw a synthetic sample (or F1) from the database to test the genotyper")
    sim.add_argument("-d", "--hdf5_file", default=None, dest="hdf5File", help=db_help)
    sim.add_argument("-e", "--hdf5_acc_file", default=None, dest="hdf5accFile", help="Column-chunked hdf5 file of the reference (accepted for compatibility)")
    sim.add_argument("-a", "--ecotype_id", dest="AccID", help="accession id to draw from; two ids as AxB with --f1")
    sim.add_argument("-n", "--number_of_snps", dest="numSNPs", help="markers to draw", type=int)
    sim.add_argument("-p", "--error_rate", dest="err_rate", help="fraction of the drawn calls replaced by random ones", default=0.001, type=float)
    sim.add_argument("--f1", action="store_true", dest="simF1", default=False, help="simulate the F1 of the two accessions given with -a")
    sim.add_argument("--het_frac", default=1, type=float, dest="rm_het", help="For simulated F1s: fraction of segregating sites kept heterozygous; the rest become homozygous ref or alt with equal probability")
    sim.add_argument("-o", "--output", dest="outFile", help="BED file to write")
    sim.add_argument("-v", "--verbose", action="store_true", dest="logDebug", default=False, help="log at DEBUG level")
    sim.set_defaults(func=simulate_snps)
    return p


def main(argv=None):
    """Exit codes as in the reference (__init__.py:155-183): 0 ok, 2 on an exception."""
    version_message = '%%(prog)s v%s (B200 matching path of SNPmatch %s)' % (__version__, __reference_version__)
    parser = get_options("SNPmatch genotype matching on NVIDIA B200", version_message)
    args = vars(parser.parse_args(argv))
    setLog(args.get('logDebug', False))
    if 'func' not in args:
        parser.print_help()
        return 0
    try:
        args['func'](args)
        return 0
    except KeyboardInterrupt:
        return 0
    except Exception as e:
        logging.exception(e)
        return 2


if __name__ == '__main__':
    sys.exit(main())
