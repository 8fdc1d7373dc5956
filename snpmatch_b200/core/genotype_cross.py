"""
`snpmatch genotype_cross` — windowed parent matching on the GPU (SURVEY 8(f)-4).

Mirrors `snpmatch/core/genotype_cross.py`: `getWindowGenotype` (:21-49), `GenotypeCross` (:52-254: parents'
segregating markers :59-116, `get_window_genotype_gts` :188-199, `genotype_cross` :210-241, `write_output_genotype_cross`
:243-250) and `potatoCrossGenotyper` (:264-287).  The parents' columns come out of the resident panel with the column kernel
(`snpm_db_read_columns`), the join of the segregating markers with the VCF markers runs on the device, and the whole
window x sample loop (counts + three-way likelihood call) is ONE kernel launch (`snpm_cross_window_genotypes`,
csrc/cross_geno.cuh) instead of `windows x samples` np.vectorize'd likelihood calls.

Out of scope: the HMM (`genotype_cross_hmm`, infer.py).  Deliberate departures: with `--father` the reference indexes the
parents' GT arrays chromosome-relative and appends arrays of unequal length (genotype_cross.py:73-82), which only works when
both parental files list exactly the same positions of one chromosome; here both parents are aligned on the union of their
positions (missing where a parent lacks the position), which is what the surrounding code expects.
"""
import logging
import os

import numpy as np

from .. import lib
from . import genomes
from . import labels
from . import parsers
from . import snp_genotype
from . import snpmatch

log = logging.getLogger(__name__)
genome = None           # set by potatoCrossGenotyper, like the module global of the reference (genotype_cross.py:273-274)


def getWindowGenotype(matchedNos, totalMarkers, lr_thres, n_marker_thres=5):
    """(geno, pval) of one window (genotype_cross.py:21-49); the likelihoods come from the device epilogue."""
    pval = ''
    geno = 'NA'
    if totalMarkers < n_marker_thres:
        return (geno, 'NA')
    assert len(matchedNos) == 3
    if np.array_equal(np.array(matchedNos), np.repeat(0, 3)):
        return (geno, 'NA')
    likes = snpmatch.GenotyperOutput.calculate_likelihoods(matchedNos, np.repeat(totalMarkers, 3).tolist())
    pval = ",".join("%.2f" % item for item in likes[1])
    if len(np.where(likes[1] == 1)[0]) > 1:      # matching to multiple
        return (1, pval)
    high_match = np.nanargmin(likes[0])
    rest = likes[1][np.nonzero(likes[1] - 1)]
    lr_next = np.nan if (len(rest) == 0 or np.all(np.isnan(rest))) else np.nanmin(rest)
    if np.isnan(lr_next):
        lr_next = lr_thres
    if high_match == 0 and lr_next >= lr_thres:
        geno = 0
    elif high_match == 2 and lr_next >= lr_thres:
        geno = 2
    if high_match == 1:
        geno = 1
    return (geno, pval)


def _row_chromosomes(panel, rows):
    starts = np.asarray(panel.chr_regions)[:, 0]
    return np.asarray(panel.chrs).astype("U")[np.searchsorted(starts, rows, side="right") - 1]


def window_calls(par_chrs, par_pos, snps_p1, snps_p2, vcf_chrs, vcf_pos, gt_codes, gen, bin_len, lr_thres, device=0):
    """The window loop of genotype_cross (genotype_cross.py:218-238) for all samples at once.

    Returns dict(chr_ix int[W], start int[W], n_matched int[W], counts int32 [W,S,3], geno int8 [W,S] (-1 = NA),
    borderline uint8 [W,S])."""
    bin_len = int(bin_len)
    ids = gen.chrs_ids
    n_win = np.array([genomes.num_windows(l, bin_len) for l in gen.chrlen], dtype=np.int64)
    off = np.concatenate([[0], np.cumsum(n_win)])
    W = int(off[-1])

    def place(chrs, pos, what):
        _, codes, uniq = labels.map_labels(chrs, lambda c: c.lower().replace("chr", ""))      # genomes.py:75,95
        distinct = np.unique(uniq)
        assert len(distinct) <= len(ids), "Please change default --genome option"
        assert len(np.intersect1d(distinct, ids)) > 0, "Please change default --genome option"
        if len(np.intersect1d(distinct, ids)) < len(ids):
            log.warning("Some reference contigs are missing in %s", what)
        lut = {c: i for i, c in enumerate(ids)}
        cix = np.array([lut.get(c, -1) for c in uniq], dtype=np.int64)[codes]
        pos = np.asarray(pos, dtype=np.int64)
        k = (pos - 1) // bin_len
        ok = (cix >= 0) & (pos >= 1) & (k < n_win[np.maximum(cix, 0)])
        return cix, np.where(ok, off[np.maximum(cix, 0)] + k, -1)

    p_cix, p_win = place(par_chrs, par_pos, "the parental markers")
    v_cix, v_win = place(vcf_chrs, vcf_pos, "given SNPs")
    p_keep, v_keep = np.flatnonzero(p_win >= 0), np.flatnonzero(v_win >= 0)
    par_pos, vcf_pos = np.asarray(par_pos, dtype=np.int64), np.asarray(vcf_pos, dtype=np.int64)
    # inner join of the markers that lie in a window on (genome chromosome, position); pairs come back ordered by
    # (chromosome, position) = window order
    i_p, i_v = snp_genotype.join_coded(p_cix[p_keep], par_pos[p_keep], v_cix[v_keep], vcf_pos[v_keep], len(ids), device=device)
    i_p, i_v = p_keep[i_p], v_keep[i_v]
    win_start = np.concatenate([[0], np.cumsum(np.bincount(p_win[i_p], minlength=W))]).astype(np.int32)
    counts, geno, border = lib.cross_window_genotypes(i_p, i_v, win_start, snps_p1, snps_p2, gt_codes, lr_thres, device=device)
    return {"chr_ix": np.repeat(np.arange(len(ids)), n_win), "start": np.concatenate([1 + bin_len * np.arange(n) for n in n_win]),
            "n_matched": np.diff(win_start), "counts": counts, "geno": geno, "borderline": border}


class GenotypeCross(object):

    def __init__(self, g, parents, binLen=0, father=None, logDebug=True, genome_id=None):
        self.logDebug = logDebug
        self.g = g
        self.genome = genomes.Genome(genome_id) if genome_id is not None else genome
        self.get_segregating_snps_parents(parents, father)
        self.window_size = int(binLen)

    def get_segregating_snps_parents(self, parents, father):
        log.info("loading genotype data for parents, and identify segregating SNPs")
        if father is not None:
            log.info("input files: %s and %s" % (parents, father))
            if not (os.path.isfile(parents) and os.path.isfile(father)):
                snpmatch.die("either of the input files do not exists, please provide VCF/BED file for parent genotype information")
            p1_snps = parsers.ParseInputs(inFile=parents, logDebug=self.logDebug)
            p2_snps = parsers.ParseInputs(inFile=father, logDebug=self.logDebug)
            commonSNPsCHR = np.zeros(0, dtype="U1")
            commonSNPsPOS = np.zeros(0, dtype=int)
            snpsP1 = np.zeros(0, dtype='int8')
            snpsP2 = np.zeros(0, dtype='int8')
            for i in np.union1d(p1_snps.chrs, p2_snps.chrs):
                ix1, ix2 = np.where(p1_snps.chrs == i)[0], np.where(p2_snps.chrs == i)[0]
                positions = np.union1d(p1_snps.pos[ix1], p2_snps.pos[ix2])
                t1 = np.full(len(positions), -1, dtype='int8')
                t2 = np.full(len(positions), -1, dtype='int8')
                if len(ix1):
                    t1[np.searchsorted(positions, p1_snps.pos[ix1])] = parsers.parseGT(p1_snps.gt[ix1])
                if len(ix2):
                    t2[np.searchsorted(positions, p2_snps.pos[ix2])] = parsers.parseGT(p2_snps.gt[ix2])
                commonSNPsCHR = np.append(commonSNPsCHR, np.repeat(i, len(positions)))
                commonSNPsPOS = np.append(commonSNPsPOS, positions)
                snpsP1, snpsP2 = np.append(snpsP1, t1), np.append(snpsP2, t2)
            segSNPsind = np.where((snpsP1 != snpsP2) & (snpsP1 >= 0) & (snpsP2 >= 0))[0]
            commonSNPsCHR, commonSNPsPOS = commonSNPsCHR[segSNPsind], commonSNPsPOS[segSNPsind]
        else:
            assert len(parents.split("x")) == 2, "parents should be provided as '6091x6191'"
            try:
                indP1 = np.where(self.g.accessions == parents.split("x")[0])[0][0]
                indP2 = np.where(self.g.accessions == parents.split("x")[1])[0][0]
            except IndexError:
                snpmatch.die("parents are not in the dataset")
            cols = self.g.g_acc.snps[:, [indP1, indP2]]           # two columns of the resident panel (column kernel)
            snpsP1, snpsP2 = cols[:, 0], cols[:, 1]
            self.p1_ix = indP1
            self.p2_ix = indP2
            # only sites where the two parents differ and both are called (genotype_cross.py:108)
            segSNPsind = np.where((snpsP1 != snpsP2) & (snpsP1 >= 0) & (snpsP2 >= 0))[0]
            commonSNPsCHR = _row_chromosomes(self.g.g_acc, segSNPsind)
            commonSNPsPOS = np.asarray(self.g.g_acc.positions)[segSNPsind]
        log.info("number of segregating snps between parents: %s", len(segSNPsind))
        self.commonSNPsCHR = np.asarray(commonSNPsCHR).astype('U')
        self.commonSNPsPOS = commonSNPsPOS
        self.snpsP1 = snpsP1[segSNPsind]
        self.snpsP2 = snpsP2[segSNPsind]
        log.info("done!")

    def genotype_cross_hmm(self, input_file, min_na_per_sample=0.8):
        raise NotImplementedError("the HMM / Viterbi genotyper (genotype_cross.py:118-185, infer.py) is outside this package's scope")

    @staticmethod
    def get_window_genotype_gts(input_gt, snpsP1_gt, snpsP2_gt, lr_thres):
        """One window of one sample (genotype_cross.py:188-199) through the same device call the batched path uses."""
        num_snps = len(input_gt)
        assert num_snps == len(snpsP1_gt), "provide same number of SNPs"
        assert num_snps == len(snpsP2_gt), "provide same number of SNPs"
        codes = parsers.parseGT(input_gt).reshape(-1, 1)
        ix = np.arange(num_snps)
        counts, _, _ = lib.cross_window_genotypes(ix, ix, [0, num_snps], snpsP1_gt, snpsP2_gt, codes, lr_thres)
        return getWindowGenotype(counts[0, 0].tolist(), num_snps, lr_thres)

    def genotype_cross(self, input_file, lr_thres, good_samples_file=None, gpu_parse=False):
        """gpu_parse: the population VCF's genotype columns are parsed on the device (parsers.read_vcf_gt_codes, which raises
        ValueError on the inputs it refuses); the window calls and the lines are the same."""
        log.info("loading input files!")
        if gpu_parse:
            snpvcf = parsers.read_vcf_gt_codes(input_file)
            gt_codes = snpvcf['gt_codes']
        else:
            snpvcf = parsers.import_vcf_file(inFile=input_file, logDebug=self.logDebug, samples_to_load=None)
            gt = snpvcf['gt']
            gt_codes = parsers.parseGT(gt.ravel()).reshape(gt.shape) if gt.size else np.zeros(gt.shape, dtype=np.int8)
        num_samples = snpvcf['samples'].shape[0]
        log.info("number of samples printed: %s" % num_samples)
        gen = self.genome
        r = window_calls(self.commonSNPsCHR, self.commonSNPsPOS, self.snpsP1, self.snpsP2, snpvcf['chr'], snpvcf['pos'], gt_codes,
                         gen, self.window_size, float(lr_thres))
        self.last_window_calls = r
        outfile_str = ['id,,,' + ",".join(snpvcf['samples']), 'pheno,' + ',' + ',0' * num_samples]
        names = np.array(["NA", "0", "1", "2"])
        for w in range(len(r["start"])):
            cid = gen.chrs_ids[r["chr_ix"][w]]
            start, end = int(r["start"][w]), int(r["start"][w]) + self.window_size - 1
            bin_str = cid + ":" + str(start) + "-" + str(end)
            cm_mid = gen.estimated_cM_distance(cid + "," + str(int(round(float(np.mean([start, end]))))))
            if r["n_matched"][w] == 0:
                geno_samples = ',NA' * num_samples
            else:
                geno_samples = "".join("," + g for g in names[r["geno"][w].astype(int) + 1])
            outfile_str.append("%s,%s,%s%s" % (bin_str, cid, cm_mid, geno_samples))
        log.info("done!")
        return np.array(outfile_str, dtype=str)

    @staticmethod
    def write_output_genotype_cross(outfile_str, output_file):
        log.info("writing file: %s" % output_file)
        with open(output_file, 'w') as outfile:
            for ef in outfile_str:
                outfile.write("%s\n" % ef)
        log.info("done!")


def potatoCrossGenotyper(args):
    global genome
    gpu_parse = bool(args.get('gpu_parse'))
    if gpu_parse and not args['hmm']:
        try:
            parsers.vcf_population_samples(args['inFile'])       # header refusals before the database goes to the device
        except ValueError as e:
            snpmatch.die(str(e))
    genome = genomes.Genome(args['genome'])
    log.info("loading database files")
    g = snp_genotype.Genotype(args['hdf5File'], args['hdf5accFile'])
    log.info("done!")
    crossgenotyper = GenotypeCross(g, args['parents'], args['binLen'], args['father'], args['logDebug'])
    if args['hmm']:
        outfile_str = crossgenotyper.genotype_cross_hmm(args['inFile'])
    else:
        try:
            outfile_str = crossgenotyper.genotype_cross(args['inFile'], float(args['lr_thres']), gpu_parse=gpu_parse)
        except ValueError as e:
            if not gpu_parse:
                raise
            snpmatch.die(str(e))
    crossgenotyper.write_output_genotype_cross(outfile_str, args['outFile'])
