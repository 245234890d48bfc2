"""Drop-in surface of the reference's hot path: same names, argument meaning and return shapes
as /root/reference/frisk/__init__.py ("F:"), backed by the CUDA library.

Two levels:

* ``main()`` / ``score_genome()`` -- the batch path a user should run: stages 2+3 of the
  reference's ``main()`` (F:1437-1507) through ``engine.Pipeline``; writes the same TSV, the same
  genome-k-mer pickle (list of dicts + 3 meta dicts, F:356-363) and the same windows DataFrame
  pickle (F:1501), honours ``--recalc/--recalcWin/--exitAfter``.
* the per-call functions ``computeKmers``, ``IvomBuild``, ``KLD`` -- kept for callers that use
  the reference's function API (e.g. its PCA stage, F:1571-1578).  Every one of them runs its
  arithmetic on the GPU (background / finalize / genome_ivom / kld kernels); they materialise
  Python dicts only to honour the reference's return types, so they are slow by construction --
  the batch path never builds a dict.

``countN``, ``calcGC``, ``calcRIP``, ``rangeMaps``, ``revComplement``, ``iterFasta`` and
``crawlGenome`` are string/dict helpers of the reference's API (a handful of counts or three
divisions); they are host glue here too.  In the batch path the same quantities (30 % rule, GC,
RIP) are computed inside the score kernel and the tests check the two agree.

There is no CPU fallback: without the CUDA library / a GPU the compute entry points raise.
"""
from __future__ import annotations

import argparse
import logging
import os
import pickle
import sys
from typing import Dict, Iterator, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib, engine

__all__ = ["LETTERS", "tempPathCheck", "countN", "calcGC", "iterFasta", "crawlGenome", "prepareMaps", "rangeMaps",
           "revComplement", "computeKmers", "IvomBuild", "KLD", "calcRIP", "makePicklePath", "mainArgs", "main",
           "scrubMirrors", "flattenKmerMap", "pcaFeatures", "pcaFeaturesFromIntervals", "score_genome", "FRISK_VERSION"]

FRISK_VERSION = "b200-0.1"
LETTERS = engine.LETTERS                   # F:70 -- alphabet and table order
_UPPER = b"ATGC"


# ------------------------------------------------------------------------------ small helpers
def tempPathCheck(args) -> None:
    """F:78-83."""
    folder = os.path.abspath(args.tempDir)
    if not os.path.isdir(folder):
        os.makedirs(folder)


def _as_bytes(sequence) -> bytes:
    return sequence.encode() if isinstance(sequence, str) else bytes(sequence)


def countN(sequence) -> Tuple[int, int]:
    """F:106-118: (# upper-case ATGC characters, # everything else)."""
    raw = _as_bytes(sequence)
    good = sum(raw.count(bytes([c])) for c in _UPPER)
    return good, len(raw) - good


def calcGC(sequence) -> float:
    """F:120-137: (G+C)/(A+T+G+C) over upper-case bases; ZeroDivisionError if there are none."""
    raw = _as_bytes(sequence)
    gc = raw.count(b"G") + raw.count(b"C")
    at = raw.count(b"A") + raw.count(b"T")
    return float(gc) / (gc + at)


def iterFasta(path: str) -> Iterator[Tuple[str, str]]:
    """F:139-164: (name, sequence) per record; records found by the library's FASTA scanner
    (same header-token and blank-line rules), sequences returned as str like the reference."""
    g_names, bodies = _fasta_records(path)
    for name, body in zip(g_names, bodies):
        yield name, body


def _fasta_records(path: str):
    import ctypes as C
    if path.endswith(".gz") or path.endswith('.gz"'):
        import gzip
        with gzip.open(path, "rb") as fh:
            data = fh.read()
    else:
        with open(path, "rb") as fh:
            data = fh.read()
    buf = np.frombuffer(data, dtype=np.uint8)
    L = _lib.lib()
    n = C.c_uint64(0)
    ptr = lambda a: C.c_void_p(a.ctypes.data) if a is not None else C.c_void_p(0)
    _lib.check(L.frisk_b200_fasta_scan(ptr(buf), len(buf), 0, None, None, None, None, None, C.byref(n)), "frisk_b200_fasta_scan")
    cap = int(n.value)
    no = np.zeros(cap, np.uint64); nl = np.zeros(cap, np.uint32); bo = np.zeros(cap, np.uint64)
    be = np.zeros(cap, np.uint64); sl = np.zeros(cap, np.uint64)
    _lib.check(L.frisk_b200_fasta_scan(ptr(buf), len(buf), cap, ptr(no), ptr(nl), ptr(bo), ptr(be), ptr(sl), C.byref(n)),
               "frisk_b200_fasta_scan")
    names = [data[int(no[i]):int(no[i]) + int(nl[i])].decode() for i in range(cap)]
    drop = bytes(range(9, 14)) + b" "
    bodies = [data[int(bo[i]):int(be[i])].translate(None, drop).decode() for i in range(cap)]
    return names, bodies


def crawlGenome(args, querySeq: str) -> Iterator[Tuple[str, str, int, int]]:
    """F:194-251: yields (window sequence, scaffold name, start, stop).  Window enumeration comes
    from the library (frisk_b200_windows); the 30 % unresolved rule (F:213, F:238) is applied here on
    the strings because this generator's contract is strings (the batch path applies it in-kernel)."""
    names, bodies = _fasta_records(querySeq)
    g = engine.PackedGenome.from_scaffolds(list(zip(names, bodies)))
    wins = g.windows(args.windowlen, args.increment, args.scaffoldsAll)
    for i in range(len(wins)):
        s = int(wins.scaf[i])
        o = int(wins.off[i] - g.scaf_off[s])
        seq = bodies[s][o:o + int(wins.length[i])]
        if countN(seq)[1] >= 0.3 * len(seq):
            continue
        yield seq, names[s], int(wins.start[i]), int(wins.stop[i])


_kmer_keys = engine.kmer_words              # all 4^k words in the reference's dict order (F:253-265)


def prepareMaps(k: int, maxk: int, kmers: Sequence[str]) -> Dict[str, int]:
    """F:253-265 (kept for signature compatibility): extends `kmers` to length maxk."""
    words = list(kmers)
    for _ in range(k, maxk):
        words = [w + c for w in words for c in LETTERS]
    return dict.fromkeys(words, 0)


def rangeMaps(kMin: int, kMax: int) -> List[Dict[str, int]]:
    """F:267-274: one zeroed dict per order."""
    return [dict.fromkeys(_kmer_keys(k), 0) for k in range(kMin, kMax + 1)]


def revComplement(kmer: str) -> str:
    """F:276-278."""
    return kmer.translate(str.maketrans("ATGC", "TACG"))[::-1]


# ------------------------------------------------------------------------------ GPU-backed functions
def _tables_to_dicts(tables_1k: np.ndarray, kmin: int, kmax: int) -> List[Dict[str, int]]:
    out = []
    for k in range(kmin, kmax + 1):
        a = _lib.table_size(1, k - 1) if k > 1 else 0
        vals = tables_1k[a:a + 4 ** k]
        out.append(dict(zip(_kmer_keys(k), (int(v) for v in vals))))
    return out


def _dicts_to_tables(maps: Sequence[Dict[str, int]], kmin: int, kmax: int) -> np.ndarray:
    """list of dicts (orders kmin..kmax) -> int64 array of orders 1..kmax (orders < kmin zero)."""
    out = np.zeros(_lib.table_size(1, kmax), dtype=np.int64)
    for k in range(kmin, kmax + 1):
        a = _lib.table_size(1, k - 1) if k > 1 else 0
        d = maps[k - kmin]
        out[a:a + 4 ** k] = np.fromiter((d[w] for w in _kmer_keys(k)), dtype=np.int64, count=4 ** k)
    return out


def computeKmers(args, genomepickle=None, window=None, genomeMode=False, pcaMode=False, kmerMap=None, getMeta=True,
                 sym=False):
    """F:280-367.  Same arguments and return value: [dict per order kmin..kmax] (+ {'totalLen'},
    {'exMax'}, {'nnTotal'} when getMeta).  The counting runs on the GPU: the sequences are packed,
    counted by frisk_b200_background (forward strand) and finalised by frisk_b200_finalize_tables
    with symmetric = genomeMode or sym (F:350)."""
    import torch
    if kmerMap is not None and sum(kmerMap[0].values()) != 0:          # F:291-293
        logging.info("kmer template is not blank!")
        sys.exit(1)
    kmin, kmax = (args.pcaMin, args.pcaMax) if pcaMode else (args.minWordSize, args.maxWordSize)   # F:309-314
    if genomeMode:
        logging.info("Computing kmers for %s" % args.hostSeq)
        g = engine.PackedGenome.from_fasta(args.hostSeq)
        mask_host = bool(args.maskHost)                                # F:336: lower-case words dropped from the genome table
    else:
        g = engine.PackedGenome.from_scaffolds(list(window))
        mask_host = False                                              # F:334-335: windows are always upper-cased
    if kmax > _lib.MAX_K:
        _lib.check(_lib.E_UNSUPPORTED, "computeKmers(kmax=%d)" % kmax)
    dg = engine.DeviceGenome(g)
    d_fwd = engine.background(dg, kmax, mask_host)
    d_tables, d_valid = engine.finalize(d_fwd, kmax, symmetric=bool(genomeMode or sym))
    torch.cuda.synchronize(dg.device)
    tables = d_tables.cpu().numpy()
    maps = _tables_to_dicts(tables, kmin, kmax)
    if getMeta:                                                        # F:356-359
        maps.append({"totalLen": g.total_len})
        maps.append({"exMax": g.ex_max(kmax, int(d_valid.item()))})
        maps.append({"nnTotal": g.nn_total})
    if genomeMode:                                                     # F:361-365
        if genomepickle:
            with open(genomepickle, "wb") as fh:
                pickle.dump(maps, fh, protocol=2)
        logging.info("Processed %d sequences" % len(g.names))
    return maps


def IvomBuild(windowKmers, args, GenomeKmers, isGenomeIVOM):
    """F:369-457: {kmax-mer: normalised IVOM value} for the kmax-mers present in the window, from the
    window's own tables or from the genome's.  The per-k-mer values come from the
    frisk_b200_genome_ivom kernel run on the chosen tables."""
    import torch
    kmin, kmax = args.minWordSize, args.maxWordSize
    kr = kmax - kmin
    src = GenomeKmers if isGenomeIVOM else windowKmers
    space = src[kr + 1]["totalLen"] - src[kr + 3]["nnTotal"]           # F:379-380
    _lib.require_device()
    dev = torch.device("cuda:0")
    d_tables = torch.from_numpy(_dicts_to_tables(src, kmin, kmax)).to(dev)
    d_ig = engine.genome_ivom(d_tables, kmin, kmax, space)
    raw = d_ig.cpu().numpy().reshape(-1, 2)[:, 0]
    keys = _kmer_keys(kmax)
    present = np.fromiter((windowKmers[kr][w] != 0 for w in keys), dtype=bool, count=len(keys))
    vals = raw[present]
    if np.isnan(vals).any():
        raise ZeroDivisionError("float division by zero")              # F:401-437
    total = vals.sum()
    if vals.size and total == 0:
        raise ZeroDivisionError("float division by zero")              # F:454
    return dict(zip((k for k, p in zip(keys, present) if p), (float(v) for v in vals / total)))


def KLD(GenomeIVOM, windowIVOM, args=None):
    """F:459-472 on the GPU (frisk_b200_kld)."""
    import ctypes as C
    import torch
    if not windowIVOM:
        return 0
    _lib.require_device()
    dev = torch.device("cuda:0")
    w = torch.tensor([float(v) for v in windowIVOM.values()], dtype=torch.float64, device=dev)
    g = torch.tensor([float(GenomeIVOM[k]) for k in windowIVOM], dtype=torch.float64, device=dev)
    out = torch.zeros(1, dtype=torch.float64, device=dev)
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(_lib.lib().frisk_b200_kld(C.c_void_p(g.data_ptr()), C.c_void_p(w.data_ptr()), w.numel(),
                                         C.c_void_p(out.data_ptr()), st), "frisk_b200_kld")
    val = float(out.item())
    if val != val:
        raise ValueError("math domain error")                          # F:470 on a non-positive ratio
    return val


def calcRIP(windowKmers, args):
    """F:474-495: PI, SI, CRI from the window's dinucleotide table (ValueError if 2 is not in
    [minWordSize, maxWordSize], like the reference's list.index)."""
    di = windowKmers[list(range(args.minWordSize, args.maxWordSize + 1)).index(2)]
    nan = float("nan")
    PI = di["TA"] / float(di["AT"]) if di["AT"] > 0 else nan
    sub = di["AC"] + di["GT"]
    SI = (di["CA"] + di["TG"]) / float(sub) if sub > 0 else nan
    CRI = PI - SI if (PI and SI) else nan                              # F:491: 0.0 falsy, NaN truthy
    return PI, SI, CRI


# ------------------------------------------------------------------------------ batch path + CLI
def scrubMirrors(kDicts):
    """F:797-811: per order, drop the k-mers whose reverse complement was already seen (table order)."""
    clean = []
    for table in kDicts:
        kept = {}
        for key, value in table.items():
            if key in kept or revComplement(key) in kept:
                continue
            kept[key] = value
        clean.append(kept)
    return clean


def flattenKmerMap(kMap, window=1, seqLen=1, kmin=1, kmax=5, prop=False):
    """F:813-831: the tables of orders kmin..kmax as one vector -- proportions within each order
    (prop=True) or counts scaled to a standard window length."""
    values = []
    for table in kMap:
        if not table or not (kmin <= len(next(iter(table))) <= kmax):
            continue
        if prop:
            total = sum(table.values())
            values.extend(float(v) / total for v in table.values())      # ZeroDivisionError like the reference
        else:
            values.extend(table.values())
    arr = np.array(values)
    return arr if prop else (float(window) / seqLen) * arr


def pcaFeatures(args, regions, device="cuda:0"):
    """The reference's loop F:1571-1591 for all regions at once: ``regions`` = [(name, sequence)];
    returns (labels, float64[n, F]) = (anomLabels, anomCounts).  One GPU kernel (one CTA per region)."""
    regions = list(regions)
    g = engine.PackedGenome.from_scaffolds(regions)
    dg = engine.DeviceGenome(g, device)
    feats = engine.region_features(dg, g.scaf_off, g.scaf_len.astype(np.uint32), args.pcaMin, args.pcaMax)
    if np.isnan(feats).any():
        raise ZeroDivisionError("float division by zero (reference F:824: a region without a valid word of some order)")
    return np.array([n for n, _ in regions]), feats


def pcaFeaturesFromIntervals(args, genome, intervals):
    """The same vectors straight from the packed planes: ``genome`` is an engine.DeviceGenome (e.g. the one the
    scores were computed from), ``intervals`` the (chrom, start, stop, ...) records of thresholdKLD / hmm2BED.
    Replaces getFasta + getBEDSeq (F:166-192: sequence = scaffold[start-1:stop], label "chrom:start:stop", records
    on unknown scaffolds or of zero length are skipped) + the per-region loop F:1571-1591 without ever
    materialising a sequence string."""
    g = genome.host
    index = {name: i for i, name in enumerate(g.names)}
    labels, off, length = [], [], []
    for rec in intervals:
        i = index.get(str(rec[0]))
        if i is None:
            logging.error("Scaffold %s not found in reference." % str(rec[0]))
            continue
        a, b = int(rec[1]) - 1, min(int(rec[2]), int(g.scaf_len[i]))
        name = ":".join([str(rec[0]), str(rec[1]), str(rec[2])])
        if b <= a or a < 0:
            logging.error("Error: Retrieved zero len sequence for %s" % name)
            continue
        labels.append(name)
        off.append(int(g.scaf_off[i]) + a)
        length.append(b - a)
    feats = engine.region_features(genome, np.array(off, np.uint64), np.array(length, np.uint32), args.pcaMin, args.pcaMax)
    if np.isnan(feats).any():
        raise ZeroDivisionError("float division by zero (reference F:824: a region without a valid word of some order)")
    return np.array(labels), feats


def makePicklePath(args, **kwargs) -> str:
    """F:497-506."""
    base = os.path.basename(args.hostSeq)
    tag = "_kmers_%s_%s_" % (args.minWordSize, args.maxWordSize)
    if kwargs["space"] == "genome":
        return os.path.join(args.tempDir, base + tag + "genome.p")
    if args.querySeq:
        base = os.path.basename(args.querySeq)
    return os.path.join(args.tempDir, base + tag + "KLD_window_%s_increment_%s.p" % (args.windowlen, args.increment))


def score_genome(args, device="cuda:0") -> engine.HotPathResult:
    """The whole hot path in one call: background tables of ``args.hostSeq`` + every window row of
    ``args.querySeq or args.hostSeq`` (F:1442, F:1478-1494)."""
    # device-side ingest: the FASTA text is copied to the GPU once and tokenised / packed there
    # (the reference reads each file three times in Python: F:170, F:203, F:297)
    # ... and everything goes through the C ABI alone (DevBuf planes, one frisk_b200_run_resident call): PyTorch is
    # never imported on this path -- its import takes several seconds, the run itself milliseconds
    # A BGZF file (bgzip, samtools) or a single gzip member (gzip, pigz) goes up compressed and is inflated on the device;
    # a multi-member .gz is inflated on the host.
    def ingest(path):
        return engine.open_genome_file(path, lambda buf, kind: engine.DeviceGenome._open_native(buf, device, kind))
    host = ingest(args.hostSeq)
    query = host if not args.querySeq or args.querySeq == args.hostSeq else ingest(args.querySeq)
    res = engine.run_resident(query, host if query is not host else None, kmin=args.minWordSize, kmax=args.maxWordSize,
                              w=args.windowlen, step=args.increment, mask_host=args.maskHost,
                              scaffolds_all=args.scaffoldsAll, rip=bool(args.RIP))
    res.raise_reference_errors()                 # the reference aborts on ZeroDivisionError (F:437, F:136)
    return res


def genome_kmers_from_result(res: engine.HotPathResult) -> list:
    """The reference's genomeKmers object (F:356-359) from a batch result."""
    return engine.genome_kmers(res.tables, res.kmin, res.kmax, res.meta)


def score_background(args, background, source: str, device="cuda:0") -> engine.HotPathResult:
    """Every window row of ``args.querySeq or args.hostSeq`` scored against stored background tables instead of tables
    counted from ``args.hostSeq``, which is only opened when it is also the query.  ``background``: (tables, kmin, kmax,
    meta) of ``engine.genome_kmers_tables``, from the reference's genomeKmers object loaded from ``source`` (F:1437)."""
    tables, kmin, kmax, meta = background
    path = args.querySeq or args.hostSeq
    query = engine.open_genome_file(path, lambda buf, kind: engine.DeviceGenome._open_native(buf, device, kind))
    # (the reference's cache key has no --maskHost, SURVEY section 5: the stored tables win, whatever the flag says now)
    logging.info("Scoring %s against the background tables in %s (orders %d..%d, totalLen %d, nnTotal %d); %s is not "
                 "counted again" % (path, source, kmin, kmax, meta[0], meta[2], args.hostSeq))
    with engine.Background(tables, kmin, kmax, meta, device) as bg:
        res = bg.run_resident(query, w=args.windowlen, step=args.increment, scaffolds_all=args.scaffoldsAll, rip=bool(args.RIP))
    res.raise_reference_errors()                 # the reference aborts on ZeroDivisionError (F:437, F:136)
    return res


def windows_frame(res: engine.HotPathResult, with_rip: bool):
    """The reference's allWindows DataFrame (F:1466-1491)."""
    import pandas as pd
    cols = {"name": res.names, "start": res.coords[:, 0], "stop": res.coords[:, 1], "windowKLD": res.rows[:, 0],
            "GC": res.rows[:, 1]}
    if with_rip:
        cols.update(PI=res.rows[:, 2], SI=res.rows[:, 3], CRI=res.rows[:, 4])
    return pd.DataFrame(cols)


def mainArgs(argv=None):
    """F:1127-1398: the reference's options (same flags, defaults and help); options of the
    downstream stages are accepted so existing command lines keep working."""
    p = argparse.ArgumentParser(description="Calculate all kmers in a given sequence", prog="frisk")
    p.add_argument("--version", action="version", version="frisk --" + str(FRISK_VERSION))
    p.add_argument("-H", "--hostSeq", type=str, required=True, help="The input host sequences (single species)")
    p.add_argument("-Q", "--querySeq", type=str, default=None,
                   help="Detect anomalous regions in this sequence by comparison to hostSeq. Defaults to hostSeq.")
    p.add_argument("--gffIn", type=str, default=None)
    p.add_argument("-O", "--outfile", type=str, default="raw_window_scores.bed", help="Write KLD-IVOM bed track to this file")
    p.add_argument("-t", "--tempDir", type=str, default="temp", help="Name of temporary directory")
    p.add_argument("--gffOutfile", type=str, default=None)
    p.add_argument("--hmmOutfile", type=str, default="2StateHmm.gff3")
    p.add_argument("--graphics", type=str, default=None)
    p.add_argument("--mergeDist", type=int, default=0)
    p.add_argument("--gffFeatures", type=str, default=None, nargs="+")
    p.add_argument("--gffRange", type=int, default=0)
    p.add_argument("-m", "--minWordSize", type=int, default=1, help="Minimum value of DNA word length")
    p.add_argument("-k", "--maxWordSize", type=int, default=8, help="Maxmimum value of DNA word length")
    p.add_argument("-w", "--windowlen", type=int, default=5000, help="Lenght of survey window")
    p.add_argument("-i", "--increment", type=int, default=2500, help="Slide survey window by this increment")
    p.add_argument("--maskHost", action="store_true", default=False)
    p.add_argument("--exitAfter", default=None, choices=[None, "GenomeKmers", "WindowKLD"], help="Exit after completing task.")
    p.add_argument("--recalc", action="store_false", default=True,
                   help="Force recalculation of reference sequence kmer counts if set.")
    p.add_argument("--recalcWin", action="store_false", default=True,
                   help="Force recalculation of KLD score for specified window length and icrement if set.")
    p.add_argument("--scaffoldsAll", action="store_true", default=False)
    p.add_argument("--threshTypeKLD", default=None, choices=[None, "percentile", "otsu"])
    p.add_argument("--percentileKLD", type=float, default=99.0)
    p.add_argument("--hmmKLD", action="store_true", default=False)
    p.add_argument("-F", "--forceThresholdKLD", type=float, default=None)
    p.add_argument("--RIP", action="store_true", default=False)
    p.add_argument("--RIPgff", type=str, default="RIP_annotation.gff3")
    p.add_argument("--minCRI", type=float, default=0.0)
    p.add_argument("--peakCRI", type=float, default=1.0)
    p.add_argument("--minPI", type=float, default=1.0)
    p.add_argument("--maxSI", type=float, default=1.0)
    p.add_argument("--runProjection", default=None, choices=[None, "PCA", "PY-TSNE", "SKL-TSNE", "IncrementalPCA", "NMF", "MDS"])
    p.add_argument("--projectionDims", type=int, default=2)
    p.add_argument("--dimReduce", default="windows", choices=["features", "windows"])
    p.add_argument("--cluster", default=None, choices=[None, "DBSCAN", "KMEANS", "SPECTRAL"])
    p.add_argument("--dumpPCAdata", action="store_true", default=False)
    p.add_argument("--spikeNormal", action="store_true", default=False)
    p.add_argument("--pcaMin", type=int, default=1)
    p.add_argument("--pcaMax", type=int, default=6)
    p.add_argument("--perplexity", type=float, default=20.0)
    p.add_argument("--tsneGradient", default="barnes_hut", choices=["barnes_hut", "exact"])
    p.add_argument("--tsneInitPCA", default="random", choices=["random", "pca"])
    p.add_argument("--epsDBSCAN", type=float, default=10)
    p.add_argument("--kClusters", type=int, default=2)
    p.add_argument("--seed", default=None)
    p.add_argument("--chrmlist", default=None, nargs="+")
    p.add_argument("--updateHMM", action="store_true", default=False)
    p.add_argument("--updateWin", type=int, default=1000)
    p.add_argument("--updateInc", type=int, default=500)
    p.add_argument("--findSelf", action="store_true", default=False)
    p.add_argument("--quiet", action="store_true", default=False, help="(frisk_b200) do not echo every window row to stdout")
    args = p.parse_args(argv)
    if args.minWordSize > args.maxWordSize:                             # F:1395-1397
        logging.error("[ERROR] Minimum kmer size (-m/--minWordSize) must be less than Maximum kmer size (-k/--maxWordSize)\n")
        sys.exit(1)
    return args


def main(argv=None):
    """Stages 1-3 of the reference's main() (F:1400-1507): genome k-mer tables, window scores, their
    caches and the raw TSV.  The downstream stages (thresholds, HMM, projection, plots: F:1509-1851)
    consume the DataFrame / TSV written here and are outside this package."""
    import pandas as pd
    logging.basicConfig(level=logging.INFO, format="%(asctime)s - %(funcName)s - %(message)s")
    args = mainArgs(argv)
    print("frisk --", FRISK_VERSION)
    genomepickle = makePicklePath(args, space="genome")
    windowsPickle = makePicklePath(args, space="window")
    tempPathCheck(args)
    with_rip = bool(args.RIP) and args.minWordSize <= 2          # F:1467 (calcRIP itself needs maxWordSize >= 2, F:478)
    if with_rip and args.maxWordSize < 2:
        raise ValueError("2 is not in list")                        # what range(...).index(2) raises at F:478

    have_genome = os.path.isfile(genomepickle) and args.recalc      # F:1437
    have_windows = os.path.isfile(windowsPickle) and args.recalcWin  # F:1454
    res = None
    if have_genome:
        logging.info("Importing previously calculated genome kmers from %s" % genomepickle)
        with open(genomepickle, "rb") as fh:
            genomeKmers = pickle.load(fh)
    if not have_genome or not have_windows:
        if have_genome:                                             # the windows against the stored tables (F:1437)
            try:                                                    # orders -m..-k of 4^k words + meta, before any device work
                background = engine.genome_kmers_tables(genomeKmers, args.minWordSize, args.maxWordSize)
            except ValueError as e:
                logging.error("[ERROR] %s: %s" % (genomepickle, e))
                sys.exit(1)
            res = score_background(args, background, genomepickle)
        else:
            logging.info("Calculating kmers for host sequence: %s" % args.hostSeq)
            res = score_genome(args)                                # one GPU pass produces both products
    if not have_genome:
        genomeKmers = genome_kmers_from_result(res)
        with open(genomepickle, "wb") as fh:
            pickle.dump(genomeKmers, fh, protocol=2)                # F:363 (protocol 2: readable by a py2 frisk)
        if args.exitAfter == "GenomeKmers":                         # F:1443-1445
            logging.info("Finished counting kmers. Exiting.")
            sys.exit(0)
        logging.info("Finished counting kmers.")

    if have_windows:
        logging.info("Importing previously calculated window KLD scores from: %s" % windowsPickle)
        allWindows = pd.read_pickle(windowsPickle)
        if "windowKLD" not in allWindows.columns:                   # F:1458-1459
            allWindows["windowKLD"] = allWindows["windowKLI"]
    else:
        allWindows = windows_frame(res, with_rip)
        outPath = os.path.join(args.tempDir, args.outfile)
        body = res.tsv_body(with_rip).decode()                      # the rows exactly as str() prints them, formatted in C
        with open(outPath, "w") as handle:                          # F:1463-1497
            handle.write("\t".join(allWindows.columns.values) + "\n")
            handle.write(body)
        if not args.quiet:
            sys.stdout.write(body)                                  # F:1494
        logging.info("Saving calculated window KLD scores as: %s" % windowsPickle)
        allWindows.to_pickle(windowsPickle, protocol=2)             # F:1501
        if args.exitAfter == "WindowKLD":                           # F:1503-1505
            logging.info("Finished calculating window KLD scores. Exiting.")
            sys.exit(0)
        logging.info("Finished calculating window KLD scores.")
    if args.hmmKLD:                                                 # F:1536-1548: 2-state HMM over the window scores
        from . import downstream
        model = downstream.fit_hmm(allWindows["windowKLD"].to_numpy(dtype=float))
        hmmBED, allWindows = downstream.hmm2BED(allWindows, model, dataCol="windowKLD")
        with open(os.path.join(args.tempDir, args.hmmOutfile), "w") as handle:
            for line in downstream.hmmBED2GFF(hmmBED):
                handle.write(line)
        logging.info("Wrote %d HMM state intervals to %s" % (len(hmmBED), os.path.join(args.tempDir, args.hmmOutfile)))
    logging.info("frisk_b200 covers the hot path only; thresholding / HMM / projection / graphics (reference "
                 "F:1509-1851) read %s and %s" % (os.path.join(args.tempDir, args.outfile), windowsPickle))
    return allWindows
