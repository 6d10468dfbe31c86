"""`epilogos` command line for the B200 scoring path (mirror of the reference's run.py:18-325, local mode).

The option set, defaults, validation messages and the output-file naming rule (run.py:158-165) are the
reference's.  What differs is the execution model: there is no SLURM fan-out (run.py:454-585) -- the stages run in
this process on the GPU, and across GPUs when the command is launched under torchrun
(`torchrun --nproc-per-node 8 -m epilogos_b200.run -i ... -l`), where every stage shards the rows of each file over
the ranks.  `-l` is therefore accepted but not required; `-x`, `-p` and the `--*-mem` options are accepted and
ignored with a note.  Step 4 selects the regions of interest: epilogos_b200.roi in single mode, and in paired mode
epilogos_b200.roi_pairwise, which also fits the null distribution and writes p-values with -n (the statistics of
roiAndVisualPairwise.py; its -d figures are not built).
"""
import csv
import errno
import os
import sys
from pathlib import Path

import click


def getNumStates(stateFile):
    """Number of data rows of the state-model TSV (helpers.py:9-17)."""
    with open(Path(stateFile), newline="") as f:
        return max(sum(1 for row in csv.reader(f, delimiter="\t") if row) - 1, 0)


def getStateNames(stateFile):
    """`short_name` column of the state-model TSV (helpers.py:20-28)."""
    with open(Path(stateFile), newline="") as f:
        return [row["short_name"] for row in csv.DictReader(f, delimiter="\t")]


def _die(message):
    print(message)
    sys.exit()


def checkFlags(mode, commandLineBool, inputDirectory, inputDirectory1, inputDirectory2, outputDirectory, stateInfo,
               exitBool, diagnosticBool, partition, pvalBool):
    """Required / incompatible flag combinations (run.py:328-375): first violated rule prints and exits."""
    required = [
        (mode == "single" and not inputDirectory, "ERROR: [-i, --input-directory] required in 'single' group mode"),
        (mode == "paired" and not inputDirectory1, "ERROR: [-a, --directory-one] required in 'paired' group mode"),
        (mode == "paired" and not inputDirectory2, "ERROR: [-b, --directory-two] required in 'paired' group mode"),
        (not outputDirectory, "ERROR: [-o, --output-directory] required"),
        (not stateInfo, "ERROR: [-n, --state-info] required"),
    ]
    incompatible = [
        (mode == "single" and inputDirectory1, "ERROR: [-m, --mode] 'single' not compatible with [-a, --directory-one] option"),
        (mode == "single" and inputDirectory2, "ERROR: [-m, --mode] 'single' not compatible with [-b, --directory-two] option"),
        (mode == "single" and diagnosticBool, "ERROR: [-m, --mode] 'single' not compatible with [-d, --diagnostic-figures] flag"),
        (mode == "single" and pvalBool, "ERROR: [-m, --mode] 'single' not compatible with [-n, --null-distribution] flag"),
        (mode == "paired" and inputDirectory, "ERROR: [-m, --mode] 'paired' not compatible with [-i, --input-directory] option"),
        (commandLineBool and exitBool, "ERROR: [-l, --cli] flag not compatible with [-x, --exit] flag"),
        (commandLineBool and partition, "Error: [-l, --cli] flag not compatible with [-p, --partition] option"),
    ]
    for table in (required, incompatible):
        for bad, message in table:
            if bad:
                _die(message)
                return


def checkGroupFlags(mode, inputDirectory, inputDirectory1, inputDirectory2, fileTag, groupFile, comparisons,
                    multigroups=()):
    """Flag rules of --groups / --compare (checked before checkFlags): first violated rule prints and exits."""
    rules = [
        (comparisons and not groupFile, "ERROR: [--compare] requires [--groups]"),
        (groupFile and not inputDirectory, "ERROR: [--groups] requires [-i, --input-directory]"),
        (groupFile and inputDirectory1, "ERROR: [--groups] not compatible with [-a, --directory-one] option"),
        (groupFile and inputDirectory2, "ERROR: [--groups] not compatible with [-b, --directory-two] option"),
        (groupFile and fileTag != "null", "ERROR: [--groups] not compatible with [-f, --file-tag] option"),
        (comparisons and mode != "paired", "ERROR: [--compare] requires [-m, --mode] 'paired'"),
        (groupFile and mode == "paired" and not comparisons and not multigroups,
         "ERROR: [-m, --mode] 'paired' with [--groups] requires at least one [--compare]"),
    ]
    for bad, message in rules:
        if bad:
            _die(message)
            return


def checkArguments(mode, saliency, inputDirPath, inputDirPath2, outputDirPath, numProcesses, numStates, numTrials,
                   samplingSize, quiescentState, groupSize, roiWidth):
    """Value checks (run.py:378-451): same exceptions / messages."""
    if mode == "single" and saliency not in (1, 2, 3):
        raise ValueError("Saliency Metric Invalid: {}".format(saliency)
                         + "Please ensure that saliency metric is either 1, 2, or 3")
    if mode == "paired" and saliency not in (1, 2):
        raise ValueError("Saliency Metric Invalid: {}".format(saliency)
                         + "Please ensure that saliency metric is either 1 or 2 "
                         + "(Saliency of 3 is unsupported for pairwise comparison")
    for d in [inputDirPath] + ([inputDirPath2] if mode == "paired" else []):
        if not d.exists():
            raise FileNotFoundError("Given path does not exist: {}".format(str(d)))
        if not d.is_dir():
            raise NotADirectoryError("Given path is not a directory: {}".format(str(d)))
        if not list(d.glob("*")):
            raise OSError(errno.ENOTEMPTY, "Ensure given directory is not empty", str(d))
    if not outputDirPath.exists():
        outputDirPath.mkdir(parents=True, exist_ok=True)
    if not outputDirPath.is_dir():
        raise NotADirectoryError("Given path is not a directory: {}".format(str(outputDirPath)))
    checks = [
        (numProcesses < 0, "ERROR: Number of cores must be positive or zero (0 means use all cores)"),
        (numTrials <= 0, "ERROR: Number of trials must be greater than zero"),
        (samplingSize <= 0, "ERROR: Sampling size must be greater than zero"),
        (quiescentState < -1, "ERROR: Quiescent state value must be positive or zero (0 means do not filter)"),
        (quiescentState >= numStates, "ERROR: Quiescent state value must be a state provided in the state model"),
        (groupSize < -1, "ERROR: Group size value must be positive or -1 (-1 means use inputted group sizes)"),
        (roiWidth < 0, "ERROR: Group size value must be greater than 0"),
    ]
    for bad, message in checks:
        if bad:
            _die(message)
            return


MAX_NULL_PERMUTATIONS = 1000000


def checkPermutationFlags(mode, nullPermutations):
    """Rules of --null-permutations (checked after every other rule): first violated rule prints and exits."""
    rules = [
        (nullPermutations is not None and mode != "paired",
         "ERROR: [--null-permutations] requires [-m, --mode] 'paired'"),
        (nullPermutations is not None and not 1 <= nullPermutations <= MAX_NULL_PERMUTATIONS,
         "ERROR: Number of null permutations must be between 1 and {}".format(MAX_NULL_PERMUTATIONS)),
    ]
    for bad, message in rules:
        if bad:
            _die(message)
            return


def checkRegionPermutationFlags(mode, roiPermutations, groupSize, roiWidth):
    """Rules of --roi-permutations (checked after every other rule): first violated rule prints and exits."""
    from .region_null import MAX_PERMUTATIONS, MAX_WINDOW
    if roiPermutations is None:
        return
    rules = [
        (mode != "paired", "ERROR: [--roi-permutations] requires [-m, --mode] 'paired'"),
        (not 1 <= roiPermutations <= MAX_PERMUTATIONS,
         "ERROR: Number of region permutations must be between 1 and {}".format(MAX_PERMUTATIONS)),
        (groupSize != -1, "ERROR: [--roi-permutations] not compatible with [-g, --group-size] option"),
        (roiWidth > MAX_WINDOW,
         "ERROR: [--roi-permutations] needs a region width [-w, --roi-width] of at most {} bins".format(MAX_WINDOW)),
    ]
    for bad, message in rules:
        if bad:
            _die(message)
            return


def checkMultigroupFlags(mode, groupFile, multigroups, groupSet, pvalBool, groupSize):
    """Rules of --multigroup (checked after every other rule): first violated rule prints and exits.  Returns the
    comparisons, each a tuple of group names."""
    if not multigroups:
        return []
    rules = [
        (not groupFile, "ERROR: [--multigroup] requires [--groups]"),
        (mode != "paired", "ERROR: [--multigroup] requires [-m, --mode] 'paired'"),
    ]
    for bad, message in rules:
        if bad:
            _die(message)
            return []
    from . import groups as _groups
    try:
        out = _groups.parseMultigroups(multigroups, groupSet)
    except _groups.GroupFileError as exc:
        _die(str(exc))
        return []
    for bad, message in ((pvalBool, "ERROR: [--multigroup] not compatible with [-n, --null-distribution] flag"),
                         (groupSize != -1, "ERROR: [--multigroup] not compatible with [-g, --group-size] option")):
        if bad:
            _die(message)
            return []
    return out


def checkStrataFlags(mode, strataFile, groupSize):
    """Rules of --strata (checked after every other rule): first violated rule prints and exits.  Returns the
    groups.Strata of the file, or None without --strata."""
    if not strataFile:
        return None
    for bad, message in ((mode != "paired", "ERROR: [--strata] requires [-m, --mode] 'paired'"),
                         (groupSize != -1, "ERROR: [--strata] not compatible with [-g, --group-size] option")):
        if bad:
            _die(message)
            return None
    from . import groups as _groups
    try:
        return _groups.parseStrata(strataFile)
    except _groups.GroupFileError as exc:
        _die(str(exc))
        return None


def deal_files(pairs, world):
    """Whole files dealt to the ranks, largest first to the least loaded rank (by size on disk): the same answer on every
    rank.  Returns a list of `world` lists of (file1, file2) pairs."""
    sizes = [Path(f).stat().st_size + (Path(f2).stat().st_size if str(f2) != "null" else 0) for f, f2 in pairs]
    order = sorted(range(len(pairs)), key=lambda i: (-sizes[i], str(pairs[i][0])))
    load = [0] * world
    out = [[] for _ in range(world)]
    for i in order:
        r = min(range(world), key=lambda q: (load[q], q))
        out[r].append(pairs[i])
        load[r] += sizes[i]
    return [sorted(part, key=lambda pr: str(pr[0])) for part in out]


def run_stages(pairs, mode, numStates, saliency, outputDirPath, fileTag, storedExpPath, numProcesses, quiescentState,
               groupSize, stateInfo, roiWidth, verbose, say, backend=None, pvalBool=False, numTrials=101,
               samplingSize=100000, diagnosticBool=False, groups=None, permutations=0, region_permutations=0, strata=None):
    """Steps 1-4 of run.main (run.py:193-303) in process.  Two ways to use several GPUs:
      rows  (default)  every file's rows are split over the ranks (helpers.splitRows); per-file tables are all-reduced and
                       score rows gathered on rank 0, which writes the files;
      files (EPILOGOS_B200_SHARD=files, needs at least as many files as ranks)  whole files are dealt to the ranks, which
                       run the unsharded stages on them and write their own outputs; the ranks meet at the barriers between
                       the stages and the per-file count tables are combined from the files, as the reference's SLURM jobs
                       do.  No file is inflated or parsed by more than one rank, and the text is written in parallel.
    Integer tables make both identical to a single-rank run.
    `groups` (a --groups run): a list of (outputDirPath, fileTag, storedExpPath, groups.Selection), one per group (single
    mode) or comparison (paired mode), run on the column subsets of the files of `pairs`, which are (file, "null").  Every
    stage keeps the reference's order: step 1 tables all groups of a file from the same counts, step 2 runs per group, step
    3 scores all groups of a file, step 4 runs per group.  A comparison passes the file itself as the stage drivers'
    second file, which the group view does not read.
    `permutations` P > 0 (paired mode): step 3 also counts P null shuffles per bin and step 4 writes
    pairwisePermutation_<tag>.txt.gz.  A multi-group comparison (a Selection with `multi`, --multigroup) scores its groups
    in step 3 (epilogos_b200.multigroup), counting P shuffles per bin when P > 0, and step 4 runs
    epilogos_b200.roi_multigroup.
    `region_permutations` P > 0 (paired mode): step 3 also finds every file's maxima of the region null over P label
    splits drawn from one seed per run, and step 4 writes regionPermutation_<tag>.txt and regionNullMaxima_<tag>.npz
    (epilogos_b200.region_null).
    `strata` (groups.Strata, paired mode): every null of step 3 shuffles biosample labels only within strata."""
    from contextlib import nullcontext
    from . import dist, expected, expectedCombination, scores, session
    world = dist.world_size()
    by_file = os.environ.get("EPILOGOS_B200_SHARD", "rows") == "files" and world > 1 and len(pairs) >= world
    mine = deal_files(pairs, world)[dist.rank()] if by_file else pairs
    alone = dist.solo if by_file else nullcontext
    if by_file:
        say("        Input files dealt to the ranks: {} files over {} GPUs".format(len(pairs), world))

    runs = groups or [(outputDirPath, fileTag, storedExpPath, None)]
    for out, _, _, _ in runs:
        Path(out).mkdir(parents=True, exist_ok=True)

    def second(f, f2, sel):
        return f if sel is not None and sel.paired else f2

    with alone():
        session.prefetch(mine, numStates, backend)       # parse all files concurrently, once (the stages re-use them)
    say("\nSTEP 1: Per data file background frequency calculation")
    with alone():
        for f, f2 in mine:
            for out, tag, _, sel in runs:
                expected.main(f, second(f, f2, sel), numStates, saliency, out, tag, numProcesses, verbose, backend=backend,
                              group=sel)
    dist.barrier()
    say("\nSTEP 2: Background frequency combination")
    for out, tag, exp_path, _ in runs:
        expectedCombination.main(out, exp_path, tag, verbose, backend=backend)
    region_seed = None
    if region_permutations > 0:
        # one seed for every file, rank and sharding mode: drawn here, by every rank together, outside dist.solo()
        from . import pairwise, region_null
        region_seed = region_null.region_seed(pairwise.run_seed())
    say("\nSTEP 3: Score calculation")
    # step 4 runs in this process right after: rank 0 hands its score arrays over in memory instead of through
    # temp_scores_*.npz (files written by other ranks, when whole files are dealt, are still read from disk)
    try:
        from . import roi as _roi_stage          # noqa: F401
        roi_here = dist.group_rank() == 0
    except ImportError:
        roi_here = False
    session.handover_enabled = roi_here
    try:
        with alone():
            for f, f2 in mine:
                for out, tag, exp_path, sel in runs:
                    scores.main(f, second(f, f2, sel), numStates, saliency, out, exp_path, tag, numProcesses,
                                quiescentState, groupSize, verbose, backend=backend, group=sel,
                                permutations=permutations, region_permutations=region_permutations,
                                region_seed=region_seed, roi_width=roiWidth, strata=strata)
    finally:
        session.handover_enabled = False
    dist.barrier()
    if mode == "single":
        say("\nSTEP 4: Finding regions of interest")
        try:
            from . import roi
        except ImportError:
            roi = None
        if roi is None:
            say("    (region-of-interest selection is not part of this build; temp_scores_*.npz kept for roiSingle)")
        elif dist.rank() == 0:
            for out, tag, exp_path, _ in runs:
                roi.main(out, stateInfo, tag, exp_path, roiWidth, verbose)
    else:
        from . import pairwise, roi_multigroup, roi_pairwise
        seed = pairwise.run_seed() if pvalBool else None      # every rank takes part in drawing a fresh seed
        say("\nSTEP 4: " + ("Fitting the null distribution, p-values and regions of interest" if pvalBool
                            else "Pairwise metrics and regions of interest"))
        if dist.rank() == 0:
            for out, tag, exp_path, sel in runs:
                if sel is not None and sel.multi is not None:
                    roi_multigroup.main(out, stateInfo, tag, exp_path, roiWidth, verbose, backend=backend)
                    continue
                roi_pairwise.main(out, stateInfo, tag, exp_path, roiWidth, pvalBool, numTrials, samplingSize,
                                  diagnosticBool, verbose, backend=backend, seed=seed)


@click.command(context_settings=dict(help_option_names=["-h", "--help"]))
@click.option("-m", "--mode", "mode", type=click.Choice(["single", "paired"]), default="single", show_default=True,
              help="single for single group epilogos and paired for 2 group epilogos")
@click.option("-l", "--local", "commandLineBool", is_flag=True,
              help="Run in this process (always the case here: the GPU path has no SLURM mode)")
@click.option("-i", "--input-directory", "inputDirectory", type=str,
              help="Path to directory that contains files to read from (ALL files in this directory will be read in)")
@click.option("-a", "--directory-one", "inputDirectory1", type=str, help="First input directory (paired)")
@click.option("-b", "--directory-two", "inputDirectory2", type=str, help="Second input directory (paired)")
@click.option("-o", "--output-directory", "outputDirectory", type=str,
              help="Output Directory (CANNOT be the same as input directory)\n")
@click.option("-j", "--state-info", "stateInfo", type=str, help="State model info file")
@click.option("-s", "--saliency", "saliency", type=int, default=1, show_default=True,
              help="Desired saliency level (1, 2, or 3)")
@click.option("-c", "--num-cores", "numProcesses", type=int, default=1,
              help="Accepted for compatibility; parallelism comes from the GPUs of the torchrun launch")
@click.option("-x", "--exit", "exitBool", is_flag=True, help="SLURM-only flag of the reference (ignored)")
@click.option("-d", "--diagnostic-figures", "diagnosticBool", is_flag=True,
              help="Paired mode diagnostic figures (not built here: matplotlib is not a dependency; a note is printed)")
@click.option("-t", "--num-trials", "numTrials", type=int, default=101, show_default=True,
              help="Paired mode with -n: the number of subsamples of the null distances that are fit (the median fit is used)")
@click.option("-z", "--sampling-size", "samplingSize", type=int, default=100000, show_default=True,
              help="Paired mode with -n: the size of each subsample of the null distances that is fit")
@click.option("-q", "--quiescent-state", "quiescentState", type=int, default=-1,
              help="If a bin contains only states of this value, it is treated as quiescent and not factored into "
                   + "fitting. If set to 0, filtering is not done. [default: last state]  No effect on a --multigroup "
                   + "comparison, which fits nothing")
@click.option("-g", "--group-size", "groupSize", type=int, default=-1, show_default=True,
              help="In pairwise epilogos controls the sizes of the shuffled arrays. "
                   + "Default is sizes of the input groups")
@click.option("-v", "--version", "version", is_flag=True, help="Print the version number and exit")
@click.option("-p", "--partition", "partition", type=str, help="SLURM-only option of the reference (ignored)")
@click.option("-n", "--null-distribution", "pvalBool", is_flag=True,
              help="Paired mode: fit the null distribution and add p-values and Benjamini-Hochberg adjusted p-values to "
                   + "pairwiseMetrics and regionsOfInterest")
@click.option("-w", "--roi-width", "roiWidth", type=int, default=0,
              help="The number of bins in a region of interest [default: 50(single)/125(paired)]")
@click.option("-f", "--file-tag", "fileTag", type=str, default="null",
              help="Tag to be appended in output filenames [default: input-directory_saliency]")
@click.option("--groups", "groupFile", type=str,
              help="Tab-separated file of biosample groups, one per line: name<TAB>columns (1-based biosample numbers and "
                   + "ranges a-b, comma-separated).  Runs every group (single mode) or every --compare (paired mode) on "
                   + "the column subsets of the files of -i, parsing each file once; outputs go to OUT/<group> or "
                   + "OUT/<A>_vs_<B>")
@click.option("--compare", "comparisons", type=str, multiple=True,
              help="Paired mode with --groups: compare group A with group B (A:B, repeatable)")
@click.option("--multigroup", "multigroups", type=str, multiple=True,
              help="Paired mode with --groups: one test per bin across the disjoint groups A,B,C,... (2 to 64, "
                   + "repeatable), written to OUT/A_B_C: multigroupMetrics_<tag>.txt.gz (per bin the size-weighted "
                   + "between-group sum of squares T of the group scores, the group and state that drive it, the sign, "
                   + "and with --null-permutations P the count of P label shuffles with a T as large, p and BH) and "
                   + "regionsOfInterest_<tag>.txt.  Not with -n or -g")
@click.option("--null-permutations", "nullPermutations", type=int, default=None,
              help="Paired mode: draw P null shuffles of every bin on the GPU and write pairwisePermutation_<tag>.txt.gz "
                   + "with each bin's count of shuffles at least as far apart as its groups, its permutation p-value "
                   + "(1 + count) / (P + 1) and the Benjamini-Hochberg adjusted p-value (1 <= P <= 1000000)")
@click.option("--roi-permutations", "roiPermutations", type=int, default=None,
              help="Paired mode: permute the biosample labels P times over the whole genome on the GPU and give every "
                   + "region of interest a family-wise p-value: the share of the P genome-wide maxima of the window sums "
                   + "that reach its own (regionPermutation_<tag>.txt, regionNullMaxima_<tag>.npz; 1 <= P <= 100000; "
                   + "not with -g)")
@click.option("--strata", "strataFile", type=str,
              help="Paired mode: tab-separated file of strata (tissue, donor, batch, ...) in the --groups format, "
                   + "name<TAB>columns; columns are numbered over [A | B] with -a/-b and as in the group file with "
                   + "--groups.  Every null (-n, --null-permutations, --multigroup p-values, --roi-permutations) then "
                   + "shuffles biosample labels only within strata, so each group keeps its make-up in every stratum.  "
                   + "Not with -g")
@click.option("--exp-freq-mem", "expFreqMem", type=int, default=20000, help="SLURM-only (ignored)")
@click.option("--exp-comb-mem", "expCombMem", type=int, default=8000, help="SLURM-only (ignored)")
@click.option("--score-mem", "scoreMem", type=int, default=40000, help="SLURM-only (ignored)")
@click.option("--roi-mem", "roiMem", type=int, default=-1, help="SLURM-only (ignored)")
def main(mode, commandLineBool, inputDirectory, inputDirectory1, inputDirectory2, outputDirectory, stateInfo, saliency,
         numProcesses, exitBool, diagnosticBool, numTrials, samplingSize, quiescentState, groupSize, version, partition,
         pvalBool, roiWidth, fileTag, groupFile, comparisons, multigroups, nullPermutations, roiPermutations, strataFile,
         expFreqMem, expCombMem, scoreMem, roiMem):
    """Information-theoretic navigation of multi-tissue functional genomic annotations (B200 scoring path)."""
    if version:
        from epilogos_b200 import __version__
        print("Version:", __version__)
        sys.exit()

    checkGroupFlags(mode, inputDirectory, inputDirectory1, inputDirectory2, fileTag, groupFile, comparisons, multigroups)
    if groupFile and mode == "paired":       # both groups of a comparison come from the files of -i
        inputDirectory, inputDirectory1, inputDirectory2 = None, inputDirectory, inputDirectory
    checkFlags(mode, commandLineBool, inputDirectory, inputDirectory1, inputDirectory2, outputDirectory, stateInfo,
               exitBool, diagnosticBool, partition, pvalBool)
    groupSet, pairs_of_groups = None, []
    if groupFile:
        from . import groups as _groups
        try:
            groupSet = _groups.parseGroups(groupFile)
            pairs_of_groups = _groups.parseComparisons(comparisons, groupSet)
        except _groups.GroupFileError as exc:
            _die(str(exc))
            return
    verbose = False
    numStates = getNumStates(stateInfo)
    # user-facing quiescent state is 1-based, 0 = no filtering (run.py:112-113)
    quiescentState = numStates - 1 if quiescentState == -1 else quiescentState - 1
    if roiWidth == 0:
        roiWidth = 50 if mode == "single" else 125                                       # run.py:116-117

    inputDirPath = Path(inputDirectory if mode == "single" else inputDirectory1).absolute()
    inputDirPath2 = Path(inputDirectory2).absolute() if mode == "paired" else Path("")
    outputDirPath = Path(outputDirectory).absolute()
    checkArguments(mode, saliency, inputDirPath, inputDirPath2, outputDirPath, numProcesses, numStates, numTrials,
                   samplingSize, quiescentState, groupSize, roiWidth)
    checkPermutationFlags(mode, nullPermutations)
    multi_of_groups = checkMultigroupFlags(mode, groupFile, multigroups, groupSet, pvalBool, groupSize)
    checkRegionPermutationFlags(mode, roiPermutations, groupSize, roiWidth)
    strata = checkStrataFlags(mode, strataFile, groupSize)

    import torch
    import torch.distributed as td
    launched = "RANK" in os.environ and "WORLD_SIZE" in os.environ
    if launched and not td.is_initialized():
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        from . import dist as _dist
        _dist.bind_to_gpu_numa(int(os.environ.get("LOCAL_RANK", "0")))
        td.init_process_group("nccl")
    from . import dist, expected, expectedCombination, scores
    lead = dist.rank() == 0

    def say(*a, **k):
        if lead:
            print(*a, **k, flush=True)

    if fileTag == "null":                                                                  # run.py:158-162
        fileTag = ("{}_s{}".format(inputDirPath.name, saliency) if mode == "single"
                   else "{}_{}_s{}".format(inputDirPath.name, inputDirPath2.name, saliency))
    storedExpPath = outputDirPath / "exp_freq_{}.npy".format(fileTag)

    say("\n\n\n        " + ("Single" if mode == "single" else "Paired") + " group epilogos on "
        + "{} GPU(s)".format(dist.world_size()))
    say("        Saliency level =", saliency, "  States =", numStates, "  Output =", str(outputDirPath))
    if mode == "paired":
        say("        Quiescent State =", "No quiescent filtering" if quiescentState == -1 else quiescentState + 1)
    if strata is not None:
        say("        " + strata.summary())

    files = sorted(p for p in inputDirPath.glob("*"))
    pairs = []
    runs = None
    if groupSet is not None:
        # every group / comparison behaves like a run on its column-subset files in a directory named after it
        sel = ([(g, "{}_s{}".format(g, saliency), groupSet.select(g)) for g in groupSet.names] if mode == "single" else
               [("{}_vs_{}".format(a, b), "{}_{}_s{}".format(a, b, saliency), groupSet.select(a, b))
                for a, b in pairs_of_groups] +
               [("_".join(m), "{}_s{}".format("_".join(m), saliency), groupSet.select_multi(m)) for m in multi_of_groups])
        runs = [(outputDirPath / d, tag, outputDirPath / d / "exp_freq_{}.npy".format(tag), s) for d, tag, s in sel]
    for f in files:
        if runs is not None:
            pairs.append((f, "null"))
            continue
        if mode == "single":
            pairs.append((f, "null"))
        else:
            match = inputDirPath2 / f.name
            if not match.exists():
                raise FileNotFoundError("File not found: {}".format(str(match))
                                        + "Please ensure corresponding files within input directories "
                                        + "directories 1 and 2 have the same name")
            pairs.append((f, match))

    run_stages(pairs, mode, numStates, saliency, outputDirPath, fileTag, storedExpPath, numProcesses, quiescentState,
               groupSize, stateInfo, roiWidth, verbose, say, pvalBool=pvalBool, numTrials=numTrials,
               samplingSize=samplingSize, diagnosticBool=diagnosticBool, groups=runs,
               permutations=nullPermutations or 0, region_permutations=roiPermutations or 0, strata=strata)
    dist.barrier()
    if launched and td.is_initialized():
        td.destroy_process_group()


if __name__ == "__main__":
    main()
