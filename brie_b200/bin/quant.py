"""brie-quant: quantify splicing isoforms and detect variable splicing events associated
with cell features -- same flags, defaults and outputs as brie/bin/quant.py:13-219, with the
fit running on libbrie_b200.so instead of TensorFlow."""
import os
import sys
import numpy as np
from optparse import OptionParser, OptionGroup

import brie_b200
from brie_b200.utils import io_utils
from brie_b200.utils.base_utils import match
from brie_b200.utils.preprocessing import filter_genes


def _init_distributed():
    """(rank, world).  Under torchrun (WORLD_SIZE > 1 in the environment) join the NCCL process
    group with this rank's GPU as the current device; otherwise a single process."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world <= 1:
        return 0, 1
    import torch
    import torch.distributed as dist
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return dist.get_rank(), world


def _read_table(path):
    delim = "," if path.endswith('csv') or path.endswith('csv.gz') else "\t"
    return np.genfromtxt(path, dtype="str", delimiter=delim)


def quant(in_file, cell_file=None, gene_file=None, out_file=None,
          LRT_index=[], layer_keys=['isoform1', 'isoform2', 'ambiguous'],
          intercept=None, intercept_mode='gene', nproc=1, min_counts=50,
          min_counts_uniq=10, min_cells_uniq=30, min_MIF_uniq=0.001,
          min_iter=5000, max_iter=20000, MC_size=1, batch_size=500000,
          pseudo_count=0.01, base_mode='full', seed=0, out_dir=None, resume=False, n_perm=0, wald=False,
          score_file=None, LRT_groups=None, wald_groups=None, score_groups=None):
    """CLI driver (quant.py:13-130).  `nproc` is accepted for compatibility (host threads are
    not on the hot path any more); `seed` keys the counter-based noise (new, default 0).
    `out_dir` (new): directory for `.npy` memory maps of the dense (cells, events) output layers
    Psi / Psi_95CI / Z_std, written event chunk by event chunk and rank by rank -- the reference keeps
    them dense in RAM (model_wrap.py:289-292, "TODO: introduce sparse matrix for this"), 80 GB each at
    1M x 20k; the output container then references the maps instead of embedding the arrays.  Under
    torchrun it defaults to `<out_file stem>.layers/`, so no (cells, events) array ever travels through a
    collective.  `resume` (new, needs out_dir): skip the event chunks a previous run of the same fit left
    there (checkpoint / restart).  `n_perm` (new): permutation replicates per tested covariate; adds the
    pooled permutation p-values and their FDR to the container (varm) and the table (fitBRIE).  `wald`
    (new): standard errors, Wald p-values and their FDR for every cell coefficient, from the fitted
    posterior without refits (fitBRIE); in the container (varm) and the table.  `score_file` (new): a table laid out
    like `cell_file` (cell ids, then one candidate covariate per column) whose candidates are score-tested against
    the fitted model without refits (fitBRIE's score_X); every fitted cell must be in it.  Results go to the
    container (varm, uns['score_ids']) and to <out>.brie_score.tsv.  `LRT_groups`, `wald_groups` (new): groups of
    `cell_file` columns tested jointly by refits and from the fitted posterior; `score_groups` (new): groups of
    `score_file` columns tested jointly (fitBRIE); results go to the container and the tables.

    Multi-GPU: launch one process per GPU (`python -m torch.distributed.run --nproc-per-node N
    -m brie_b200.bin.quant ...`); every rank reads the input, fits its own event shard
    (fitBRIE) and rank 0 writes the outputs."""
    rank, world = _init_distributed()
    if out_file is None:
        print("No given out_file, use the dir for input file.")
        out_file = os.path.dirname(os.path.abspath(in_file)) + "/brie_quant.h5ad"
    os.makedirs(os.path.dirname(os.path.abspath(out_file)), exist_ok=True)
    if out_dir is None and world > 1:
        out_dir = ".".join(os.path.abspath(out_file).split('.')[:-1]) + ".layers"
    if resume and out_dir is None:
        print("[BRIE2] Error: --resume needs --outDir.")
        sys.exit(1)

    if in_file.endswith(".h5ad"):
        adata = io_utils.read_h5ad(in_file)
    elif in_file.endswith(".npz"):
        adata = io_utils.read_npz(in_file)
    else:
        print("[BRIE2] Error: input needs to be .h5ad or .npz")
        sys.exit(1)

    Xc, Xc_ids = None, None
    if cell_file is not None:                                    # quant.py:47-66
        tab = _read_table(cell_file)
        idx = match(adata.obs.index, tab[1:, 0]).astype(float)
        mm1 = idx == idx
        mm2 = idx[mm1].astype(int)
        print("[BRIE2] %.1f%% cells are matched with features" % (np.mean(mm1) * 100))
        Xc = tab[mm2 + 1, 1:].astype(np.float32)
        Xc_ids = tab[0, 1:]
        adata = adata[mm1, :]

    score_X, score_ids = None, None
    if score_file is not None:
        tab = _read_table(score_file)
        idx = match(adata.obs.index, tab[1:, 0]).astype(float)
        if not (idx == idx).all():
            print("[BRIE2] Error: %d of %d cells are missing from --scoreFile." % ((idx != idx).sum(), len(idx)))
            sys.exit(1)
        score_X = tab[idx.astype(int) + 1, 1:].astype(np.float32)
        score_ids = tab[0, 1:]
        print("[BRIE2] %d candidate covariates for score tests" % len(score_ids))

    print("layers:", layer_keys)                                 # quant.py:69-75
    import torch
    adata = filter_genes(adata, min_counts=min_counts, min_counts_uniq=min_counts_uniq,
                         min_cells_uniq=min_cells_uniq, min_MIF_uniq=min_MIF_uniq,
                         uniq_layers=layer_keys[:2], ambg_layers=layer_keys[2:], copy=True,
                         device="cuda" if torch.cuda.is_available() else None)

    Xg, Xg_ids = None, None
    if gene_file is not None:                                    # quant.py:78-98
        tab = _read_table(gene_file)
        idx = match(adata.var.index, tab[1:, 0]).astype(float)
        mm1 = idx == idx
        mm2 = idx[mm1].astype(int)
        print("[BRIE2] %.1f%% genes are matched with features" % (np.mean(mm1) * 100))
        Xg = tab[mm2 + 1, 1:].astype(np.float32)
        Xg_ids = tab[0, 1:]
        adata = adata[:, mm1]

    print(adata)
    tau_prior = [1, 1] if 'unspliced' in adata.layers else [3, 27]     # quant.py:102-105 (unused downstream)

    from brie_b200.models import fitBRIE
    from brie_b200.models.model_wrap import check_groups
    n_cols = 0 if Xc is None else Xc.shape[1]
    for flag, groups, n in (("--LRTgroups", LRT_groups, n_cols), ("--waldGroups", wald_groups, n_cols),
                            ("--scoreGroups", score_groups, 0 if score_X is None else score_X.shape[1])):
        try:
            check_groups(groups, n, flag)
        except ValueError as e:
            print("[BRIE2] Error: %s (columns of %s)." % (e, "--scoreFile" if flag == "--scoreGroups" else "-c"))
            sys.exit(1)
    groups = {k: v for k, v in (('LRT_groups', LRT_groups), ('wald_groups', wald_groups),
                                 ('score_groups', score_groups)) if v is not None}
    fitBRIE(adata, Xc=Xc, Xg=Xg, LRT_index=LRT_index, layer_keys=layer_keys,
            intercept=intercept, intercept_mode=intercept_mode,
            min_iter=min_iter, max_iter=max_iter, MC_size=MC_size, batch_size=batch_size,
            pseudo_count=pseudo_count, base_mode=base_mode, tau_prior=tau_prior, seed=seed, n_perm=n_perm, wald=wald,
            score_X=score_X, **groups, **(dict(out_dir=out_dir, resume=resume, out_keys=('Psi', 'Psi95CI', 'Z_std')) if out_dir is not None else {}))

    adata.uns['brie_version'] = brie_b200.__version__
    adata.uns['Xc_ids'] = Xc_ids
    adata.uns['Xg_ids'] = Xg_ids
    if score_ids is not None:
        adata.uns['score_ids'] = score_ids

    if rank != 0:                                                # every rank holds the full result; one writes it
        return adata
    if hasattr(adata, 'write_npz') and not io_utils._anndata:    # no anndata/h5py here: npz container
        out_file = ".".join(out_file.split('.')[:-1]) + '.npz' if out_file.endswith('.h5ad') else out_file
        adata.write_npz(out_file)
    else:
        adata.write_h5ad(out_file)

    out_table_file = ".".join(out_file.split('.')[:-1]) + '.brie_ident.tsv'
    df = io_utils.dump_results(adata)
    df.to_csv(out_table_file, sep='\t', header=True, index=True, index_label='GeneID', float_format='%.3e')
    if score_ids is not None:
        io_utils.score_table(adata).to_csv(".".join(out_file.split('.')[:-1]) + '.brie_score.tsv', sep='\t',
                                           header=True, index=True, index_label='GeneID', float_format='%.3e')
    return adata


def main():
    parser = OptionParser()
    parser.add_option("--inFile", "-i", dest="in_file", default=None,
        help="Input read count matrices in AnnData h5ad or brie npz format.")
    parser.add_option("--cellFile", "-c", dest="cell_file", default=None,
        help=("File for cell features in tsv[.gz] with cell and feature ids."))
    parser.add_option("--geneFile", "-g", dest="gene_file", default=None,
        help=("File for gene features in tsv[.gz] with gene and feature ids."))
    parser.add_option("--out_file", "-o", dest="out_file", default=None,
        help="Full path of output file for annData in h5ad [default: $inFile/brie_quant.h5ad]")
    parser.add_option("--LRTindex", dest="LRT_index", default="None",
        help="Index (0-based) of cell features to test with LRT: All, None "
             "or comma separated integers [default: %default]")
    parser.add_option("--testBase", dest="test_base", default="full",
        help="Features in testing base model: full, null  [default: %default]")
    parser.add_option("--interceptMode", dest="intercept_mode", default="None",
        help="Intercept mode: gene, cell or None [default: %default]")
    parser.add_option("--layers", dest="layers", default="isoform1,isoform2,ambiguous",
        help="Comma separated layers two or three for estimating Psi [default: %default]")

    group1 = OptionGroup(parser, "Gene filtering")
    group1.add_option("--minCount", type="int", dest="min_count", default=50,
        help="Minimum total counts for fitltering genes [default: %default]")
    group1.add_option("--minUniqCount", type="int", dest="min_uniq_count", default=10,
        help="Minimum unique counts for fitltering genes [default: %default]")
    group1.add_option("--minCell", type="int", dest="min_cell", default=30,
        help="Minimum number of cells with unique count for fitltering genes [default: %default]")
    group1.add_option("--minMIF", type="float", dest="min_MIF", default=0.001,
        help="Minimum minor isoform frequency in unique count [default: %default]")

    group2 = OptionGroup(parser, "VI Optimization")
    group2.add_option("--MCsize", type="int", dest="MC_size", default=3,
        help="Sample size for Monte Carlo Expectation [default: %default]")
    group2.add_option("--minIter", type="int", dest="min_iter", default=5000,
        help="Minimum number of iterations [default: %default]")
    group2.add_option("--maxIter", type="int", dest="max_iter", default=20000,
        help="Maximum number of iterations [default: %default]")
    group2.add_option("--batchSize", type=int, dest="batch_size", default=500000,
        help="Element size per batch: n_gene * total cell [default: %default]")
    group2.add_option("--pseudoCount", type=float, dest="pseudo_count", default=0.01,
        help="Pseudo count to add on unique count matrices [default: %default]")
    group2.add_option("--nproc", "-p", type=int, dest="nproc", default=6,
        help="Number of processes for computing [default: %default]")
    group2.add_option("--seed", type=int, dest="seed", default=0,
        help="Key of the counter-based MC noise and initial values [default: %default]")
    group3 = OptionGroup(parser, "Large outputs (not in the reference)")
    group3.add_option("--outDir", dest="out_dir", default=None,
        help="Directory for .npy memory maps of the dense output layers Psi, Psi_95CI, Z_std (written "
             "chunk by chunk; the output file references them) [default: in RAM; <out_file>.layers under torchrun]")
    group3.add_option("--resume", action="store_true", dest="resume", default=False,
        help="With --outDir: skip the event chunks a previous run of the same fit has finished")
    group4 = OptionGroup(parser, "Calibration (not in the reference)")
    group4.add_option("--nPerm", type=int, dest="n_perm", default=0,
        help="Permutation replicates per tested feature: refit the model with that feature's cells permuted "
             "--nPerm times and add p-values against the permutation null pooled over all events, with their "
             "FDR (columns <feature>_pval_perm, <feature>_FDR_perm) [default: %default]")
    group4.add_option("--wald", action="store_true", dest="wald", default=False,
        help="Standard errors and Wald p-values of every cell coefficient from the fitted posterior, without "
             "refits, with their FDR over all events (columns <feature>_se, <feature>_pval_wald, "
             "<feature>_FDR_wald); covers every feature, also those not in --LRTindex")
    group4.add_option("--scoreFile", dest="score_file", default=None,
        help="Candidate cell covariates in tsv[.gz] laid out like --cellFile (cell ids, then one candidate per "
             "column), score-tested against the fitted model from its posterior without refits; every fitted cell "
             "must be in it.  Writes <out>.brie_score.tsv (columns <id>_score_z, <id>_pval_score, <id>_FDR_score)")
    group4.add_option("--LRTgroups", dest="LRT_groups", default=None,
        help="Groups of cell features (0-based columns of --cellFile) to test jointly with one refit per group, e.g. "
             "the indicator columns of a categorical: ';'-separated groups of ','-separated indices, e.g. \"1,2,3;4,5\" "
             "(columns <id>+<id>_ELBO_gain_group, _pval_group, _FDR_group)")
    group4.add_option("--waldGroups", dest="wald_groups", default=None,
        help="Groups of fitted cell features to test jointly with Wald tests from the fitted posterior, without "
             "refits; same syntax as --LRTgroups (columns <id>+<id>_pval_wald_group, _FDR_wald_group)")
    group4.add_option("--scoreGroups", dest="score_groups", default=None,
        help="Groups of --scoreFile columns to score-test jointly; same syntax as --LRTgroups (columns "
             "<id>+<id>_score_stat_group, _pval_score_group, _FDR_score_group in <out>.brie_score.tsv)")
    parser.add_option_group(group1)
    parser.add_option_group(group2)
    parser.add_option_group(group3)
    parser.add_option_group(group4)

    (options, args) = parser.parse_args()
    if len(sys.argv[1:]) == 0:
        print("Welcome to brie-quant in BRIE v%s!\n" % (brie_b200.__version__))
        print("use -h or --help for help on argument.")
        sys.exit(1)
    if options.in_file is None:
        print("[BRIE2] Error: need --h5adFile for count matrices in annData.")
        sys.exit(1)

    if options.LRT_index.upper() == "NONE":                      # quant.py:198-203
        LRT_index = []
    elif options.LRT_index.upper() == "ALL":
        LRT_index = None
    else:
        LRT_index = np.array(options.LRT_index.split(","), float).astype(int)
    intercept = None if options.intercept_mode.upper() in ["GENE", 'CELL'] else 0   # quant.py:205
    if options.n_perm < 0:
        print("[BRIE2] Error: --nPerm needs to be 0 or more.")
        sys.exit(1)
    if options.n_perm > 0 and LRT_index is not None and len(LRT_index) == 0:
        print("[BRIE2] Error: --nPerm needs tested features (--LRTindex).")
        sys.exit(1)
    groups = {}
    for flag, key in (("--LRTgroups", "LRT_groups"), ("--waldGroups", "wald_groups"), ("--scoreGroups", "score_groups")):
        text = getattr(options, key)
        if text is not None:
            try:
                groups[key] = [[int(k) for k in G.split(",")] for G in text.split(";")]
            except ValueError:
                print("[BRIE2] Error: %s needs ';'-separated groups of ','-separated column indices, got %r."
                      % (flag, text))
                sys.exit(1)
    if "score_groups" in groups and options.score_file is None:
        print("[BRIE2] Error: --scoreGroups needs --scoreFile.")
        sys.exit(1)

    quant(options.in_file, options.cell_file, options.gene_file,
          options.out_file, LRT_index, options.layers.split(','),
          intercept, options.intercept_mode, options.nproc, options.min_count,
          options.min_uniq_count, options.min_cell, options.min_MIF,
          options.min_iter, options.max_iter, options.MC_size,
          options.batch_size, options.pseudo_count, options.test_base, options.seed,
          options.out_dir, options.resume, options.n_perm, options.wald,
          **({} if options.score_file is None else dict(score_file=options.score_file)), **groups)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.barrier()
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
