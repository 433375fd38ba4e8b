"""Train / evaluate entry point — the reference's ``qa_cpg/run_cpg.py`` kept, driving the sm_100a kernels.

    python -m coper_b200.run_cpg --dataset WN18RR --model-type cpg --data-dir temp/WN18RR/data/WN18RR
    python -m coper_b200.run_cpg --synthetic wn18rr --max-steps 200          # no dataset files needed
    torchrun --nproc-per-node 8 -m coper_b200.run_cpg --dataset WN18RR             # entity-sharded over 8 GPUs

Where the reference edits flags in source (``run_cpg.py:38-46``: ``use_cpg``, ``use_parameter_lookup``,
``save_best_embeddings``, ``model_load_path``, the loader instance) they are command-line options here; everything else
follows the script: config lookup by ``(dataset, model type)`` (``:49-60``), the composed model name (``:63-84``), the
``temp/<dataset>/{summaries,checkpoints,evaluation,configs}/<model name>`` directory layout with the run config dumped
next to the outputs (``:87-105``), the step loop with loss logging every ``log_steps`` (``:209-223``), evaluation every
``eval_steps`` on dev / test through ``ranking_and_hits`` (``:18-35,226-236``), best-dev checkpoint + embedding pickle
(``:238-252``) and ``--model-load-path`` = restore, evaluate test, exit (``:205-208``).  TensorBoard summaries are
replaced by the log lines (SURVEY §5.5).

Under ``torchrun`` (one process per GPU) the entity table is sharded by entity id and the batch (the config's
``batch_size``, unchanged) is split over the ranks (``ConvE(..., shard=..., data_parallel=True)``): every rank reads the
same batches from its own, identically seeded loader; rank 0 logs and writes the config / embedding pickle, every rank
saves the checkpoint of its own rows.  Sampled-label configurations (``num_labels``) train sharded the same way: every
rank stages the same global [B, num_labels] ids / labels (or draws them on its GPU with ``--device-sampling``, identically
on every rank) and scores the ones its entity rows own; ``--full-1n`` switches to full 1-N labels, as on one GPU.
"""
from __future__ import annotations

import argparse
import logging
import os
import pickle
import sys

import numpy as np
import yaml

logger = logging.getLogger("coper_b200.run_cpg")

LOADERS = {"nations": "NationsLoader", "umls": "UMLSLoader", "kinship": "KinshipLoader", "WN18RR": "WN18RRLoader",
           "YAGO3-10": "YAGO310Loader", "FB15k-237": "FB15k237Loader", "countries_S1": "CountriesS1Loader",
           "countries_S2": "CountriesS2Loader", "countries_S3": "CountriesS3Loader", "WN18": "WN18Loader",
           "FB15k": "FB15kLoader", "nell-995": "NELL995Loader"}


def _evaluate(model, batches, name, results_dir, step):
    """run_cpg.py:18-35: metrics through ranking_and_hits, returned as the dict the loop compares."""
    from .metrics import ranking_and_hits
    mr, mrr, hits = ranking_and_hits(model, results_dir, batches, name)
    metrics = {"mr": mr, "mrr": mrr}
    for k, v in hits.items():
        metrics["hits@%d" % k] = v
    logger.info("step %d | %s | MR %.3f MRR %.5f %s", step, name, mr, mrr,
                " ".join("H@%d %.4f" % (k, v) for k, v in sorted(hits.items())))
    return metrics


def model_name_of(cfg, model_descr, dataset_name, use_cpg, clean):
    name = ("{}-{}-ent_emb_{}-rel_emb_{}-batch_{}-prop_neg_{}-num_labels_{}-OnePosPerSampl_{}-bn_momentum_{}-eval_{}"
            "-dropouts_{}_{}_{}_{}").format(
        model_descr, dataset_name, cfg.model.entity_embedding_size, cfg.model.relation_embedding_size,
        cfg.training.batch_size, cfg.training.prop_negatives, cfg.training.num_labels,
        cfg.training.get("one_positive_label_per_sample"), cfg.model.get("batch_norm_momentum"),
        cfg.eval.validation_metric, cfg.model.input_dropout, cfg.model.feature_map_dropout, cfg.model.output_dropout,
        cfg.context.context_rel_dropout)
    if use_cpg:
        name += "-context_batchnorm_{}".format(cfg.context.context_rel_use_batch_norm)
    if clean:
        name += "-CLEAN"
    return name


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--dataset", default="WN18RR", help="one of: " + ", ".join(sorted(LOADERS)))
    ap.add_argument("--model-type", default="cpg", choices=["cpg", "plain", "param_lookup"])
    ap.add_argument("--config", default=None, help="YAML file overriding the shipped config of (dataset, model type)")
    ap.add_argument("--data-dir", default=None, help="directory holding the split files train/valid|dev/test.txt, or <dataset>.tar.gz (extracted on first use)")
    ap.add_argument("--working-dir", default=None)
    ap.add_argument("--synthetic", default=None, help="run on a synthetic KG of this BASELINE shape instead of files")
    ap.add_argument("--full-1n", action="store_true", help="train with full 1-N labels (num_labels: null)")
    ap.add_argument("--device-sampling", action="store_true",
                    help="sampled-label configs: draw the [B, num_labels] ids / labels on the GPU (coper_sample_labels)")
    ap.add_argument("--max-steps", type=int, default=None)
    ap.add_argument("--eval-batches", type=int, default=None, help="cap the number of eval batches (synthetic runs)")
    ap.add_argument("--prec", default="fp16x3", choices=["fp32", "tf32x3", "fp16x3", "bf16"])
    ap.add_argument("--is-test", action="store_true")
    ap.add_argument("--needs-test-set-cleaning", action="store_true")
    ap.add_argument("--no-save-best-embeddings", action="store_true")
    ap.add_argument("--model-load-path", default=None)
    ap.add_argument("--predict-topk", type=int, default=None, metavar="K",
                    help="with --model-load-path: write the K most likely tails of every test query (filtered by the "
                         "known true tails) to <evaluation dir>/predictions_test.tsv")
    ap.add_argument("--score-triples", default=None, metavar="FILE",
                    help="with --model-load-path: score the tab-separated (head, relation, tail) lines of FILE and write "
                         "them with their logit and sigmoid(logit) to <evaluation dir>/scores_<FILE name without its "
                         "extension>.tsv")
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args(argv)
    if args.score_triples is not None and args.model_load_path is None:
        ap.error("--score-triples needs --model-load-path")
    if args.predict_topk is not None:
        if args.model_load_path is None:
            ap.error("--predict-topk needs --model-load-path")
        from ._lib import TOPK_MAX
        if not 1 <= args.predict_topk <= TOPK_MAX:
            ap.error("--predict-topk K needs 1 <= K <= %d" % TOPK_MAX)
    logging.basicConfig(level=logging.INFO, format="%(asctime)s %(name)s %(levelname)s %(message)s")

    from . import configs, data, synthetic
    from .models import ConvE
    from .sharding import EntityShard
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        import torch
        import torch.distributed as dist
        local = int(os.environ.get("LOCAL_RANK", str(rank)))
        # one GPU per rank over NCCL; if the box has fewer devices than local ranks (the single-GPU test tier) the
        # ranks share a device and the exchange steps run over gloo (host-staged, coper_b200/sharding.py)
        ndev = torch.cuda.device_count()
        shared_device = ndev < int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
        local = local % max(ndev, 1) if shared_device else local
        torch.cuda.set_device(local)
        if not dist.is_initialized():
            if shared_device:
                dist.init_process_group("gloo")
            else:
                dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        if rank != 0:
            logging.getLogger().setLevel(logging.WARNING)
    use_cpg, use_parameter_lookup = args.model_type == "cpg", args.model_type == "param_lookup"
    dataset_name = args.dataset
    cfg = configs.load_config(args.config) if args.config else configs.load_config(dataset_name, args.model_type)
    if args.full_1n or args.synthetic:
        cfg.training.num_labels = None
    if args.max_steps is not None:
        cfg.training.max_steps = args.max_steps

    conv_h = 10
    if args.synthetic:
        s = synthetic.SHAPES[args.synthetic]
        cfg.model.entity_embedding_size, cfg.model.relation_embedding_size = s["ent_emb_size"], s["rel_emb_size"]
        if args.model_type == "plain":      # the relation image is stacked under the entity image (models.py:361)
            cfg.model.relation_embedding_size = s["ent_emb_size"]
        cfg.training.batch_size = s["batch"]
        num_ent, num_rel, conv_h = s["num_ent"], s["num_rel"], s["H"]
        dataset_name = "synthetic-" + args.synthetic
        clean = False
        B = cfg.training.batch_size
        train_pool = synthetic.make_batches(num_ent, num_rel, B, 64, seed=args.seed + 1)

        def train_iter():
            i = 0
            while True:
                yield train_pool[i % len(train_pool)]
                i += 1
        n_eval = args.eval_batches or 4
        eval_sets = {k: synthetic.make_batches(num_ent, num_rel, B, n_eval, seed=args.seed + 100 + j)
                     for j, k in enumerate(("dev", "test"))}
        make_eval = lambda which: iter(eval_sets[which])
        train_batches = train_iter()
    else:
        cls = getattr(data, LOADERS[dataset_name])
        try:
            loader = cls(is_test=args.is_test, needs_test_set_cleaning=args.needs_test_set_cleaning)
        except TypeError:
            loader = cls()
        clean = loader.needs_test_set_cleaning
        dataset_name = loader.dataset_name
        working = args.working_dir or os.path.join(os.getcwd(), "temp", dataset_name)
        data_dir = args.data_dir or os.path.join(working, "data", dataset_name)
        # rank 0 extracts / parses / writes the id files and the CSR cache (atomically); the other ranks wait at the
        # barrier and then load the finished cache, so every rank sees the same ids and num_ent
        if world > 1 and rank != 0:
            dist.barrier()
        loader.maybe_create_tf_record_files(data_dir)
        if world > 1 and rank == 0:
            dist.barrier()
        num_ent, num_rel = loader.num_ent, loader.num_rel
        B = cfg.training.batch_size
        train_batches = loader.train_dataset(
            directory=data_dir, batch_size=B, include_inv_relations=True, prop_negatives=cfg.training.prop_negatives,
            num_labels=cfg.training.num_labels, cache=cfg.training.cache_data,
            one_positive_label_per_sample=cfg.training.get("one_positive_label_per_sample", False), seed=args.seed,
            device_sampling=args.device_sampling)

        def make_eval(which):
            it = loader.eval_dataset(directory=data_dir, dataset_type=which, batch_size=B, include_inv_relations=False)
            if args.eval_batches:
                import itertools
                it = itertools.islice(it, args.eval_batches)
            return it

    model_name = model_name_of(cfg, args.model_type, dataset_name, use_cpg, clean)
    logger.info("Model name: %s", model_name)
    working_dir = args.working_dir or os.path.join(os.getcwd(), "temp", dataset_name)
    ckpt_dir = os.path.join(working_dir, "checkpoints", model_name, "model_weights.ckpt")
    eval_path = os.path.join(working_dir, "evaluation", model_name)
    config_save_dir = os.path.join(working_dir, "configs", model_name)
    for d in (ckpt_dir, eval_path, config_save_dir):
        os.makedirs(d, exist_ok=True)
    ckpt_path = os.path.join(ckpt_dir, "model_weights.ckpt")
    embed_file = os.path.join(eval_path, "best_embeddings.ckpt")
    if rank == 0:
        with open(os.path.join(config_save_dir, "config.yml"), "w") as outfile:
            yaml.dump(_plain(cfg), outfile, default_flow_style=False)

    triples = None
    if args.score_triples is not None:      # read (and reject) the file before the model is built
        triples = _read_triples(args.score_triples, None if args.synthetic else _id_names(data_dir), num_ent, num_rel)
    md = configs.model_descriptors(cfg, num_ent, num_rel, use_cpg, use_parameter_lookup)
    split_batch = world > 1 and cfg.training.batch_size % world == 0 and not use_parameter_lookup
    model = ConvE(md, seed=args.seed, prec=args.prec, conv_in_height=conv_h, init_fast=num_ent > 1_000_000,
                  shard=EntityShard(num_ent, rank, world), data_parallel=split_batch,
                  graphs_multi_gpu=not (world > 1 and dist.get_backend() == "gloo"))
    logger.info("Number of entities: %d", num_ent)
    logger.info("Number of relations: %d", num_rel)

    validation_metric = cfg.eval.validation_metric
    lower_better = validation_metric == "mr"
    best_dev = {validation_metric: np.inf if lower_better else -np.inf}
    test_at_best = {}
    best_iter = None
    if args.model_load_path is not None:
        model.load_checkpoint(args.model_load_path)
        _evaluate(model, make_eval("test"), "test", eval_path, 0)
        if args.predict_topk is not None:
            names = None if args.synthetic else _id_names(data_dir)
            _write_predictions(model, make_eval("test"), args.predict_topk, names,
                               os.path.join(eval_path, "predictions_test.tsv"), rank == 0)
        if triples is not None:
            base = os.path.splitext(os.path.basename(args.score_triples))[0]
            _write_triple_scores(model, triples, cfg.training.batch_size,
                                 os.path.join(eval_path, "scores_%s.tsv" % base), rank == 0)
        return _finish(world)
    loss = None
    for step in range(cfg.training.max_steps):
        batch = next(train_batches)
        while split_batch and len(batch["e1"]) % world:      # the short batch that ends an epoch cannot be split evenly
            batch = next(train_batches)
        loss_dev = model.train_step(batch)
        if step % cfg.eval.log_steps == 0:
            loss = float(loss_dev.item())
            logger.info("Step %6d | Loss: %10.4f", step, loss)
        if step % cfg.eval.eval_steps == 0:
            logger.info("Evaluating model with name %s ...", model_name)
            metrics_dev = metrics_test = None
            if cfg.eval.eval_on_dev:
                metrics_dev = _evaluate(model, make_eval("dev"), "dev_evaluation", eval_path, step)
            if cfg.eval.eval_on_test:
                metrics_test = _evaluate(model, make_eval("test"), "test_evaluation", eval_path, step)
            if metrics_dev is not None and metrics_test is not None:
                improved = (metrics_dev[validation_metric] < best_dev[validation_metric]) if lower_better else \
                    (best_dev[validation_metric] < metrics_dev[validation_metric])
                if improved:
                    best_dev, test_at_best, best_iter = metrics_dev, metrics_test, step
                    if not args.no_save_best_embeddings:
                        ent = model.full_entity_table().cpu().numpy()          # (a collective when sharded)
                        obj = ent if use_parameter_lookup else [model.variables["rel_emb"].cpu().numpy(), ent]
                        if rank == 0:
                            with open(embed_file, "wb") as fh:
                                pickle.dump(obj, fh)
                    logger.info("Step %d. Saving checkpoint at %s...", step, ckpt_path)
                    model.save_checkpoint(ckpt_path)
                logger.info("Best dev %s so far is at step %s. Best dev metrics: %s", validation_metric, best_iter,
                            str(best_dev))
                logger.info("Test metrics at best dev: %s", str(test_at_best))
    if loss is not None:
        logger.info("final logged loss %.6f; best dev step %s", loss, best_iter)
    return _finish(world)


def _id_names(data_dir):
    """(entity names, relation names) indexed by id from entities.txt / relations.txt, or None without them.  Ids are
    line numbers, blank lines included, as the loader assigns them (data.py)."""
    out = []
    for f in ("entities.txt", "relations.txt"):
        path = os.path.join(data_dir, f)
        if not os.path.exists(path):
            return None
        with open(path) as fh:
            out.append([line.strip() for line in fh])
    return tuple(out)


def _write_predictions(model, batches, k, names, path, write):
    """One line per query: e1, relation, then k (entity, score) pairs, best first, tab-separated.  Every rank runs
    predict_topk (a collective when sharded); ``write`` selects the rank that writes the file."""
    ent = (lambda i: names[0][i]) if names else str
    rel = (lambda i: names[1][i]) if names else str
    fh = open(path, "w") if write else None
    n = 0
    for batch in batches:
        scores, ids = model.predict_topk(batch, k=k, filtered=True)
        scores, ids = scores.cpu().numpy(), ids.cpu().numpy()
        if fh is None:
            continue
        e1, r = np.asarray(batch["e1"]).reshape(-1), np.asarray(batch["rel"]).reshape(-1)
        for b in range(len(e1)):
            cols = [ent(int(e1[b])), rel(int(r[b]))]
            for s, i in zip(scores[b], ids[b]):
                if i >= 0:
                    cols += [ent(int(i)), "%.6g" % s]
            fh.write("\t".join(cols) + "\n")
            n += 1
    if fh is not None:
        fh.close()
        logger.info("wrote the top-%d predictions of %d test queries to %s", k, n, path)


def _read_triples(path, names, num_ent, num_rel):
    """Tab-separated (head, relation, tail) lines -> (e1, rel, e2) int64 arrays and the input columns.  Names map
    through ``names`` (entities.txt / relations.txt); without them the columns are integer ids.  A name that is not
    known, an id out of range or a line without three columns exits with the file and line number."""
    index = [{n: i for i, n in enumerate(t)} for t in names] if names else None
    ids, cols = [], []
    with open(path) as fh:
        for lineno, line in enumerate(fh, 1):
            line = line.rstrip("\r\n")
            if not line.strip():
                continue
            f = line.split("\t")
            if len(f) != 3:
                sys.exit("%s:%d: expected 3 tab-separated columns (head, relation, tail), got %d" % (path, lineno, len(f)))
            row = []
            for col, what, kind, n in ((f[0], "entity", 0, num_ent), (f[1], "relation", 1, num_rel),
                                       (f[2], "entity", 0, num_ent)):
                if index is not None:
                    i = index[kind].get(col.strip(), -1)
                    if i < 0:
                        sys.exit("%s:%d: unknown %s name %r" % (path, lineno, what, col))
                else:
                    try:
                        i = int(col)
                    except ValueError:
                        sys.exit("%s:%d: %r is not an integer %s id (the dataset has no name files)" %
                                 (path, lineno, col, what))
                    if not 0 <= i < n:
                        sys.exit("%s:%d: %s id %d out of range [0, %d)" % (path, lineno, what, i, n))
                row.append(i)
            ids.append(row)
            cols.append(f)
    ids = np.asarray(ids, dtype=np.int64).reshape(-1, 3)
    return ids[:, 0], ids[:, 1], ids[:, 2], cols


def _write_triple_scores(model, triples, batch_size, path, write):
    """One line per input line: its three columns, the logit (%.6g) and sigmoid(logit).  Every rank scores (a
    collective when sharded); ``write`` selects the rank that writes the file."""
    e1, rel, e2, cols = triples
    fh = open(path, "w") if write else None
    for i in range(0, len(e1), batch_size):
        sl = slice(i, i + batch_size)
        s = model.score_candidates({"e1": e1[sl], "rel": rel[sl]}, e2[sl].reshape(-1, 1)).cpu().numpy()[:, 0]
        if fh is None:
            continue
        sig = 0.5 * (1.0 + np.tanh(0.5 * s.astype(np.float64)))
        for j in range(len(s)):
            fh.write("\t".join(cols[i + j] + ["%.6g" % s[j], "%.6g" % sig[j]]) + "\n")
    if fh is not None:
        fh.close()
        logger.info("wrote the scores of %d triples to %s", len(e1), path)


def _finish(world):
    """Multi-process runs leave without tearing NCCL down: destroy_process_group() blocks once collectives have been
    captured into CUDA graphs; everything is synchronised and flushed first."""
    if world > 1:
        import torch
        torch.cuda.synchronize()
        logging.shutdown()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    return 0


def _plain(d):
    return {k: _plain(v) if isinstance(v, dict) else v for k, v in d.items()}


if __name__ == "__main__":
    sys.exit(main())
