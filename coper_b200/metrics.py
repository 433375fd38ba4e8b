"""Evaluator: filtered MR / MRR / Hits@k — mirror of ``qa_cpg/metrics.py:23-86``.

Same name, arguments, logging and return triple ``(mr, mrr, {k: hits})`` as the reference's
``ranking_and_hits``; the per-batch work changes: instead of copying ``[B,N]`` logits and a dense fp32
filter to the host and running B full ``argsort``s in a Python loop (metrics.py:40-57), the model
scores, masks and ranks on the device (``ConvE.filtered_ranks`` -> ``coper_filtered_rank``) and only the
B integer ranks come back.  ``data_iterator_handle`` is any iterable of batch dicts
(``e1, e2, rel, e2_multi`` per models.py:135-152; exhaustion plays the role of tf.errors.OutOfRangeError,
metrics.py:59).  ``session`` is accepted and ignored.
"""
from __future__ import annotations

import logging
import os

import numpy as np

from .models import has_known_tails

__all__ = ["ranking_and_hits"]

logger = logging.getLogger(__name__)


def _write_data_to_file(file_path, data):
    mode = "a" if os.path.exists(file_path) else "w+"
    with open(file_path, mode) as handle:
        handle.write(str(data) + "\n")


def ranking_and_hits(model, results_dir, data_iterator_handle, name, session=None,
                     hits_to_compute=(1, 3, 5, 10, 20), enable_write_to_file=False, return_ranks=False):
    os.makedirs(results_dir, exist_ok=True)
    logger.info("")
    logger.info("-" * 50)
    logger.info(name)
    logger.info("-" * 50)
    logger.info("")

    ranks = []
    ties = 0
    count = 0
    pending = []
    n_cand = set()
    for batch in data_iterator_handle:
        if "candidates" in batch:
            # rank among the batch's C given candidates (OGB-style negatives), filtered iff it carries the true tails
            rank_dev, n_equal_dev = model.candidate_ranks(batch, batch["candidates"], filtered=has_known_tails(batch))
            n_cand.add(int(batch["candidates"].shape[1]))
        else:
            rank_dev, n_equal_dev = model.filtered_ranks(batch)
        # keep the device busy: read the previous batch's ranks while this one runs
        pending.append((rank_dev.clone(), n_equal_dev.clone()))
        if len(pending) > 1:
            r, e = pending.pop(0)
            ranks.append(r.cpu().numpy())
            ties += int(e.sum().item())
        count += int(batch["e1"].shape[0])
    for r, e in pending:
        ranks.append(r.cpu().numpy())
        ties += int(e.sum().item())
    ranks = np.concatenate(ranks).astype(np.int64) if ranks else np.zeros(0, np.int64)
    if ties:
        logger.warning("%d unfiltered scores tie with a gold score; the reference's argsort order is "
                       "unspecified for those (reported rank = 1 + #strictly greater)", ties)
    if n_cand:
        logger.info("Ranks are against C = %s given candidates per query, not against all entities.",
                    "/".join(str(c) for c in sorted(n_cand)))
    logger.info("Evaluated %d samples." % count)

    hits = {}
    for hits_level in hits_to_compute:                            # metrics.py:53-57,65-72
        hits_value = np.mean([1.0 if r <= hits_level else 0.0 for r in ranks])
        logger.info("Hits @%d: %10.6f", hits_level, hits_value)
        hits[hits_level] = hits_value
        if enable_write_to_file:
            _write_data_to_file(os.path.join(results_dir, "hits_at_{}.txt".format(hits_level)), hits_value)

    mr = np.mean(ranks)                                           # metrics.py:75-76
    mrr = np.mean(1.0 / np.array(ranks))
    logger.info("Mean rank: %10.6f", mr)
    logger.info("Mean reciprocal rank: %10.6f", mrr)
    if enable_write_to_file:
        _write_data_to_file(os.path.join(results_dir, "mean_rank.txt"), mr)
        _write_data_to_file(os.path.join(results_dir, "mrr.txt"), mrr)
    logger.info("-" * 50)
    if return_ranks:
        return mr, mrr, hits, ranks
    return mr, mrr, hits
