"""Config flag system of the reference, kept (``qa_cpg/run_cpg.py:49-60``, ``qa_cpg/configs/*.yaml``).

The reference reads ``configs/config_<dataset>_<cpg|plain|param_lookup>.yaml`` into a nested attribute dict with the
sections ``model / context / training / eval``.  Here the same structure is produced by :func:`load_config`:

* ``load_config(path_to_yaml)`` parses a user YAML file with ``yaml.safe_load`` (the reference's bare ``yaml.load(file)``
  raises on PyYAML >= 6, SURVEY Q13);
* ``load_config(dataset_name, model_type)`` builds the shipped configuration of that dataset from the table below — the
  hyper-parameters are the reference's (one row of overrides per shipped file, on top of the values every file shares),
  with its known config hazards fixed and flagged: ``nell-995`` cpg uses ``entity_embedding_size`` 200 instead of 225
  (225 is not a multiple of the conv image height 10, ``models.py:355`` fails on it), ``umls`` cpg gets the missing
  ``batch_norm_*`` keys, ``input_dropout: 2`` of ``nell-995-test`` is kept (the flag is parsed and unused, Q4).

``AttributeDict`` mirrors ``qa_cpg/utils/dict_with_attributes.py:1-9``.
"""
from __future__ import annotations

import copy
import os
from typing import Optional

import yaml

__all__ = ["AttributeDict", "load_config", "model_descriptors", "SHIPPED"]


class AttributeDict(dict):
    """Nested dict whose keys are also attributes (``cfg.model.entity_embedding_size``)."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        for k, v in list(self.items()):
            if isinstance(v, dict) and not isinstance(v, AttributeDict):
                self[k] = AttributeDict(v)

    def __getattr__(self, name):
        try:
            return self[name]
        except KeyError as exc:
            raise AttributeError(name) from exc

    def __setattr__(self, name, value):
        self[name] = value


_COMMON = {
    "model": dict(entity_embedding_size=200, relation_embedding_size=200, concat_rel=False, input_dropout=0.2,
                  feature_map_dropout=0.3, output_dropout=0.2, label_smoothing_epsilon=0.1, batch_norm_momentum=0.1,
                  batch_norm_train_stats=True),
    "context": dict(context_rel_conv=None, context_rel_out=None, context_rel_dropout=0.2,
                    context_rel_use_batch_norm=True),
    "training": dict(learning_rate=0.001, batch_size=512, device="/GPU:0", max_steps=2000000, prop_negatives=10.0,
                     num_labels=100, one_positive_label_per_sample=False, cache_data=True),
    "eval": dict(validation_metric="hits@1", log_steps=100, ckpt_steps=50000, eval_steps=5000, summary_steps=100,
                 eval_on_train=False, eval_on_dev=True, eval_on_test=True, add_loss_summaries=True,
                 add_variable_summaries=False, add_tensor_summaries=False),
}

_G_LINEAR = {"context.context_rel_out": []}          # CPG generates the FC layer linearly from the relation embedding
# (dataset, model_type) -> overrides ("section.key": value)
SHIPPED = {
    ("FB15k-237", "cpg"): {**_G_LINEAR, "model.relation_embedding_size": 32, "model.batch_norm_momentum": 0.99,
                           "training.prop_negatives": 100.0, "training.num_labels": 1000},
    ("FB15k-237", "plain"): {"training.max_steps": 4000000, "eval.summary_steps": 500},
    ("FB15k", "cpg"): {**_G_LINEAR, "model.relation_embedding_size": 32, "model.batch_norm_momentum": 0.99,
                       "training.prop_negatives": 100.0, "training.num_labels": 1000},
    ("WN18RR", "cpg"): {**_G_LINEAR, "model.relation_embedding_size": 8},
    ("WN18RR", "param_lookup"): {**_G_LINEAR, "model.relation_embedding_size": 8},
    ("WN18RR", "plain"): {"training.max_steps": 4000000, "eval.summary_steps": 500},
    ("WN18", "cpg"): {**_G_LINEAR, "model.relation_embedding_size": 8, "model.do_parameter_lookup": False},
    ("YAGO03-10", "cpg"): {**_G_LINEAR, "training.max_steps": 10000000, "training.one_positive_label_per_sample": True,
                           "training.cache_data": False, "eval.log_steps": 500, "eval.ckpt_steps": 10000000,
                           "eval.eval_steps": 100},
    ("YAGO03-10", "plain"): {"training.max_steps": 10000000, "training.one_positive_label_per_sample": True,
                             "training.cache_data": False, "eval.ckpt_steps": 10000000, "eval.eval_steps": 100},
    ("YAGO3-10", "cpg"): {**_G_LINEAR, "model.relation_embedding_size": 37, "context.context_rel_dropout": 0.5,
                          "training.batch_size": 128, "training.max_steps": 100000000, "training.prop_negatives": 1.0,
                          "training.num_labels": 1000, "training.one_positive_label_per_sample": True,
                          "training.cache_data": False, "eval.eval_steps": 15000},
    ("kinship", "cpg"): {**_G_LINEAR, "model.relation_embedding_size": 50, "model.input_dropout": 0.5,
                         "model.feature_map_dropout": 0.5, "model.output_dropout": 0.5,
                         "model.batch_norm_train_stats": False, "context.context_rel_dropout": 0.5,
                         "training.max_steps": 8000, "eval.log_steps": 50, "eval.ckpt_steps": 1000,
                         "eval.eval_steps": 10, "eval.summary_steps": 10},
    ("kinship", "param_lookup"): {**_G_LINEAR, "model.relation_embedding_size": 1, "model.input_dropout": 0.5,
                                  "model.feature_map_dropout": 0.5, "model.output_dropout": 0.5,
                                  "model.batch_norm_train_stats": False, "model.do_parameter_lookup": True,
                                  "context.context_rel_dropout": 0.5, "training.max_steps": 8000, "eval.log_steps": 50,
                                  "eval.ckpt_steps": 1000, "eval.eval_steps": 10, "eval.summary_steps": 10},
    ("kinship", "plain"): {"model.batch_norm_train_stats": False, "training.max_steps": 50000, "eval.log_steps": 50,
                           "eval.ckpt_steps": 1000, "eval.eval_steps": 100},
    ("nations", "cpg"): {**_G_LINEAR, "model.relation_embedding_size": 8, "model.batch_norm_train_stats": False,
                         "training.max_steps": 1000, "training.num_labels": 50, "eval.log_steps": 10,
                         "eval.ckpt_steps": 1000, "eval.eval_steps": 10, "eval.summary_steps": 10},
    ("nations", "plain"): {"model.batch_norm_train_stats": False, "training.max_steps": 1000,
                           "training.prop_negatives": 1.0, "training.num_labels": None, "eval.log_steps": 10,
                           "eval.ckpt_steps": 1000, "eval.eval_steps": 10, "eval.summary_steps": 10},
    ("nell-995-test", "cpg"): {**_G_LINEAR, "model.relation_embedding_size": 32, "model.input_dropout": 2,
                               "model.batch_norm_momentum": 0.99, "context.context_rel_dropout": 0.5,
                               "training.learning_rate": 0.003, "training.max_steps": 10000000,
                               "training.prop_negatives": 100.0, "training.num_labels": 1000, "eval.ckpt_steps": 60000,
                               "eval.summary_steps": 1000},
    ("nell-995-test", "plain"): {"training.learning_rate": 0.003, "training.max_steps": 10000000,
                                 "training.prop_negatives": 100.0, "training.num_labels": 1000,
                                 "eval.ckpt_steps": 10000000},
    # reference file says entity_embedding_size: 225, which models.py:355 cannot reshape to [-1, 10, d // 10, 1]
    ("nell-995", "cpg"): {**_G_LINEAR, "model.entity_embedding_size": 200, "model.relation_embedding_size": 32,
                          "training.learning_rate": 0.003, "training.max_steps": 10000000,
                          "training.prop_negatives": 100.0, "training.num_labels": 1000, "eval.ckpt_steps": 10000000,
                          "eval.summary_steps": 1000},
    ("nell-995", "plain"): {"training.learning_rate": 0.003, "training.max_steps": 10000000,
                            "training.prop_negatives": 100.0, "training.num_labels": 1000,
                            "eval.ckpt_steps": 10000000},
    # g_MLP (one hidden layer of 64) and full 1-N training; reference file lacks the batch_norm_* keys
    ("umls", "cpg"): {"context.context_rel_out": [64], "training.max_steps": 1000, "training.prop_negatives": 1.0,
                      "training.num_labels": None, "eval.ckpt_steps": 1000, "eval.eval_steps": 10,
                      "eval.summary_steps": 10},
    ("umls", "param_lookup"): {**_G_LINEAR, "model.relation_embedding_size": 8, "model.batch_norm_train_stats": False,
                               "training.batch_size": 5, "training.max_steps": 1000, "training.num_labels": 10,
                               "training.one_positive_label_per_sample": True, "eval.log_steps": 10,
                               "eval.ckpt_steps": 1000, "eval.eval_steps": 100, "eval.summary_steps": 10},
    ("umls", "plain"): {"model.batch_norm_train_stats": False, "training.max_steps": 50000, "eval.ckpt_steps": 10000,
                        "eval.eval_steps": 100},
}


def load_config(dataset_or_path: str, model_type: Optional[str] = None) -> AttributeDict:
    """``load_config('configs/my.yaml')`` or ``load_config('WN18RR', 'cpg')`` (run_cpg.py:49-60)."""
    if model_type is None or os.path.exists(dataset_or_path):
        with open(dataset_or_path, "r") as fh:
            return AttributeDict(yaml.safe_load(fh))
    key = (dataset_or_path, model_type)
    if key not in SHIPPED:
        raise KeyError("no shipped configuration config_%s_%s (available: %s)" % (
            dataset_or_path, model_type, ", ".join("%s_%s" % k for k in sorted(SHIPPED))))
    cfg = copy.deepcopy(_COMMON)
    for dotted, value in SHIPPED[key].items():
        section, name = dotted.split(".")
        cfg[section][name] = copy.deepcopy(value)
    return AttributeDict(cfg)


def model_descriptors(cfg: AttributeDict, num_ent: int, num_rel: int, use_cpg: bool = True,
                      use_parameter_lookup: bool = False) -> dict:
    """The dict ``run_cpg.py:115-137`` hands to ``ConvE`` (same keys; ``hidden_dropout`` is the config's
    ``feature_map_dropout``, ``use_negative_sampling`` is ``num_labels is not None``)."""
    m, c, t, e = cfg.model, cfg.context, cfg.training, cfg.eval
    del use_cpg          # as in the reference, the context_* values decide (plain configs carry context_rel_out: null)
    return {
        "use_negative_sampling": t.get("num_labels") is not None,
        "label_smoothing_epsilon": m.label_smoothing_epsilon,
        "num_ent": num_ent, "num_rel": num_rel,
        "ent_emb_size": m.entity_embedding_size, "rel_emb_size": m.relation_embedding_size,
        "concat_rel": m.concat_rel,
        "context_rel_conv": c.context_rel_conv,
        "context_rel_out": c.context_rel_out,
        "context_rel_dropout": c.context_rel_dropout,
        "context_rel_use_batch_norm": c.context_rel_use_batch_norm,
        "input_dropout": m.input_dropout, "hidden_dropout": m.feature_map_dropout,
        "output_dropout": m.output_dropout, "learning_rate": t.learning_rate, "batch_size": t.batch_size,
        "add_loss_summaries": e.add_loss_summaries, "add_variable_summaries": e.add_variable_summaries,
        "add_tensor_summaries": e.add_tensor_summaries,
        "batch_norm_momentum": m.get("batch_norm_momentum", 0.1),
        "batch_norm_train_stats": m.get("batch_norm_train_stats", False),
        "do_parameter_lookup": use_parameter_lookup,
        "loss": m.get("loss", "bce"),       # "bce" (the reference's objective) or "softmax_ce" (include/coper.h)
    }
