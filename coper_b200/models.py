"""Host-side mirror of the reference model object (``qa_cpg/models.py``) driving libcoper_sm100.

``ConvE(model_descriptors)`` takes the same descriptor dict the reference builds at
``run_cpg.py:115-137`` and exposes the same variable names (``.variables['ent_emb'|'rel_emb'|
'conv1_weights'|'conv1_bias'|'fc_weights'|'fc_bias'|'pred_bias']``, ``models.py:316-325``).  Where
the reference returns graph tensors to ``session.run`` (``run_cpg.py:210-219``, ``metrics.py:40-42``),
this object offers the equivalent eager calls:

    loss = model.train_step(batch)          # == session.run((model.loss, model.train_op), {is_train: True})
    scores = model.predict_all(batch)       # == session.run(model.predictions_all)
    ranks, n_equal = model.filtered_ranks(batch)   # metrics.py:44-51 done on device
    scores = model.score_candidates(batch, candidates)         # [B, C] logits of given tails (-1 = padding)
    ranks, n_equal = model.candidate_ranks(batch, candidates)  # rank of e2 among C given candidates

PyTorch is used only for device memory, streams, CUDA graphs and torch.distributed; every
arithmetic step of the hot path is a call into the C ABI (``include/coper.h``).  There is no
CPU / PyTorch fallback: without the CUDA library or a GPU this raises.

Supported configurations = the three model types the reference ships configs for: ``cpg`` (``context_rel_out: [...]``,
g_linear ``[]`` or g_MLP ``[n, ...]``), ``plain`` (``context_rel_out: null``: shared FC weights, relation image stacked
under the entity image) and ``param_lookup`` (``do_parameter_lookup``: per-relation tables), plus CPG-generated conv
filters (``context_rel_conv: [...]`` together with ``context_rel_out``); training with full 1-N labels
(``num_labels: null``) or with sampled labels (``use_negative_sampling``, ``models.py:438-443``:
``batch['lookup_values']`` [B, L] or labels drawn on the device), both entity-sharded across GPUs.  Evaluation ranks
against all N entities, or against C given candidates per query (``candidate_ranks``).  ``concat_rel`` and generated
conv filters combined with shared FC weights / parameter tables raise NotImplementedError (no shipped configuration
uses them, SURVEY §8f row 4).

Engines (``prec``): ``fp32`` (CUDA-core FFMA, the on-device parity reference), ``tf32x3`` / ``fp16x3`` (fp32-class
3-term compensated tcgen05 engines), ``bf16`` (tcgen05, the 10 M-entity throughput path; its scorer + BCE + dq run as
one fused kernel).
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional

import numpy as np
import torch

from . import _lib, sharding
from ._lib import (CPG_BWD_DCB_ACCUMULATE, CPG_BWD_INPUT_GRADS_ONLY, CPG_BWD_REUSE_FWD, CPG_BWD_WEIGHT_GRADS_ONLY, PREC,
                   call, call_plain, ptr)
from .sharding import EntityShard

BN_EPS = 1e-3           # tf.layers.batch_normalization default epsilon (models.py:386-388)
CLIP_NORM = 5.0         # models.py:199
SALT_FEATURE_MAP = 1 << 40
SALT_OUTPUT = 2 << 40
SALT_SAMPLE = 4 << 40   # on-device label sampling (coper_sample_labels)
SALT_CTX = 3 << 40      # + (net_id * 64 + layer) << 32


def _xavier_(t: torch.Tensor, gen: torch.Generator):
    """tf.contrib.layers.xavier_initializer: U(+-sqrt(6/(fan_in+fan_out))) (models.py:208)."""
    shape = t.shape
    if len(shape) == 1:
        fan_in = fan_out = shape[0]
    else:
        rec = int(np.prod(shape[:-2])) if len(shape) > 2 else 1
        fan_in, fan_out = shape[-2] * rec, shape[-1] * rec
    lim = math.sqrt(6.0 / (fan_in + fan_out))
    t.copy_((torch.rand(t.shape, generator=gen, dtype=torch.float32) * 2 - 1) * lim)


class _BatchNorm:
    """Parameters + scratch of one tf.layers.batch_normalization site."""

    def __init__(self, C, dev):
        f = dict(dtype=torch.float32, device=dev)
        self.C = C
        self.gamma, self.beta = torch.ones(C, **f), torch.zeros(C, **f)
        self.moving_mean, self.moving_var = torch.zeros(C, **f), torch.ones(C, **f)
        self.a, self.b, self.mean, self.invstd = (torch.empty(C, **f) for _ in range(4))
        self.dgamma, self.dbeta, self.c1, self.c2 = (torch.zeros(C, **f) for _ in range(4))


class ContextualParameterGenerator:
    """Variables of one CPG (models.py:32-54): ``projections`` [in,n] per layer, optional BN per hidden layer."""

    def __init__(self, context_size: List[int], name: str, shape: List[int], zero_init: bool, use_batch_norm: bool,
                 dev, gen):
        self.name, self.shape = name, list(shape)
        self.num_elements = int(np.prod(shape))
        sizes = list(context_size) + [self.num_elements]
        self.projections: List[torch.Tensor] = []
        for i in range(len(sizes) - 1):
            t = torch.zeros(sizes[i], sizes[i + 1], dtype=torch.float32)
            if not zero_init:
                _xavier_(t, gen)
            self.projections.append(t.to(dev))
        self.use_batch_norm = use_batch_norm
        self.bns = [_BatchNorm(n, dev) for n in context_size[1:]]
        self.hidden = list(context_size[1:])


def has_known_tails(batch: Dict) -> bool:
    """Does the batch carry the known true tails of its queries (``e2_multi``, or ``e2_multi_rowptr`` / ``e2_multi_col``)?"""
    return "e2_multi_rowptr" in batch or batch.get("e2_multi") is not None


class _BatchSlot:
    """Static device buffers of one batch size (pointer-stable -> CUDA-graph friendly).  Fields that a variant does not
    use are None; lazily filled ones start as None / {} / 0."""

    def __init__(self, m: "ConvE", B: int):
        dev, f32 = m.dev, torch.float32
        d, dr, F, C = m.ent_emb_size, m.rel_emb_size, m.F, m.C
        Ns = m.shard.rows
        z = lambda *s, dt=f32: torch.zeros(*s, dtype=dt, device=dev)
        lib = _lib.load()
        self.B, self.ld, self.words = B, -(-Ns // 32) * 32, -(-Ns // 32)
        # query ids + CSR row pointers live in ONE device block so that a host batch needs one H2D copy for them:
        # [e1 | rel | e2] int64 [3, B] followed by rowptr int32 [B + 1]
        head_words = 6 * B + (B + 2)
        self.d_head = z(head_words, dt=torch.int32)
        self.h_head = torch.zeros(head_words, dtype=torch.int32).pin_memory()
        idx64 = self.d_head[:6 * B].view(torch.int64).view(3, B)
        self.e1, self.rel, self.e2 = idx64[0], idx64[1], idx64[2]
        self.h_head_np = self.h_head.numpy()
        self.h_idx_np = self.h_head_np[:6 * B].view(np.int64).reshape(3, B)
        self.h_rowptr_np = self.h_head_np[6 * B:6 * B + B + 1]
        self.x0, self.r = z(B, d), z(B, dr)
        Fc = m.F_conv
        self.z, self.f = z(B, Fc), z(B, F)
        # concat_rel: the conv block works on contiguous [B, F_conv] buffers; f / df hold [conv features | rel_emb]
        self.fconv, self.dfconv = (z(B, Fc), z(B, Fc)) if m.concat_rel else (self.f, None)
        self.y, self.q = z(B, d), z(B, d)
        self.q_prep = None
        if m.E_prep is not None:
            self.q_prep = torch.zeros(lib.coper_prepared_bytes(B, d, m.prec), dtype=torch.uint8, device=dev)
        self.dq, self.dy, self.df, self.dz, self.dx0, self.dr = z(B, d), z(B, d), z(B, F), z(B, Fc), z(B, d), z(B, dr)
        if not m.concat_rel:
            self.dfconv = self.df
        R1 = B * m.OH * m.OW
        nch = max(lib.coper_colstats_chunks(R1), lib.coper_colstats_chunks(B))
        maxC = max([C, d] + [n for gcp in m.generators for n in gcp.hidden])
        self.stat = z(nch * maxC * 2)
        self.stat1 = z(maxC * 2)
        self.stat_all = None          # data-parallel front end: every rank's statistics partials (first use)
        # allocated on first use (each exactly once, so captured graphs keep valid pointers):
        #   S  logits fp32 [B, ld] (predict_all / the two-pass ranking of the fp32 engine)
        #   G  dL/dS in the scorer's operand form (train); never read by the host
        self.S = self.G = None
        # label / filter bits: query-major rows for the fp32 engine, the entity-major matrix for the tensor pipe
        self.bits = z(B, self.words, dt=torch.int32) if m.prec == 0 else None
        self.bitsT = z(max(Ns, 1), -(-B // 32), dt=torch.int32) if m.prec != 0 else None
        self.loss_sum = z(1, dt=torch.float64)
        self.gold = z(B)
        self.rank_counts = z(2, B, dt=torch.int32)       # one buffer: cleared by one fill per evaluation batch
        self.n_greater, self.n_equal = self.rank_counts[0], self.rank_counts[1]
        self.rank = z(B, dt=torch.int32)
        self.loss_mean = z(1, dt=torch.float64)
        self.dwc_part, self.dbc_part = z(B, m.conv_filter_height * m.conv_filter_width * C), z(B, C)
        dcw = m.fc_weights.projections[-1].shape[0]
        dcb = m.fc_bias.projections[-1].shape[0]
        # the CPG workspace is kept apart: the backward reuses the operands the forward prepared in it
        ws_cpg = max(lib.coper_cpg_fc_fwd_workspace_bytes(B, dcw, F, d, m.prec),
                     lib.coper_cpg_fc_bwd_workspace_bytes(B, dcw, F, d, m.prec))
        self.ws_cpg = torch.empty(ws_cpg, dtype=torch.uint8, device=dev)
        self.ws_cpg_bytes = ws_cpg
        ws = max(lib.coper_score1n_bce_workspace_bytes(B, Ns, d, m.prec),
                 lib.coper_score1n_workspace_bytes(B, Ns, d, m.prec),
                 lib.coper_segscatter_workspace_bytes(B), lib.coper_score1n_rank_workspace_bytes(B, d, m.prec))
        self.ws = torch.empty(ws, dtype=torch.uint8, device=dev)
        self.ws_bytes = ws
        # context nets: activations per hidden layer for the two generators
        self.ctx = {}
        for cpg in m.generators:
            self.ctx[cpg.name] = {"pre": [z(B, n) for n in cpg.hidden], "act": [z(B, n) for n in cpg.hidden],
                                  "dact": [z(B, n) for n in cpg.hidden], "dpre": [z(B, n) for n in cpg.hidden]}
        self.dcw, self.dcb = z(B, dcw), z(B, dcb)
        # contexts the forward pass used for the FC weights / bias and the conv filter / bias generators
        self.cw = self.cb = self.ccw = self.ccb = None
        # per-query filters [B, KH*KW*C], biases [B, C], context gradients (generated conv filters)
        self.wq = self.bq = self.dccw = self.dccb = None
        if m.conv_w_gen is not None:
            KK = m.conv_filter_height * m.conv_filter_width * C
            self.wq, self.bq = z(B, KK), z(B, C)
            self.dccw = z(B, m.conv_w_gen.projections[-1].shape[0])
            self.dccb = z(B, m.conv_b_gen.projections[-1].shape[0])
        self.xc = self.dxc = self.cconst = None
        self.f_sq = self.dy_sq = self.df_scratch = None
        if m.variant == "plain":          # the stacked [entity image; relation image] and its gradient
            self.xc, self.dxc = z(B, d + dr), z(B, d + dr)
            self.cconst = torch.ones(B, 1, dtype=f32, device=dev)
        if m.variant == "param_lookup":   # one-hot(rel) context; squared operands of the slice-wise bookkeeping
            self.cconst = z(B, m.num_rel)
            self.f_sq, self.dy_sq, self.df_scratch = z(B, F), z(B, d), z(B, F)
        self.dx0_sq = z(B, d) if m.use_negative_sampling else None
        self.dr_sq = z(B, dr)
        # sub-slots, each built once per key: sampled labels (by L), top-k (by k), given candidates (by C)
        self.samp: Dict[int, _SampledSlot] = {}
        self.topk: Dict[int, _TopkSlot] = {}
        self.cand: Dict[int, _CandSlot] = {}
        # the sampled-label step: its [B, L] sub-slot and (num_labels, prop_negatives) when drawn on the device
        self.cur_samp, self.cur_sampling = None, None
        # pinned staging for host batches; csr_gen counts reallocations of col (graphs that captured the old pointer
        # must not be replayed)
        self.csr_cap, self.csr_gen = 0, 0
        self.rowptr = self.d_head[6 * B:6 * B + B + 1]
        self.col = self.h_col = self.h_col_np = None
        self.h2d_event = None


class _SampledSlot:
    """[B, L] lookup ids / labels of the sampled-label step, their pinned staging, scores, dL/dS and workspace."""

    def __init__(self, m: "ConvE", B: int, L: int):
        f = dict(dtype=torch.float32, device=m.dev)
        self.L = L
        self.lookup = torch.zeros(B, L, dtype=torch.int32, device=m.dev)
        self.labels, self.scores, self.g = (torch.zeros(B, L, **f) for _ in range(3))
        self.h_lookup = torch.zeros(B, L, dtype=torch.int32).pin_memory()
        self.h_labels = torch.zeros(B, L, dtype=torch.float32).pin_memory()
        lib = _lib.load()
        nbytes = lib.coper_score_sampled_sharded_workspace_bytes(B, L) if m.world > 1 else \
            lib.coper_score_sampled_workspace_bytes(B, L)
        self.ws = torch.empty(nbytes, dtype=torch.uint8, device=m.dev)


class _TopkSlot:
    """(B, k) outputs of predict_topk, the scorer's workspace and, under entity sharding, the per-rank lists."""

    def __init__(self, m: "ConvE", B: int, k: int):
        lib, dev, P = _lib.load(), m.dev, m.world
        self.scores = torch.empty(B, k, dtype=torch.float32, device=dev)
        self.ids = torch.empty(B, k, dtype=torch.int64, device=dev)
        if m.E_prep is not None:
            self.ws_bytes = lib.coper_score1n_topk_workspace_bytes(B, m.shard.rows, m.ent_emb_size, k, m.prec)
        else:
            self.ws_bytes = lib.coper_topk_scores_workspace_bytes(B, m.shard.rows, k)
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=dev)
        self.local_scores = self.local_ids = self.all_scores = self.all_ids = None
        if P > 1:        # this rank's list, and every rank's list after the exchange
            self.local_scores, self.local_ids = torch.empty_like(self.scores), torch.empty_like(self.ids)
            self.all_scores = torch.empty(P, B, k, dtype=torch.float32, device=dev)
            self.all_ids = torch.empty(P, B, k, dtype=torch.int64, device=dev)


class _CandSlot:
    """(B, C) slot: int32 [B, C] candidates followed by the [B] gold ids in one device block, staged through one
    pinned host block (one copy per call), the [B, C] scores and the rank outputs."""

    def __init__(self, m: "ConvE", B: int, C: int):
        dev = m.dev
        self.C = C
        self.d_ids = torch.zeros(B * C + B, dtype=torch.int32, device=dev)
        self.cand, self.e2 = self.d_ids[:B * C].view(B, C), self.d_ids[B * C:]
        self.h_ids = torch.zeros(B * C + B, dtype=torch.int32).pin_memory()
        self.h_np = self.h_ids.numpy()
        self.scores = torch.zeros(B, C, dtype=torch.float32, device=dev)
        self.gold = torch.zeros(B, dtype=torch.float32, device=dev)
        self.counts = torch.zeros(2, B, dtype=torch.int32, device=dev)
        self.n_greater, self.n_equal = self.counts[0], self.counts[1]
        self.rank = torch.zeros(B, dtype=torch.int32, device=dev)


def _slot(table: Dict, key, cls, *args):
    """table[key], built as cls(*args) on first use (exactly once: captured graphs keep valid pointers)."""
    if key not in table:
        table[key] = cls(*args)
    return table[key]


class ConvE:
    def __init__(self, model_descriptors: Dict, device: Optional[str] = None, seed: int = 0, prec: str = "fp32",
                 shard: Optional[EntityShard] = None, reference_bug_compat: bool = True,
                 conv_in_height: int = 10, process_group=None, use_graphs: bool = True,
                 init_fast: bool = False, graphs_multi_gpu: bool = False, data_parallel: bool = False,
                 overlap_grad_allreduce: bool = True):
        md = model_descriptors
        _lib.load()
        if not torch.cuda.is_available():
            raise _lib.CoperError("coper_b200.ConvE needs a CUDA device (sm_100a); no CPU fallback exists")
        self.dev = torch.device(device or "cuda:%d" % torch.cuda.current_device())
        torch.cuda.set_device(self.dev)
        # ---- descriptors (models.py:98-128)
        self.use_negative_sampling = md.get("use_negative_sampling", False)
        self.label_smoothing_epsilon = float(md["label_smoothing_epsilon"])
        self.num_ent, self.num_rel = int(md["num_ent"]), int(md["num_rel"])
        self.ent_emb_size, self.rel_emb_size = int(md["ent_emb_size"]), int(md["rel_emb_size"])
        self.is_parameter_lookup = md.get("do_parameter_lookup", False)
        self.conv_filter_height = md.get("conv_filter_height", 3)
        self.conv_filter_width = md.get("conv_filter_width", 3)
        self.conv_num_channels = md.get("conv_num_channels", 32)
        self.concat_rel = md.get("concat_rel", False)
        self.context_rel_conv = md.get("context_rel_conv", None)
        self.context_rel_out = md.get("context_rel_out", None)
        self.context_rel_dropout = float(md.get("context_rel_dropout", 0.0) or 0.0)
        self.context_rel_use_batch_norm = bool(md.get("context_rel_use_batch_norm", False))
        self.input_dropout = md.get("input_dropout", 0.0)          # parsed, unused (models.py:366-370)
        self.hidden_dropout = float(md.get("hidden_dropout", 0.0) or 0.0)
        self.output_dropout = float(md.get("output_dropout", 0.0) or 0.0)
        self.batch_norm_momentum = float(md.get("batch_norm_momentum", 0.1))
        self.batch_norm_train_stats = bool(md.get("batch_norm_train_stats", False))
        self.learning_rate = float(md.get("learning_rate", 1e-3))
        # the three model types the reference ships configurations for (configs/config_*_{cpg,plain,param_lookup}.yaml)
        #   cpg           context_rel_out = [...]: FC weights / bias generated from the relation embedding
        #   plain         context_rel_out = context_rel_conv = null: the relation embedding, reshaped, is stacked under
        #                 the entity image (models.py:360-362); ONE shared FC weight [F, d] (models.py:334-340, 410)
        #   param_lookup  do_parameter_lookup: FC weights / bias are rows of per-relation tables (models.py:79-94,
        #                 279-287), no relation embedding (models.py:210, 180)
        # Both of the latter run on the SAME fused generate-and-apply kernels: shared weights are a linear generator
        # applied to the constant context [1], table rows one applied to one-hot(rel) (adding exact zeros).
        if self.concat_rel and self.is_parameter_lookup:
            raise NotImplementedError("concat_rel needs the relation embedding, which do_parameter_lookup does not "
                                      "create (models.py:180, 406-407 would fail the same way)")
        if self.context_rel_conv is not None and (self.is_parameter_lookup or self.context_rel_out is None):
            raise NotImplementedError("generated conv filters (context_rel_conv) are built together with generated "
                                      "FC weights (context_rel_out: [...]) only")
        if self.is_parameter_lookup:
            if self.context_rel_out is None:
                raise NotImplementedError("do_parameter_lookup needs context_rel_out: [] (config_*_param_lookup.yaml)")
            self.variant = "param_lookup"
        else:
            self.variant = "plain" if self.context_rel_out is None else "cpg"
        H_ent = int(conv_in_height)                                 # models.py:261 hard-codes 10
        if self.ent_emb_size % H_ent:
            raise ValueError("entity_embedding_size %d is not a multiple of the conv image height %d "
                             "(models.py:355 would fail the same way)" % (self.ent_emb_size, H_ent))
        self.W = self.ent_emb_size // H_ent
        self.H = H_ent                                              # height of the image the conv sees
        if self.variant == "plain":
            if self.rel_emb_size != self.ent_emb_size:
                raise ValueError("plain ConvE stacks the relation image under the entity image: "
                                 "relation_embedding_size must equal entity_embedding_size (models.py:361-362)")
            self.H = 2 * H_ent                                      # models.py:264-265
        self.OH, self.OW = self.H - self.conv_filter_height + 1, self.W - self.conv_filter_width + 1
        self.C = self.conv_num_channels
        self.F_conv = self.OH * self.OW * self.C                     # models.py:268
        # concat_rel (models.py:270-271, 406-407): the relation embedding is appended to the flattened conv features
        self.F = self.F_conv + (self.rel_emb_size if self.concat_rel else 0)
        self.prec = PREC[prec]                                       # scorer / CPG contraction arithmetic
        self.shard = shard or EntityShard(self.num_ent)
        self.group = process_group
        self.world = self.shard.world
        if self.shard.rows <= 0:
            raise ValueError("%r owns no entity rows: %d entities cannot be sharded %d ways in blocks of %d rows - use "
                             "fewer ranks for this table" % (self.shard, self.num_ent, self.world, self.shard.per))
        # data-parallel front end (SURVEY §8e): every rank receives the GLOBAL batch [Bg], runs lookups' conv / CPG /
        # FC on its own Bg/P rows (batch-norm statistics synchronised), all-gathers q and scores all Bg queries
        # against its entity rows; replicated-parameter gradients are all-reduced in one flat bucket.
        self.dp = bool(data_parallel) and self.world > 1
        if self.dp and self.variant == "param_lookup":
            raise NotImplementedError("data-parallel front end: the per-relation tables' IndexedSlices bookkeeping is "
                                      "single-process; use the replicated front end")
        self.group_big = None
        if self.dp and overlap_grad_allreduce:
            import torch.distributed as dist
            ranks = dist.get_process_group_ranks(process_group) if process_group is not None else None
            self.group_big = dist.new_group(ranks=ranks)          # collective: every rank builds its model here
        self.bug_compat = bool(reference_bug_compat)
        # the entity-gradient GEMM dE = G^T.q (HBM-bound) depends on nothing the rest of the backward pass produces and
        # nothing there depends on it until the head-entity scatter: it is enqueued on a second stream and runs under
        # the latency-bound FC / CPG / conv backward chain (fork / join are captured into the step's CUDA graph)
        self._side = torch.cuda.Stream(device=self.dev)
        self._side_pending = False
        # programmatic dependent launch pays on the launch-bound steps of the named datasets and costs on the HBM-bound
        # step of a 10 M-row table (DESIGN 4.6): per model, by the size of the entity table
        self._pdl = int(self.shard.rows) * int(self.ent_emb_size) <= (64 << 20)
        # CUDA graphs: the device side of a train / eval step is a fixed kernel sequence over pointer-stable buffers
        # (step counter, dropout seed and clip scale live in device memory), so it is captured once per batch size
        # and replayed with one launch.  The sharded path captures its NCCL collectives into the same graph
        # (graphs_multi_gpu; all ranks replay the same sequence).
        self.use_graphs = use_graphs
        self.graphs_multi_gpu = graphs_multi_gpu
        self.graph_kernel_launches = 0
        self.beta1, self.beta2, self.adam_eps = 0.9, 0.999, 1e-8    # amsgrad.py:22-24

        # ---- variables (models.py:203-336); entity-sharded rows are initialised from the full-table
        # stream so that a P-way sharded model holds exactly the rows of the unsharded one.
        gen = torch.Generator().manual_seed(seed)
        dev, f32 = self.dev, torch.float32
        d, dr = self.ent_emb_size, self.rel_emb_size
        # the table is drawn as ONE stream in row chunks (a P-way sharded model then holds exactly the rows of the
        # unsharded one) but only this rank's rows are kept: no [N, d] host copy at 10 M entities
        lim = math.sqrt(6.0 / (self.num_ent + d))
        self.ent_emb = torch.empty(self.shard.rows, d, dtype=f32, device=dev)
        step = 1 << 18
        for r0 in range(0, self.num_ent, step):
            r1 = min(self.num_ent, r0 + step)
            if r0 >= self.shard.hi and init_fast:
                break
            blk = (torch.rand(r1 - r0, d, generator=gen, dtype=f32) * 2 - 1) * lim
            lo, hi = max(r0, self.shard.lo), min(r1, self.shard.hi)
            if lo < hi:
                self.ent_emb[lo - self.shard.lo:hi - self.shard.lo].copy_(blk[lo - r0:hi - r0])
        if init_fast:                                  # later draws need not line up with the full stream
            gen = torch.Generator().manual_seed(seed + 7919)
        self.rel_emb = None
        if self.variant != "param_lookup":
            self.rel_emb = torch.empty(self.num_rel, dr, dtype=f32)
            _xavier_(self.rel_emb, gen)
            self.rel_emb = self.rel_emb.to(dev)
        self.conv_w_gen = self.conv_b_gen = None
        if self.context_rel_conv is None:
            w = torch.empty(self.conv_filter_height, self.conv_filter_width, 1, self.C, dtype=f32)
            _xavier_(w, gen)
            self.conv1_weights = w.to(dev)
            self.conv1_bias = torch.zeros(self.C, dtype=f32, device=dev)
        else:
            # conv filter / bias generated per query (models.py:216-241); applied per example (models.py:375-381)
            cctx = [dr] + list(self.context_rel_conv)
            self.conv_w_gen = ContextualParameterGenerator(
                cctx, "conv1_weights", [self.conv_filter_height, self.conv_filter_width, 1, self.C], False,
                self.context_rel_use_batch_norm, dev, gen)
            self.conv_b_gen = ContextualParameterGenerator(cctx, "conv1_bias", [self.C], True,
                                                           self.context_rel_use_batch_norm, dev, gen)
            self.conv1_weights, self.conv1_bias = self.conv_w_gen, self.conv_b_gen
        if self.variant == "cpg":
            ctx = [dr] + list(self.context_rel_out)
        else:                      # constant context [1] (shared weights) / one-hot(rel) (table rows)
            ctx = [1] if self.variant == "plain" else [self.num_rel]
        self.fc_weights = ContextualParameterGenerator(ctx, "fc_weights", [self.F, d], False,
                                                       self.context_rel_use_batch_norm, dev, gen)
        self.fc_bias = ContextualParameterGenerator(ctx, "fc_bias", [d], self.variant != "param_lookup",
                                                    self.context_rel_use_batch_norm, dev, gen)
        if self.variant == "plain":                                  # Xavier limits of the [F, d] variable
            w = torch.empty(self.F, d, dtype=f32)
            _xavier_(w, gen)
            self.fc_weights.projections[0].copy_(w.view(1, -1))
        self.generators = [self.fc_weights, self.fc_bias] + \
            ([self.conv_w_gen, self.conv_b_gen] if self.conv_w_gen is not None else [])
        self.conv1_bn = _BatchNorm(self.C, dev)
        self.fc_bn = _BatchNorm(d, dev)
        self.pred_bias = torch.zeros(self.shard.rows, dtype=f32, device=dev)
        self.variables = {"ent_emb": self.ent_emb, "conv1_weights": self.conv1_weights,
                          "conv1_bias": self.conv1_bias, "fc_weights": self.fc_weights, "fc_bias": self.fc_bias,
                          "pred_bias": self.pred_bias}
        if self.rel_emb is not None:
            self.variables["rel_emb"] = self.rel_emb                 # models.py:326-327
        if self.variant == "plain":                                  # plain tf variables (models.py:334-340)
            self.variables["fc_weights"] = self.fc_weights.projections[0].view(self.F, d)
            self.variables["fc_bias"] = self.fc_bias.projections[0].view(d)
        self._identity = {}
        self._bufs = {}
        self._graphs = {}
        self._build_trainables()
        self.refresh_prepared()
        # device-resident step state: {lr_t, beta1^t, beta2^t, -} and the dropout seed
        self.step_state = torch.tensor([0.0, self.beta1, self.beta2, 0.0], dtype=f32, device=dev)
        # (data-parallel ranks draw different masks for their different rows: rank offset in the high bits)
        self.seed_dev = torch.tensor([seed * 1000003 + 12345 + ((self.shard.rank << 32) if self.dp else 0)],
                                     dtype=torch.int64, device=dev)
        self.clip_out = torch.zeros(2, dtype=f32, device=dev)       # {scale, norm}
        self.global_step = 0

    # ------------------------------------------------------------------------------------------
    def _build_trainables(self):
        """(name, param, sharded?) for everything optimizer.compute_gradients would return (models.py:198)."""
        tr = [("ent_emb", self.ent_emb, True), ("pred_bias", self.pred_bias, True)]
        if self.rel_emb is not None:
            tr.append(("rel_emb", self.rel_emb, False))
        if self.conv_w_gen is None:
            tr += [("conv1_weights", self.conv1_weights, False), ("conv1_bias", self.conv1_bias, False)]
        self._last_w_name = "fc_weights/CPG/Projection%d" % (len(self.fc_weights.projections) - 1)
        self._last_b_name = "fc_bias/CPG/Projection%d" % (len(self.fc_bias.projections) - 1)
        if self.variant != "cpg":        # tf variable names: 'fc_weights' / 'fc_bias' (models.py:334-340, 86)
            self._last_w_name, self._last_b_name = "fc_weights", "fc_bias"
        for cpg in self.generators:
            if self.variant != "cpg":
                tr.append((cpg.name, cpg.projections[0], False))
                continue
            for i, p in enumerate(cpg.projections):
                tr.append(("%s/CPG/Projection%d" % (cpg.name, i), p, False))
            if cpg.use_batch_norm:
                for i, bn in enumerate(cpg.bns):
                    tr.append(("%s/CPG/Projection%d/BatchNorm/gamma" % (cpg.name, i), bn.gamma, False))
                    tr.append(("%s/CPG/Projection%d/BatchNorm/beta" % (cpg.name, i), bn.beta, False))
        for nm, bn in (("Conv1BN", self.conv1_bn), ("FCBN", self.fc_bn)):
            tr.append((nm + "/gamma", bn.gamma, False))
            tr.append((nm + "/beta", bn.beta, False))
        self.trainables = tr
        self.grads = {n: torch.zeros_like(p) for n, p, _ in tr}
        if self.dp:
            # gradients that every rank only holds a partial sum of (its own rows of the batch) live in ONE flat
            # buffer; BN gamma / beta gradients come out of the synchronised statistics and the entity-table
            # gradients are row-sharded: neither is in the bucket.  The generator's last projection (dc*F*d floats,
            # 66 MB at the WN18RR shape) sits at the front: its all-reduce is issued as soon as the CPG backward has
            # written it, on a second communicator, and overlaps the rest of the backward pass.
            last_w = self._last_w_name
            names = [n for n, _, sh in tr if not sh and not n.endswith("/gamma") and not n.endswith("/beta")]
            names = [last_w] + [n for n in names if n != last_w]
            sizes = [-(-self.grads[n].numel() // 64) * 64 for n in names]
            extra = -(-self.rel_emb.numel() // 64) * 64                      # sum of squared rel_emb slices
            self.flat_grads = torch.zeros(sum(sizes) + extra, dtype=torch.float32, device=self.dev)
            off = 0
            for n, sz in zip(names, sizes):
                self.grads[n] = self.flat_grads[off:off + self.grads[n].numel()].view(self.grads[n].shape)
                off += sz
            self._flat_gsq_rel = self.flat_grads[off:off + self.rel_emb.numel()].view(self.rel_emb.shape)
            self.flat_big, self.flat_small = self.flat_grads[:sizes[0]], self.flat_grads[sizes[0]:]
        # the batch-norm backward kernels write dgamma / dbeta straight into the gradient list (no copies in the step)
        for nm, bn in (("Conv1BN", self.conv1_bn), ("FCBN", self.fc_bn)):
            bn.dgamma, bn.dbeta = self.grads[nm + "/gamma"], self.grads[nm + "/beta"]
        for cpg in self.generators:
            if self.variant == "cpg" and cpg.use_batch_norm:
                for i, bn in enumerate(cpg.bns):
                    bn.dgamma = self.grads["%s/CPG/Projection%d/BatchNorm/gamma" % (cpg.name, i)]
                    bn.dbeta = self.grads["%s/CPG/Projection%d/BatchNorm/beta" % (cpg.name, i)]
        self.vhat = {n: torch.zeros_like(p) for n, p, _ in tr}
        # variables read only through embedding_lookup get an IndexedSlices gradient in TF -> sparse AMSGrad rule
        # (slots accumulate) and a slice-wise contribution to the global norm (include/coper.h, coper_param_desc)
        self.sparse_vars = {"rel_emb"} if self.variant != "param_lookup" else {"fc_weights", "fc_bias"}
        if self.use_negative_sampling:
            # sampled labels (models.py:438-443): ent_emb / pred_bias are read only through gathers as well
            self.sparse_vars |= {"ent_emb", "pred_bias"}
        self.grad_sq = {n: torch.zeros_like(p) for n, p, _ in tr if n in self.sparse_vars}
        if self.dp:
            self.grad_sq["rel_emb"] = self._flat_gsq_rel
        if not self.bug_compat:
            self.m = {n: torch.zeros_like(p) for n, p, _ in tr}
            self.v = {n: torch.zeros_like(p) for n, p, _ in tr}
        else:
            self.m = {n: torch.zeros_like(p) for n, p, _ in tr if n in self.sparse_vars}
            self.v = {n: torch.zeros_like(p) for n, p, _ in tr if n in self.sparse_vars}
        # tensor-pipe operand copies of the two big GEMM operands, kept current by the optimizer kernel
        self.E_prep = self.P_prep = None
        lib = _lib.load()
        d = self.ent_emb_size
        # emission from inside the optimizer kernel needs operand pitch == row length; otherwise re-convert per step
        # (fp16x3: the kernel also tracks max |theta| and rolls the operand's power-of-two scale, csrc/common.cuh)
        self._emit_prepared = d % (4 if self.prec == PREC["tf32x3"] else 8) == 0
        if self.prec != 0:
            Pw = self.fc_weights.projections[-1]
            self.E_prep = torch.zeros(lib.coper_prepared_bytes(self.shard.rows, d, self.prec), dtype=torch.uint8,
                                      device=self.dev)
            self.P_prep = torch.zeros(lib.coper_prepared_bytes(Pw.shape[0] * self.F, d, self.prec), dtype=torch.uint8,
                                      device=self.dev)
        # multi-tensor work list (include/coper.h: coper_param_desc, COPER_MT_CHUNK)
        desc = np.zeros(len(tr), dtype=_lib.PARAM_DESC)
        chunks, offsets = [], [0]
        last_w = self._last_w_name
        for i, (n, p, _) in enumerate(tr):
            desc[i]["theta"], desc[i]["grad"], desc[i]["vhat"] = p.data_ptr(), self.grads[n].data_ptr(), \
                self.vhat[n].data_ptr()
            if n in self.m:
                desc[i]["m"], desc[i]["v"] = self.m[n].data_ptr(), self.v[n].data_ptr()
            if n in self.sparse_vars:
                desc[i]["grad_sq"], desc[i]["mode"] = self.grad_sq[n].data_ptr(), 1
            desc[i]["n"] = p.numel()
            prep = self.E_prep if n == "ent_emb" else self.P_prep if n == last_w else None
            if prep is not None and self._emit_prepared:
                desc[i]["prepared"], desc[i]["prepared_prec"] = prep.data_ptr(), self.prec
            nch = max(1, -(-p.numel() // _lib.MT_CHUNK))
            chunks += [(i, c) for c in range(nch)]
            offsets.append(len(chunks))
        self.mt_desc = torch.from_numpy(desc.view(np.uint8).copy()).to(self.dev)
        # tensor-pipe engines with full 1-N labels: the dE GEMM epilogue and the head-entity scatter hand over the
        # squared norm of the entity gradient (coper.h: COPER_GRAD_NORM_EXTERNAL), so the clip does not re-read [N, d]
        self._norm_fused = self.prec != 0 and not self.use_negative_sampling
        desc_ext = desc.copy()
        desc_ext[0]["mode"] |= 2
        assert tr[0][0] == "ent_emb"
        self.mt_desc_ext = torch.from_numpy(desc_ext.view(np.uint8).copy()).to(self.dev)
        # ... and the norm pass does not even launch blocks for that tensor's chunks (160 k of them at 10 M entities)
        chunks_ext = [c for c in chunks if c[0] != 0]
        n0 = len(chunks) - len(chunks_ext)
        self.mt_chunks_ext = torch.tensor(chunks_ext or [(1, 0)], dtype=torch.int32).to(self.dev)
        self.mt_offsets_ext = torch.tensor([0] + [max(0, o - n0) for o in offsets[1:]], dtype=torch.int32).to(self.dev)
        self.mt_nchunks_ext = len(chunks_ext)
        self.dE_sumsq = torch.zeros(1, dtype=torch.float64, device=self.dev)
        # arrival counter of the single-launch batch-norm statistics (coper_bn_stats_finalize); zero between launches
        self.sync_word = torch.zeros(1, dtype=torch.int32, device=self.dev)
        self.norm_delta = torch.zeros(4096, dtype=torch.float64, device=self.dev)
        self._norm_fused_now = False
        self._norm_delta_n = 0
        self.mt_chunks = torch.tensor(chunks, dtype=torch.int32).to(self.dev)
        self.mt_offsets = torch.tensor(offsets, dtype=torch.int32).to(self.dev)
        self.mt_nchunks = len(chunks)
        self.mt_partials = torch.zeros(len(chunks), dtype=torch.float64, device=self.dev)
        self.sumsq = torch.zeros(len(tr), dtype=torch.float64, device=self.dev)

    def _ident(self, C):
        if C not in self._identity:
            f = dict(dtype=torch.float32, device=self.dev)
            self._identity[C] = (torch.ones(C, **f), torch.zeros(C, **f))
        return self._identity[C]

    # ------------------------------------------------------------------------------------------
    def load_variables(self, params: Dict):
        """Load variables from the oracle's naming (numpy arrays; full, unsharded tables)."""
        def put(dst, src):
            dst.copy_(torch.as_tensor(np.ascontiguousarray(src), dtype=torch.float32).reshape(dst.shape))
        s = self.shard
        put(self.ent_emb, params["ent_emb"][s.lo:s.hi])
        put(self.pred_bias, params["pred_bias"][s.lo:s.hi])
        if self.rel_emb is not None:
            put(self.rel_emb, params["rel_emb"])
        if self.conv_w_gen is None:
            put(self.conv1_weights, params["conv1_weights"])
            put(self.conv1_bias, params["conv1_bias"])
        for cpg, key in [(g, g.name) for g in self.generators]:
            for t, a in zip(cpg.projections, params[key + "_proj"]):
                put(t, a)
            for bn, b in zip(cpg.bns, params[key + "_bn"]):
                self._put_bn(bn, b)
        self._put_bn(self.conv1_bn, params["Conv1BN"])
        self._put_bn(self.fc_bn, params["FCBN"])
        self.refresh_prepared()

    # checkpoint = every variable + BN moving statistics + optimizer slots + step state (tf.train.Saver over all
    # global variables, run_cpg.py:189,252); entity-sharded models save / load their own rows (one file per rank)
    def state_dict(self) -> Dict[str, torch.Tensor]:
        sd = {"var/" + n: p for n, p, _ in self.trainables}
        sd.update({"vhat/" + n: v for n, v in self.vhat.items()})
        sd.update({"m/" + n: v for n, v in self.m.items()})
        sd.update({"v/" + n: v for n, v in self.v.items()})
        bns = [("Conv1BN", self.conv1_bn), ("FCBN", self.fc_bn)]
        for cpg in self.generators:
            bns += [("%s/CPG/Projection%d/BatchNorm" % (cpg.name, i), bn) for i, bn in enumerate(cpg.bns)]
        for nm, bn in bns:
            sd["bn/%s/moving_mean" % nm], sd["bn/%s/moving_var" % nm] = bn.moving_mean, bn.moving_var
            if not any(nm + "/gamma" == n for n, _, _ in self.trainables):      # BN without trainable scale/shift
                sd["bn/%s/gamma" % nm], sd["bn/%s/beta" % nm] = bn.gamma, bn.beta
        sd["step_state"], sd["seed_dev"] = self.step_state, self.seed_dev
        return sd

    def save_checkpoint(self, path: str):
        if self.world > 1:
            path = "%s.rank%d" % (path, self.shard.rank)
        torch.save({"state": {k: v.detach().cpu() for k, v in self.state_dict().items()},
                    "global_step": self.global_step, "shard": (self.shard.lo, self.shard.hi, self.num_ent)}, path)

    def load_checkpoint(self, path: str):
        if self.world > 1:
            path = "%s.rank%d" % (path, self.shard.rank)
        ck = torch.load(path, map_location="cpu")
        if tuple(ck["shard"]) != (self.shard.lo, self.shard.hi, self.num_ent):
            raise ValueError("checkpoint was written for entity rows %s, this model owns %s" % (
                ck["shard"], (self.shard.lo, self.shard.hi, self.num_ent)))
        own = self.state_dict()
        missing = set(own) - set(ck["state"])
        if missing:
            raise KeyError("checkpoint lacks %s" % sorted(missing))
        for k, dst in own.items():
            dst.copy_(ck["state"][k].to(dst.dtype))
        self.global_step = int(ck["global_step"])
        self.refresh_prepared()

    def full_entity_table(self) -> torch.Tensor:
        """[num_ent, d] on every rank: all-gather of the (padded) row shards (run_cpg.py:245-248 pickles the table)."""
        if self.world == 1:
            return self.ent_emb
        per, d = self.shard.per, self.ent_emb_size
        mine = torch.zeros(per, d, dtype=torch.float32, device=self.dev)
        mine[:self.shard.rows].copy_(self.ent_emb)
        out = torch.empty(self.world * per, d, dtype=torch.float32, device=self.dev)
        sharding.gather_batch(out, mine, self.world, self.group)
        return out[:self.num_ent]

    def refresh_prepared(self):
        """(Re)build the tensor-pipe operand copies after the variables were written from outside the optimizer."""
        if self.E_prep is None:
            return
        d = self.ent_emb_size
        Pw = self.fc_weights.projections[-1]
        call("coper_prepare_operand", ptr(self.ent_emb), self.shard.rows, d, d, self.prec, ptr(self.E_prep))
        call("coper_prepare_operand", ptr(Pw), Pw.shape[0] * self.F, d, d, self.prec, ptr(self.P_prep))

    @staticmethod
    def _put_bn(bn, b):
        for k in ("gamma", "beta", "moving_mean", "moving_var"):
            getattr(bn, k).copy_(torch.as_tensor(np.asarray(b[k]), dtype=torch.float32))

    # ------------------------------------------------------------------------------------------
    def _buffers(self, B: int, key=None):
        """The batch slot of batch size B (key: the slot's name in ``_bufs``, default B)."""
        return _slot(self._bufs, B if key is None else key, _BatchSlot, self, B)

    def _local_buffers(self, bg):
        """Data-parallel front end: buffer set of this rank's Bg/P rows; its query ids alias the global batch."""
        P, r = self.world, self.shard.rank
        if bg.B % P:
            raise ValueError("data-parallel batch %d is not a multiple of the world size %d" % (bg.B, P))
        Bl = bg.B // P
        bl = self._buffers(Bl, key=("dp", bg.B))
        bl.e1, bl.rel, bl.e2 = (t[r * Bl:(r + 1) * Bl] for t in (bg.e1, bg.rel, bg.e2))
        return bl

    def _scores_buf(self, b):
        if b.S is None:
            b.S = torch.zeros(b.B, b.ld, dtype=torch.float32, device=self.dev)
        return b.S

    def _grad_buf(self, b):
        if b.G is None:
            nbytes = _lib.load().coper_score1n_bce_G_bytes(b.B, self.shard.rows, self.prec)
            b.G = torch.zeros(-(-nbytes // 4), dtype=torch.float32, device=self.dev)
        return b.G

    def _ensure_csr(self, b, nnz):
        if b.csr_cap < nnz:
            cap = max(1024, int(nnz * 1.5))
            b.col = torch.zeros(cap, dtype=torch.int32, device=self.dev)
            b.csr_gen += 1
            b.h_col = torch.zeros(cap, dtype=torch.int32).pin_memory()
            b.h_col_np = b.h_col.numpy()
            b.csr_cap = cap

    # ------------------------------------------------------------------------------------------
    def stage_batch(self, batch: Dict, need_e2: bool = False):
        """Host batch -> device buffers.  Schema follows models.py:135-152: int64 ``e1``/``rel``/``e2`` [B];
        ``e2_multi`` either as the reference's dense fp32 multi-hot [B, N] or, as the TFRecord stores it
        (data.py:574-594), the list of positive ids in CSR form (``e2_multi_rowptr``, ``e2_multi_col``).
        Returns (buffers, nnz or None)."""
        e1 = batch["e1"]
        B = int(e1.shape[0])
        b = self._buffers(B)
        if b.h2d_event is not None:
            b.h2d_event.synchronize()          # previous async copies out of the pinned staging are done
        s = self.shard
        on_device = isinstance(e1, torch.Tensor) and e1.is_cuda
        has_csr = "e2_multi_rowptr" in batch
        if on_device:
            b.e1.copy_(e1)
            b.rel.copy_(batch["rel"])
            if need_e2:
                b.e2.copy_(batch["e2"])
        else:
            b.h_idx_np[0] = e1
            b.h_idx_np[1] = batch["rel"]
            if need_e2:
                b.h_idx_np[2] = batch["e2"]
        if has_csr:
            rp, col = batch["e2_multi_rowptr"], batch["e2_multi_col"]
            nnz = int(col.shape[0])
            self._ensure_csr(b, nnz)
            if isinstance(rp, torch.Tensor) and rp.is_cuda:
                b.rowptr.copy_(rp)
                b.col[:nnz].copy_(col)
                if not on_device:
                    b.d_head[:6 * B].copy_(b.h_head[:6 * B], non_blocking=True)
            else:
                b.h_rowptr_np[:] = rp
                b.h_col_np[:nnz] = col
                if on_device:
                    b.rowptr.copy_(b.h_head[6 * B:6 * B + B + 1], non_blocking=True)
                else:
                    b.d_head.copy_(b.h_head, non_blocking=True)          # ids + row pointers: one copy
                b.col[:nnz].copy_(b.h_col[:nnz], non_blocking=True)
            if self.prec == 0:
                call("coper_csr_to_bits", ptr(b.rowptr), ptr(b.col), B, s.lo, s.hi, ptr(b.bits))
            else:
                call("coper_csr_to_bits_t", ptr(b.rowptr), ptr(b.col), B, s.lo, s.hi, ptr(b.bitsT))
        elif not on_device:
            b.d_head[:6 * B].copy_(b.h_head[:6 * B], non_blocking=True)
        if not has_csr and batch.get("e2_multi") is not None:
            dense = batch["e2_multi"]
            if not (isinstance(dense, torch.Tensor) and dense.is_cuda):
                dense = torch.as_tensor(np.asarray(dense), dtype=torch.float32).to(self.dev, non_blocking=True)
            if s.world > 1:
                dense = dense[:, s.lo:s.hi].contiguous()
            dense = dense.contiguous()
            if self.prec == 0:
                call("coper_dense_to_bits", ptr(dense), B, s.rows, ptr(b.bits))
            else:
                call("coper_dense_to_bits_t", ptr(dense), B, s.rows, s.rows, ptr(b.bitsT))
        if b.h2d_event is None:
            b.h2d_event = torch.cuda.Event()
        b.h2d_event.record()
        return b

    # ------------------------------------------------------------------------------------------
    def _bn_forward(self, bn: _BatchNorm, x, R, C, b, use_batch, is_train, bessel, relu, keep_post, salt, out):
        lib = _lib.load()
        nch = 0
        stat, Rt = b.stat, R
        if use_batch and not self.dp:        # statistics + finalize: one launch (the last block to arrive finalises)
            call("coper_bn_stats_finalize", ptr(x), R, C, ptr(b.stat), ptr(self.sync_word), ptr(bn.gamma), ptr(bn.beta),
                 ptr(bn.moving_mean), ptr(bn.moving_var), self.batch_norm_momentum, BN_EPS, int(is_train), int(bessel),
                 ptr(bn.a), ptr(bn.b), ptr(bn.mean), ptr(bn.invstd))
            call("coper_bn_act_fwd", ptr(x), R, C, ptr(bn.a), ptr(bn.b), int(relu), keep_post, ptr(self.seed_dev), salt,
                 ptr(out))
            return
        if not use_batch and not is_train and keep_post >= 1.0:      # inference: moving statistics, one launch
            call("coper_bn_act_fwd_moving", ptr(x), R, C, ptr(bn.gamma), ptr(bn.beta), ptr(bn.moving_mean),
                 ptr(bn.moving_var), BN_EPS, int(relu), ptr(out))
            return
        if use_batch:
            nch = lib.coper_colstats_chunks(R)
            call("coper_colstats", ptr(x), R, C, ptr(b.stat))
            if self.dp:          # synchronised batch statistics: every rank finalises over all ranks' chunk partials
                stat, nch, Rt = self._gather_stats(b, nch * C * 2), nch * self.world, R * self.world
        call("coper_bn_finalize", ptr(stat), nch, Rt, C, ptr(bn.gamma), ptr(bn.beta), ptr(bn.moving_mean),
             ptr(bn.moving_var), self.batch_norm_momentum, BN_EPS, int(use_batch), int(use_batch and is_train),
             int(bessel), ptr(bn.a), ptr(bn.b), ptr(bn.mean), ptr(bn.invstd))
        call("coper_bn_act_fwd", ptr(x), R, C, ptr(bn.a), ptr(bn.b), int(relu), keep_post, ptr(self.seed_dev), salt,
             ptr(out))

    def _bn_backward(self, bn: _BatchNorm, dout, x, R, C, b, use_batch, relu, keep_post, salt_post, keep_pre,
                     salt_pre, dx, apply=True):
        """apply=False: statistics only (dgamma, dbeta, c1, c2) - the caller's next kernel forms dx itself."""
        lib = _lib.load()
        nch = lib.coper_colstats_chunks(R)
        if not self.dp:
            call("coper_bn_act_bwd_stats_finalize", ptr(dout), ptr(x), R, C, ptr(bn.a), ptr(bn.b), ptr(bn.mean),
                 ptr(bn.invstd), int(relu), keep_post, ptr(self.seed_dev), salt_post, ptr(b.stat), ptr(self.sync_word),
                 int(use_batch), ptr(bn.dgamma), ptr(bn.dbeta), ptr(bn.c1), ptr(bn.c2))
        else:
            call("coper_bn_act_bwd_stats", ptr(dout), ptr(x), R, C, ptr(bn.a), ptr(bn.b), ptr(bn.mean), ptr(bn.invstd),
                 int(relu), keep_post, ptr(self.seed_dev), salt_post, ptr(b.stat))
        stat, Rt = b.stat, R
        if self.dp:              # gradient statistics over the global batch (also makes dgamma / dbeta global)
            stat, nch, Rt = self._gather_stats(b, nch * C * 2), nch * self.world, R * self.world
            call("coper_bn_act_bwd_finalize", ptr(stat), nch, Rt, C, int(use_batch), ptr(bn.dgamma), ptr(bn.dbeta),
                 ptr(bn.c1), ptr(bn.c2))
        if apply:
            call("coper_bn_act_bwd_apply", ptr(dout), ptr(x), R, C, ptr(bn.a), ptr(bn.b), ptr(bn.mean), ptr(bn.invstd),
                 ptr(bn.c1), ptr(bn.c2), int(relu), keep_post, ptr(self.seed_dev), salt_post, keep_pre, salt_pre, ptr(dx))

    def _gather_stats(self, b, n):
        if b.stat_all is None:
            b.stat_all = torch.zeros(self.world * b.stat.numel(), dtype=torch.float32, device=self.dev)
        return sharding.gather_stat_partials(b.stat_all[:self.world * n], b.stat[:n], self.world, self.group)

    def _ctx_forward(self, cpg: ContextualParameterGenerator, net_id, b, is_train):
        """Hidden layers of CPG.generate (models.py:59-68): matmul -> [BN] -> relu -> dropout."""
        h = b.r
        B = b.B
        keep = 1.0 - (self.context_rel_dropout if is_train else 0.0)
        bufs = b.ctx[cpg.name]
        for i, n in enumerate(cpg.hidden):
            P = cpg.projections[i]
            call("coper_sgemm", 0, 0, B, n, P.shape[0], ptr(h), P.shape[0], ptr(P), n, ptr(bufs["pre"][i]), n, 0)
            salt = SALT_CTX + ((net_id * 64 + i) << 32)
            if cpg.use_batch_norm:
                use_batch = self.batch_norm_train_stats and is_train
                self._bn_forward(cpg.bns[i], bufs["pre"][i], B, n, b, use_batch, is_train, False, True, keep, salt,
                                 bufs["act"][i])
            else:
                one, zero = self._ident(n)
                call("coper_bn_act_fwd", ptr(bufs["pre"][i]), B, n, ptr(one), ptr(zero), 1, keep,
                     ptr(self.seed_dev), salt, ptr(bufs["act"][i]))
            h = bufs["act"][i]
        return h

    def _ctx_backward(self, cpg: ContextualParameterGenerator, net_id, b, dctx, dr_out, accumulate):
        """Back through the hidden layers; writes projection/BN grads, accumulates into dr_out [B,dr]."""
        B = b.B
        bufs = b.ctx[cpg.name]
        keep = 1.0 - self.context_rel_dropout
        dh = dctx
        for i in reversed(range(len(cpg.hidden))):
            n = cpg.hidden[i]
            P = cpg.projections[i]
            inp = b.r if i == 0 else bufs["act"][i - 1]
            salt = SALT_CTX + ((net_id * 64 + i) << 32)
            if cpg.use_batch_norm:
                bn = cpg.bns[i]
                use_batch = self.batch_norm_train_stats
                self._bn_backward(bn, dh, bufs["pre"][i], B, n, b, use_batch, True, keep, salt, 1.0, 0,
                                  bufs["dpre"][i])
            else:
                one, zero = self._ident(n)
                call("coper_bn_act_bwd_apply", ptr(dh), ptr(bufs["pre"][i]), B, n, ptr(one), ptr(zero), ptr(zero),
                     ptr(one), ptr(zero), ptr(zero), 1, keep, ptr(self.seed_dev), salt, 1.0, 0, ptr(bufs["dpre"][i]))
            k_in = P.shape[0]
            # dP_i = inp^T . dpre ; dinp = dpre . P_i^T
            call("coper_sgemm", 1, 0, k_in, n, B, ptr(inp), k_in, ptr(bufs["dpre"][i]), n,
                 ptr(self.grads["%s/CPG/Projection%d" % (cpg.name, i)]), n, 0)
            if i == 0:
                call("coper_sgemm", 0, 1, B, k_in, n, ptr(bufs["dpre"][i]), n, ptr(P), n, ptr(dr_out), k_in,
                     int(accumulate))
            else:
                call("coper_sgemm", 0, 1, B, k_in, n, ptr(bufs["dpre"][i]), n, ptr(P), n, ptr(bufs["dact"][i - 1]),
                     k_in, 0)
                dh = bufs["dact"][i - 1]
        if not cpg.hidden:
            if accumulate:
                dr_out.add_(dctx)     # g_linear: context == relation embedding
            else:
                dr_out.copy_(dctx)

    # ------------------------------------------------------------------------------------------
    def _forward_q(self, b, is_train: bool, advance: bool = False):
        """Lookups -> conv block -> fused CPG-FC -> FC block; leaves q in b.q (models.py:176-183, 354-426)."""
        B, d = b.B, self.ent_emb_size
        s = self.shard
        # both lookups and (training) the step-state advance: one launch
        rel = self.rel_emb is not None
        call("coper_gather_rows2", ptr(self.ent_emb), s.lo, s.hi, d, ptr(b.e1), B, ptr(b.x0),
             ptr(self.rel_emb) if rel else None, 0, self.num_rel if rel else 0, self.rel_emb_size if rel else 0,
             ptr(b.rel) if rel else None, B if rel else 0, ptr(b.r) if rel else None,
             ptr(self.step_state) if advance else None, ptr(self.seed_dev) if advance else None,
             self.learning_rate, self.beta1, self.beta2)
        sharding.exchange_rows(b.x0, self.world, self.group)
        self._front_end(b, is_train, gather_rel=False)

    def _front_end(self, b, is_train: bool, gather_rel: bool = True):
        """b.x0, b.rel -> b.q for the rows of buffer set b (conv block, fused CPG-FC, FC block)."""
        B, d, dr, F, C = b.B, self.ent_emb_size, self.rel_emb_size, self.F, self.C
        x_img = b.x0
        if self.rel_emb is not None and gather_rel:
            call("coper_gather_rows", ptr(self.rel_emb), 0, self.num_rel, dr, ptr(b.rel), B, ptr(b.r))
        if self.variant == "plain":          # models.py:360-362: rows 0..H/2 = entity image, the rest = relation image
            b.xc[:, :d].copy_(b.x0)
            b.xc[:, d:].copy_(b.r)
            x_img = b.xc
        elif self.variant == "param_lookup":
            b.cconst.zero_()
            b.cconst.scatter_(1, b.rel.view(-1, 1), 1.0)
        if self.conv_w_gen is None:
            call("coper_conv_fwd", ptr(x_img), B, self.H, self.W, ptr(self.conv1_weights), ptr(self.conv1_bias),
                 self.conv_filter_height, self.conv_filter_width, C, 0, ptr(b.z))
        else:
            KK = self.conv_filter_height * self.conv_filter_width * C
            b.ccw = self._ctx_forward(self.conv_w_gen, 2, b, is_train)
            b.ccb = self._ctx_forward(self.conv_b_gen, 3, b, is_train)
            Pc, Pcb = self.conv_w_gen.projections[-1], self.conv_b_gen.projections[-1]
            call("coper_sgemm", 0, 0, B, KK, Pc.shape[0], ptr(b.ccw), Pc.shape[0], ptr(Pc), KK, ptr(b.wq), KK, 0)
            call("coper_sgemm", 0, 0, B, C, Pcb.shape[0], ptr(b.ccb), Pcb.shape[0], ptr(Pcb), C, ptr(b.bq), C, 0)
            call("coper_conv_fwd", ptr(x_img), B, self.H, self.W, ptr(b.wq), ptr(b.bq),
                 self.conv_filter_height, self.conv_filter_width, C, 1, ptr(b.z))
        use_batch = self.batch_norm_train_stats and is_train
        keep1 = 1.0 - (self.hidden_dropout if is_train else 0.0)
        self._bn_forward(self.conv1_bn, b.z, B * self.OH * self.OW, C, b, use_batch, is_train, True, True, keep1,
                         SALT_FEATURE_MAP, b.fconv)
        if self.concat_rel:                  # tf.concat([fc_input, rel_emb], axis=1)  (models.py:406-407)
            b.f[:, :self.F_conv].copy_(b.fconv)
            b.f[:, self.F_conv:].copy_(b.r)
        if self.variant == "cpg":
            cw = self._ctx_forward(self.fc_weights, 0, b, is_train)
            cb = self._ctx_forward(self.fc_bias, 1, b, is_train)
        else:
            cw = cb = b.cconst
        Pw, Pb = self.fc_weights.projections[-1], self.fc_bias.projections[-1]
        keep2 = 1.0 - (self.output_dropout if is_train else 0.0)
        call("coper_cpg_fc_fwd", ptr(cw), ptr(b.f), ptr(Pw), ptr(self.P_prep), ptr(cb), ptr(Pb), B, Pw.shape[0], F, d,
             Pb.shape[0], keep2, ptr(self.seed_dev), SALT_OUTPUT, ptr(b.y), ptr(b.ws_cpg), b.ws_cpg_bytes, self.prec)
        self._bn_forward(self.fc_bn, b.y, B, d, b, use_batch, is_train, False, True, 1.0, 0, b.q)
        b.cw, b.cb = cw, cb

    def _forward_q_dp(self, bg, bl, is_train: bool):
        """Data-parallel forward: masked gather of all Bg head rows -> reduce-scatter (each rank receives ITS rows,
        summed over the owning shards) -> front end on Bg/P rows -> all-gather q."""
        s, d = self.shard, self.ent_emb_size
        call("coper_gather_rows", ptr(self.ent_emb), s.lo, s.hi, d, ptr(bg.e1), bg.B, ptr(bg.x0))
        sharding.scatter_rows(bg.x0, bl.x0, self.world, self.group)
        self._front_end(bl, is_train)
        sharding.gather_batch(bg.q, bl.q, self.world, self.group)

    def _eval_q(self, b):
        """Evaluation forward pass: q of every query of b (moving statistics, no dropout).  A batch that does not split
        evenly over the ranks runs the data-parallel front end replicated, with identical results."""
        if self.dp and b.B % self.world == 0:
            self._forward_q_dp(b, self._local_buffers(b), False)
        else:
            self._forward_q(b, False)

    def _train_device(self, b, apply: bool = True):
        """fwd + bwd (+ clip + AMSGrad when apply) on staged buffers; everything is enqueued, nothing syncs.
        apply=False leaves the gradients for a later _clip_and_apply()."""
        self._train_device_impl(b, self._local_buffers(b) if self.dp else b, apply)

    def _train_device_impl(self, bg, b, apply):
        """bg: buffers of the batch the scorer sees; b: buffers of the rows this rank's front end owns
        (b is bg unless the front end is data-parallel)."""
        dp = b is not bg
        B, d, dr, F, C = b.B, self.ent_emb_size, self.rel_emb_size, self.F, self.C
        s, g = self.shard, self.grads
        Ns = s.rows
        if dp:
            call("coper_step_state_advance", ptr(self.step_state), ptr(self.seed_dev), self.learning_rate, self.beta1,
                 self.beta2)
            self._forward_q_dp(bg, b, True)
        else:
            self._forward_q(b, True, advance=True)
        pos = np.float32(np.float32(1.0 - self.label_smoothing_epsilon) * np.float32(1.0)
                         + np.float32(1.0 / self.num_ent))                     # models.py:450 in fp32
        neg = np.float32(1.0 / self.num_ent)
        inv_count = 1.0 / (float(bg.B) * float(self.num_ent))                # mean over B*N (models.py:451)
        self._norm_fused_now = self._norm_fused and bg.B <= 4096       # (the scatter correction is the small-M kernel's)
        rel_cleared = loss_done = False
        if self.use_negative_sampling:
            self._sampled_scorer(bg)
        elif self._norm_fused_now:
            call("coper_score1n_bce_fwd_bwd_norm", ptr(bg.q), ptr(self.ent_emb), ptr(self.E_prep), ptr(self.pred_bias),
                 ptr(bg.bitsT), bg.B, Ns, d, float(pos), float(neg), inv_count, ptr(bg.loss_sum),
                 ptr(self._grad_buf(bg)), bg.ld, ptr(bg.dq), None, ptr(g["pred_bias"]), ptr(self.dE_sumsq), ptr(bg.ws),
                 bg.ws_bytes, self.prec)
            self._side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(self._side):
                if self.rel_emb is not None:     # cleared here, off the main chain, for the scatter after the join
                    g["rel_emb"].zero_()
                    self.grad_sq["rel_emb"].zero_()
                    rel_cleared = True
                call("coper_score1n_bce_dE", ptr(self._grad_buf(bg)), bg.B, Ns, d, inv_count, ptr(g["ent_emb"]),
                     ptr(self.dE_sumsq), ptr(g["pred_bias"]), ptr(bg.ws), bg.ws_bytes, self.prec)
                if self.world == 1:              # the mean loss the caller reads (models.py:451)
                    torch.div(bg.loss_sum, float(bg.B) * float(self.num_ent), out=bg.loss_mean)
                    loss_done = True
            self._side_pending = True
        else:
            call("coper_score1n_bce_fwd_bwd", ptr(bg.q), ptr(self.ent_emb), ptr(self.E_prep), ptr(self.pred_bias),
                 ptr(bg.bits if self.prec == 0 else bg.bitsT), bg.B, Ns, d, float(pos), float(neg), inv_count,
                 ptr(bg.loss_sum), ptr(self._grad_buf(bg)), bg.ld, ptr(bg.dq), ptr(g["ent_emb"]),
                 ptr(g["pred_bias"]), ptr(bg.ws), bg.ws_bytes, self.prec)
        # entity-sharded scorer: every rank scored all B queries against its rows -> sum the partial loss and
        # the partial dq = G_shard . E_shard (SURVEY §8e step 4); dE / dbias stay local.
        if dp:      # each rank only needs the summed dq of its own rows
            sharding.scatter_dq(bg.dq, b.dq, bg.loss_sum, self.world, self.group)
        else:
            sharding.reduce_scorer_partials(b.loss_sum, b.dq, self.world, self.group)
        if not loss_done and not self.use_negative_sampling:
            torch.div(bg.loss_sum, float(bg.B) * float(self.num_ent), out=bg.loss_mean)
        use_batch = self.batch_norm_train_stats
        keep1, keep2 = 1.0 - self.hidden_dropout, 1.0 - self.output_dropout
        # FC block backward: relu -> FCBN -> output dropout (models.py:414-419)
        self._bn_backward(self.fc_bn, b.dq, b.y, B, d, b, use_batch, True, 1.0, 0, keep2, SALT_OUTPUT, b.dy)
        Pw, Pb = self.fc_weights.projections[-1], self.fc_bias.projections[-1]
        nw, nb = len(self.fc_weights.projections) - 1, len(self.fc_bias.projections) - 1
        # the generator's weight gradients (dP^, dPb) feed nothing but the clip / optimizer: they are computed on the
        # side stream while the chain through df / dc continues (DESIGN 4.5)
        split_w = not dp and self.variant != "param_lookup"
        reuse = CPG_BWD_REUSE_FWD if self.prec != 0 else 0
        # g_linear (no hidden generator layers: both contexts ARE the relation embedding): d rel_emb = dc + dcb is formed
        # by the call itself - dc lands in b.dr, the bias generator's dcb is added to it
        linear = self.variant == "cpg" and not self.fc_weights.hidden and not self.fc_bias.hidden
        if linear:
            reuse |= CPG_BWD_DCB_ACCUMULATE
        dcw_out, dcb_out = (b.dr, b.dr) if linear else (b.dcw, b.dcb)
        cpg_bwd_args = (ptr(b.cw), ptr(b.f), ptr(Pw), ptr(self.P_prep), ptr(b.cb), ptr(Pb), ptr(b.dy), B,
                        Pw.shape[0], F, d, Pb.shape[0], ptr(g[self._last_w_name]), ptr(g[self._last_b_name]),
                        ptr(b.df), ptr(dcw_out), ptr(dcb_out), ptr(b.ws_cpg), b.ws_cpg_bytes, self.prec)
        call("coper_cpg_fc_bwd", *cpg_bwd_args, reuse | (CPG_BWD_INPUT_GRADS_ONLY if split_w else 0))
        if split_w:
            self._side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(self._side):
                call("coper_cpg_fc_bwd", *cpg_bwd_args, reuse | CPG_BWD_WEIGHT_GRADS_ONLY)
            self._side_pending = True
        if self.variant == "param_lookup":
            # the tables are read through embedding_lookup (models.py:91): IndexedSlices gradients, one [F*d] / [d]
            # slice per query.  The slice-wise norm and the sparse AMSGrad rule need, per table row, the sum of the
            # SQUARED slices = onehot^T . (f^2 (x) dy^2): the same contraction on the squared operands.
            torch.mul(b.f, b.f, out=b.f_sq)
            torch.mul(b.dy, b.dy, out=b.dy_sq)
            call("coper_cpg_fc_bwd", ptr(b.cw), ptr(b.f_sq), ptr(Pw), ptr(self.P_prep), ptr(b.cb), ptr(Pb),
                 ptr(b.dy_sq), B, Pw.shape[0], F, d, Pb.shape[0], ptr(self.grad_sq["fc_weights"]),
                 ptr(self.grad_sq["fc_bias"]), ptr(b.df_scratch), ptr(b.dcw), ptr(b.dcb), ptr(b.ws_cpg),
                 b.ws_cpg_bytes, self.prec, 0)
        big_work = None
        if dp and self.group_big is not None:
            big_work = sharding.reduce_replicated_grads(self.flat_big, self.world, self.group_big, async_op=True)
        if self.variant == "cpg" and not linear:
            self._ctx_backward(self.fc_weights, 0, b, b.dcw, b.dr, False)
            self._ctx_backward(self.fc_bias, 1, b, b.dcb, b.dr, True)
        # conv block backward: feature-map dropout -> relu -> Conv1BN -> conv (models.py:373-391)
        R1 = B * self.OH * self.OW
        if self.concat_rel:                  # tf.concat backward: conv part | d rel_emb (added to the generators' part)
            b.dfconv.copy_(b.df[:, :self.F_conv])
            if self.variant == "cpg":
                b.dr.add_(b.df[:, self.F_conv:])
        # shared filters: the Conv1BN backward is folded into the conv backward (dz never goes to HBM)
        fold = self.conv_w_gen is None
        self._bn_backward(self.conv1_bn, b.dfconv, b.z, R1, C, b, use_batch, True, keep1, SALT_FEATURE_MAP, 1.0, 0, b.dz,
                          apply=not fold)
        plain = self.variant == "plain"
        KK = self.conv_filter_height * self.conv_filter_width * C
        if self.conv_w_gen is not None:
            # per-example filters: dz -> dx0 and, per query, dWq [B, KK] / dbq [B, C]; then back through the generators
            call("coper_conv_bwd", ptr(b.dz), ptr(b.x0), B, self.H, self.W, ptr(b.wq), self.conv_filter_height,
                 self.conv_filter_width, C, 1, ptr(b.dx0), ptr(b.dwc_part), ptr(b.dbc_part))
            for gen_, ctx_, dq_, dctx_, width, net in ((self.conv_w_gen, b.ccw, b.dwc_part, b.dccw, KK, 2),
                                                       (self.conv_b_gen, b.ccb, b.dbc_part, b.dccb, C, 3)):
                Pl = gen_.projections[-1]
                dcc = Pl.shape[0]
                last = "%s/CPG/Projection%d" % (gen_.name, len(gen_.projections) - 1)
                call("coper_sgemm", 1, 0, dcc, width, B, ptr(ctx_), dcc, ptr(dq_), width, ptr(g[last]), width, 0)
                call("coper_sgemm", 0, 1, B, dcc, width, ptr(dq_), width, ptr(Pl), width, ptr(dctx_), dcc, 0)
                self._ctx_backward(gen_, net, b, dctx_, b.dr, True)
        else:
            bn1 = self.conv1_bn
            call("coper_conv_bwd_bn", ptr(b.dfconv), ptr(b.z), ptr(b.xc if plain else b.x0), B, self.H, self.W,
                 ptr(self.conv1_weights), self.conv_filter_height, self.conv_filter_width, C, 0, ptr(bn1.a), ptr(bn1.b),
                 ptr(bn1.mean), ptr(bn1.invstd), ptr(bn1.c1), ptr(bn1.c2), 1, keep1, ptr(self.seed_dev),
                 SALT_FEATURE_MAP, ptr(b.dxc if plain else b.dx0), ptr(b.dwc_part), ptr(b.dbc_part), ptr(b.dz))
            if plain:                            # tf.concat backward: the two halves of the stacked image
                b.dx0.copy_(b.dxc[:, :d])
                b.dr.copy_(b.dxc[:, d:])
                if self.concat_rel:
                    b.dr.add_(b.df[:, self.F_conv:])
            slabs = _lib.load().coper_conv_bwd_slabs(B, self.H, self.W, self.conv_filter_height,
                                                     self.conv_filter_width, C, 0)
            call("coper_reduce_partials2", ptr(b.dwc_part), KK, ptr(g["conv1_weights"]), ptr(b.dbc_part), C,
                 ptr(g["conv1_bias"]), slabs, 1.0, 0)
        # gradients of the two embedding gathers (models.py:176-178): deterministic segmented scatter
        # IndexedSlices bookkeeping (rel_emb always; ent_emb with sampled labels): the same pass also accumulates the
        # per-row sums of the SQUARED slices (slice-wise global norm + sparse AMSGrad rule)
        small = B <= 4096
        gsq_e = self.grad_sq["ent_emb"] if self.use_negative_sampling else None
        if dp:      # every shard needs dx0 of ALL queries whose head entity it owns
            sharding.gather_batch(bg.dx0, b.dx0, self.world, self.group)
        if self._side_pending:      # join: the scatter below adds into dE, the clip reads every gradient
            torch.cuda.current_stream().wait_stream(self._side)
            self._side_pending = False
        rel = self.rel_emb is not None
        if rel and not rel_cleared:
            g["rel_emb"].zero_()
            self.grad_sq["rel_emb"].zero_()
        if bg.B <= 4096:      # head-entity scatter, with the relation scatter as its second job: one launch
            rel_job = (ptr(b.rel), B, ptr(b.dr), dr, ptr(g["rel_emb"]), ptr(self.grad_sq["rel_emb"]), 0, self.num_rel) \
                if rel else (None, 0, None, 0, None, None, 0, 0)
            call("coper_segscatter_add_pair", ptr(bg.e1), bg.B, ptr(bg.dx0), d, ptr(g["ent_emb"]), ptr(gsq_e), s.lo, s.hi,
                 ptr(self.norm_delta) if self._norm_fused_now else None, *rel_job)
            if self._norm_fused_now:
                self._norm_delta_n = bg.B
        else:
            call("coper_segscatter_add", ptr(bg.e1), bg.B, ptr(bg.dx0), d, ptr(g["ent_emb"]), s.lo, s.hi, ptr(bg.ws),
                 bg.ws_bytes)
            if gsq_e is not None:
                torch.mul(bg.dx0, bg.dx0, out=bg.dx0_sq)
                call("coper_segscatter_add", ptr(bg.e1), bg.B, ptr(bg.dx0_sq), d, ptr(gsq_e), s.lo, s.hi, ptr(bg.ws),
                     bg.ws_bytes)
            if rel and small:
                call("coper_segscatter_add_sq", ptr(b.rel), B, ptr(b.dr), dr, ptr(g["rel_emb"]),
                     ptr(self.grad_sq["rel_emb"]), 0, self.num_rel)
            elif rel:
                call("coper_segscatter_add", ptr(b.rel), B, ptr(b.dr), dr, ptr(g["rel_emb"]), 0, self.num_rel, ptr(b.ws),
                     b.ws_bytes)
                torch.mul(b.dr, b.dr, out=b.dr_sq)
                call("coper_segscatter_add", ptr(b.rel), B, ptr(b.dr_sq), dr, ptr(self.grad_sq["rel_emb"]), 0,
                     self.num_rel, ptr(b.ws), b.ws_bytes)
        if dp:      # partial sums over this rank's rows -> all-reduce of the flat bucket
            if big_work is not None:
                sharding.reduce_replicated_grads(self.flat_small, self.world, self.group)
                big_work.wait()
            else:
                sharding.reduce_replicated_grads(self.flat_grads, self.world, self.group)
        if apply:
            self._clip_and_apply()

    def _sampled_scorer(self, b):
        """models.py:438-443 + 448-453 on the staged [B, L] lookup ids / labels (b.cur_samp).  Entity-sharded: every
        rank scores all B x L positions whose id it owns; loss_sum and dq are its partials (summed by the caller)."""
        sb, g, gsq, s = b.cur_samp, self.grads, self.grad_sq, self.shard
        for t in (g["ent_emb"], gsq["ent_emb"], g["pred_bias"], gsq["pred_bias"]):
            t.zero_()
        if b.cur_sampling is not None:       # labels drawn on the device from the staged CSR positives (data.py:228-277)
            L, prop_negatives = b.cur_sampling
            # every rank draws the same [B, L], the single-GPU draw of this seed and step: the data-parallel seed word
            # carries rank << 32 (per-rank dropout masks), which the salt takes off again (the kernel keys on seed + salt)
            salt = (SALT_SAMPLE - ((s.rank << 32) if self.dp else 0)) % (1 << 64)
            call("coper_sample_labels", ptr(b.rowptr), ptr(b.col), b.B, self.num_ent, L,
                 int(1.0 / (1.0 + prop_negatives) * L), ptr(self.seed_dev), salt, ptr(sb.lookup), ptr(sb.labels))
        args = (ptr(b.q), ptr(self.ent_emb), ptr(self.pred_bias), ptr(sb.lookup), ptr(sb.labels), b.B, sb.L,
                self.num_ent, self.ent_emb_size, 1.0 - self.label_smoothing_epsilon, 1.0 / self.num_ent,
                1.0 / (float(b.B) * float(sb.L)), ptr(b.loss_sum), ptr(sb.scores), ptr(sb.g), ptr(b.dq),
                ptr(g["ent_emb"]), ptr(gsq["ent_emb"]), ptr(g["pred_bias"]), ptr(gsq["pred_bias"]))
        if self.world > 1:
            call("coper_score_sampled_bce_fwd_bwd_sharded", *args, s.lo, s.hi, ptr(sb.ws), sb.ws.numel())
        else:
            call("coper_score_sampled_bce_fwd_bwd", *args, ptr(sb.ws), sb.ws.numel())

    def _clip_and_apply(self):
        """tf.clip_by_global_norm(5.0) (models.py:199) + AMSGrad apply (amsgrad.py:130-159): one multi-tensor
        launch per phase over the whole variable list."""
        nt = len(self.trainables)
        fused = self._norm_fused_now
        if fused and self.mt_nchunks_ext > 0:
            descs, chunks, nchunks, offsets = self.mt_desc_ext, self.mt_chunks_ext, self.mt_nchunks_ext, self.mt_offsets_ext
        else:
            descs, chunks, nchunks, offsets = (self.mt_desc_ext if fused else self.mt_desc, self.mt_chunks,
                                               self.mt_nchunks, self.mt_offsets)
        # per-tensor squared norms; fused: |dE|^2 (tensor 0) = the dE GEMM epilogue's sum + the change the head-entity
        # scatter made to it; single GPU: the clip factor comes out of the same finishing launch
        one = self.world == 1
        call("coper_mt_sumsq_clip", ptr(descs), nt, ptr(chunks), nchunks, ptr(offsets), ptr(self.mt_partials),
             ptr(self.sumsq), 0 if fused else -1, ptr(self.dE_sumsq) if fused else None, 1 if fused else 0,
             ptr(self.norm_delta) if fused else None, self._norm_delta_n if fused else 0, CLIP_NORM,
             ptr(self.clip_out) if one else None)
        if not one:
            # trainables 0,1 (ent_emb, pred_bias) are row-sharded: their squared norms add across ranks;
            # every other gradient is replicated (identical on all ranks) and is counted once.
            sharding.reduce_sharded_sumsq(self.sumsq[:2], self.world, self.group)
            call("coper_clip_scale_n", ptr(self.sumsq), nt, CLIP_NORM, ptr(self.clip_out))
        call("coper_mt_amsgrad", ptr(self.mt_desc), ptr(self.mt_chunks), self.mt_nchunks, ptr(self.step_state),
             self.beta1, self.beta2, self.adam_eps, ptr(self.clip_out), int(self.bug_compat))
        if not self._emit_prepared:
            self.refresh_prepared()

    # ------------------------------------------------------------------------------------------
    def _launch_mode(self):
        """Process-wide launch switches of the library, set before this model enqueues kernels (a replayed graph keeps
        what it was captured with)."""
        call_plain("coper_set_pdl", int(self._pdl))

    def _run_graphed(self, key, fn):
        """First call: eager (allocates buffers, sets kernel attributes).  Second call: capture, then replay."""
        if not self.use_graphs or (self.world > 1 and not self.graphs_multi_gpu):
            self._launch_mode()
            fn()
            return
        st = self._graphs.get(key)
        if st is None:
            self._launch_mode()
            fn()
            self._graphs[key] = "warm"
            return
        if st == "warm":
            self._launch_mode()
            g = torch.cuda.CUDAGraph()
            torch.cuda.synchronize()
            lib = _lib.load()
            k0 = lib.coper_launch_count()
            # thread_local capture mode: other threads (e.g. the NCCL watchdog polling events) must not invalidate
            # or block the capture when the step contains collectives
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                fn()
            self._graphs[key] = st = (g, lib.coper_launch_count() - k0)
        st[0].replay()
        self.graph_kernel_launches += st[1]      # kernels of this library executed by the replay

    def train_step(self, batch: Dict, apply_update: bool = True):
        """One reference training step (run_cpg.py:210-219).  Returns the loss as a 0-d device tensor
        (float64 -> call .item() to read it; that is the step's only device->host transfer).  The tensor is a view
        of the step's own buffer, written inside the captured step: valid until the next step of the same batch size."""
        if self.use_negative_sampling:
            return self._train_step_sampled(batch, apply_update)
        b = self.stage_batch(batch)
        self._run_train(("train", b.B), b, apply_update)
        return b.loss_mean[0]

    def _run_train(self, key, b, apply: bool):
        """The device step on staged buffers b: graphed when it applies the update, eager when it only computes the
        gradients (the caller applies them later with _clip_and_apply)."""
        if apply:
            self._run_graphed(key, lambda: self._train_device(b))
        else:
            self._launch_mode()
            self._train_device(b, apply=False)
        self.global_step += 1

    def _train_step_sampled(self, batch: Dict, apply_update: bool):
        """Sampled-label step: ``batch['lookup_values']`` int32 [B, L] entity ids and ``batch['e2_multi']`` fp32 [B, L]
        their labels (data.py:228-312 produce them; models.py:165,438-443 consume them)."""
        sampling = batch.get("sample_on_device")
        if sampling is not None:
            # (num_labels, prop_negatives): the batch carries the CSR id lists of the known-true tails instead of
            # pre-sampled [B, L] ids / labels; coper_sample_labels draws them inside the (graph-captured) device step
            L = int(sampling[0])
            if not 0 < L <= self.num_ent or "e2_multi_rowptr" not in batch:
                raise ValueError("sample_on_device=(num_labels, prop_negatives) needs e2_multi_rowptr / e2_multi_col "
                                 "and 0 < num_labels <= num_ent")
            b = self.stage_batch({k: batch[k] for k in ("e1", "rel", "e2", "e2_multi_rowptr", "e2_multi_col")
                                  if k in batch})
            sb = _slot(b.samp, L, _SampledSlot, self, b.B, L)
            b.cur_sampling = (L, float(sampling[1]))
        else:
            lookup, labels = batch["lookup_values"], batch["e2_multi"]
            if lookup is None or len(lookup.shape) != 2 or lookup.shape[1] == 0 \
                    or tuple(labels.shape) != tuple(lookup.shape):
                raise ValueError("sampled-label training needs lookup_values [B, L] and e2_multi [B, L] "
                                 "(L = num_labels)")
            b = self.stage_batch({k: batch[k] for k in ("e1", "rel", "e2") if k in batch})
            L = int(lookup.shape[1])
            sb = _slot(b.samp, L, _SampledSlot, self, b.B, L)
            b.cur_sampling = None
            for src, dev_t, host_t, dt in ((lookup, sb.lookup, sb.h_lookup, torch.int32),
                                          (labels, sb.labels, sb.h_labels, torch.float32)):
                if isinstance(src, torch.Tensor) and src.is_cuda:
                    dev_t.copy_(src)
                else:
                    host_t.copy_(torch.as_tensor(np.asarray(src), dtype=dt))
                    dev_t.copy_(host_t, non_blocking=True)
        b.h2d_event.record()
        b.cur_samp = sb
        self._run_train(("train_sampled", b.B, L, b.cur_sampling, b.csr_gen if b.cur_sampling else 0), b, apply_update)
        return b.loss_sum[0] / (float(b.B) * float(sb.L))

    def predict_all(self, batch: Dict):
        """Logits of every query against this rank's entity rows: [B, rows] view (metrics.py:40-42)."""
        b = self.stage_batch(batch)
        self._launch_mode()
        self._eval_q(b)
        self._score(b)
        return b.S[:, :self.shard.rows]

    def predict_topk(self, batch: Dict, k: int = 10, filtered: bool = True):
        """The k most likely tail entities of each query (e1, rel, ?): (scores fp32 [B, k], ids int64 [B, k]).
        Scores are the logits ``predict_all`` computes; entities are sorted by score descending, then by id ascending.
        ``filtered=True`` excludes the known true tails ``batch['e2_multi*']`` (the standard filtered prediction;
        ``e2`` is not needed and not excluded).  A query with fewer than k eligible entities is padded with
        (-inf, -1).  Under entity sharding every rank returns the same global result.  Both tensors are buffers of the
        (batch size, k) slot, overwritten by the next call with the same batch size and k (clone them to keep them).
        Speed (DESIGN §6d): well ahead of ``predict_all`` + ``torch.topk`` at 1 M+ entities and small k; at WN18RR's
        40 k entities with k >= 10, and at k = 100 below 10 M entities, that route is faster."""
        k = int(k)
        if not 1 <= k <= _lib.TOPK_MAX:
            raise ValueError("k must be in [1, %d], got %d" % (_lib.TOPK_MAX, k))
        keys = ("e1", "rel")
        if filtered:
            if not has_known_tails(batch):
                raise ValueError("filtered top-k needs the known true tails: e2_multi, or e2_multi_rowptr / e2_multi_col")
            keys += ("e2_multi_rowptr", "e2_multi_col", "e2_multi")
        b = self.stage_batch({key: batch[key] for key in keys if key in batch})
        t = _slot(b.topk, k, _TopkSlot, self, b.B, k)
        self._run_graphed(("topk", b.B, k, bool(filtered)), lambda: self._topk_device(b, t, filtered))
        return t.scores, t.ids

    def _topk_device(self, b, t, filtered):
        self._eval_q(b)
        s, d, k = self.shard, self.ent_emb_size, t.scores.shape[1]
        out_s, out_i = (t.local_scores, t.local_ids) if self.world > 1 else (t.scores, t.ids)
        if self.E_prep is not None:
            # tensor-pipe engines: top-k straight from the scorer's accumulators, logits never written
            call("coper_prepare_operand", ptr(b.q), b.B, d, d, self.prec, ptr(b.q_prep))
            call("coper_score1n_topk_prepared", ptr(b.q_prep), ptr(self.E_prep), ptr(self.pred_bias), b.B, s.rows, d,
                 ptr(b.bitsT) if filtered else None, s.lo, k, ptr(out_s), ptr(out_i), ptr(t.ws), t.ws_bytes, self.prec)
        else:
            self._score(b)
            call("coper_topk_scores", ptr(b.S), b.ld, b.B, s.rows, ptr(b.bits) if filtered else None, s.lo, k,
                 ptr(out_s), ptr(out_i), ptr(t.ws), t.ws_bytes)
        if self.world > 1:
            all_s, all_i = sharding.gather_topk(out_s, out_i, self.world, self.group, out=(t.all_scores, t.all_ids))
            call("coper_topk_merge", ptr(all_s), ptr(all_i), all_s.shape[0], b.B, k, ptr(t.scores), ptr(t.ids))

    def _score(self, b):
        d = self.ent_emb_size
        if self.E_prep is not None:
            call("coper_prepare_operand", ptr(b.q), b.B, d, d, self.prec, ptr(b.q_prep))
            call("coper_score1n_fwd_prepared", ptr(b.q_prep), ptr(self.E_prep), ptr(self.pred_bias), b.B,
                 self.shard.rows, d, ptr(self._scores_buf(b)), b.ld, self.prec)
        else:
            call("coper_score1n_fwd", ptr(b.q), ptr(self.ent_emb), ptr(self.pred_bias), b.B, self.shard.rows, d,
                 ptr(self._scores_buf(b)), b.ld, ptr(b.ws), b.ws_bytes, self.prec)

    def filtered_ranks(self, batch: Dict):
        """Filtered rank of ``e2`` for each query (metrics.py:44-51) computed on device.
        ``batch['e2_multi*']`` is the filter set (all known true tails).  Returns int32 device tensors
        (rank, n_equal); rank == the reference's rank whenever n_equal == 0.  Both are buffers of the batch-size slot,
        overwritten by the next call with the same batch size (clone them to keep them, as metrics.py does)."""
        self._check_e2(batch["e2"])
        b = self.stage_batch(batch, need_e2=True)
        if self.prec != 0:          # the gold entity joins the filter set (metrics.py:44-46 never compares it)
            call("coper_bits_t_set", ptr(b.e2), b.B, self.shard.lo, self.shard.hi, ptr(b.bitsT))
        self._run_graphed(("rank", b.B), lambda: self._rank_device(b))
        return b.rank, b.n_equal

    def _check_e2(self, e2):
        """Host gold tails must be entity ids (device ones are taken as they are)."""
        if not (isinstance(e2, torch.Tensor) and e2.is_cuda):
            e2 = np.asarray(e2)
            if int(e2.min()) < 0 or int(e2.max()) >= self.num_ent:
                raise ValueError("e2 out of range (train rows carry e2 = -1 in the reference; SURVEY Q17)")

    def _rank_device(self, b):
        self._eval_q(b)
        s = self.shard
        d = self.ent_emb_size
        b.rank_counts.zero_()
        if self.E_prep is not None:
            # tensor-pipe engines: rank counts straight from the scorer's accumulators, logits never written
            call("coper_prepare_operand", ptr(b.q), b.B, d, d, self.prec, ptr(b.q_prep))
            call("coper_score1n_gold_prepared", ptr(b.q_prep), ptr(self.E_prep), ptr(self.pred_bias), b.B, s.rows, d,
                 ptr(b.e2), s.lo, ptr(b.gold), ptr(b.ws), b.ws_bytes, self.prec)
            sharding.reduce_gold(b.gold, self.world, self.group)
            call("coper_score1n_rank_prepared", ptr(b.q_prep), ptr(self.E_prep), ptr(self.pred_bias), b.B, s.rows, d,
                 ptr(b.gold), ptr(b.bitsT), ptr(b.n_greater), ptr(b.n_equal), self.prec)
        else:
            self._score(b)
            call("coper_gold_scores", ptr(b.S), b.ld, b.B, s.rows, ptr(b.e2), s.lo, ptr(b.gold))
            sharding.reduce_gold(b.gold, self.world, self.group)
            call("coper_filtered_rank", ptr(b.S), b.ld, b.B, s.rows, ptr(b.e2), s.lo, ptr(b.gold), ptr(b.bits),
                 ptr(b.n_greater), ptr(b.n_equal))
        sharding.reduce_counts(b.n_greater, b.n_equal, self.world, self.group)
        torch.add(b.n_greater, 1, out=b.rank)        # inside the captured step: the caller reads b.rank
        return b.rank, b.n_equal

    # ------------------------------------------------------------------------------------------ given candidates
    def score_candidates(self, batch: Dict, candidates):
        """Logits of given tails: ``candidates`` int [B, C] of global entity ids (host or device), -1 = padding.
        Returns fp32 [B, C] with s[b, j] = q[b].E[candidates[b, j]] + bias[candidates[b, j]] and -inf at padding;
        ``batch`` needs ``e1`` and ``rel`` only.  Host candidates outside [-1, num_ent) raise ValueError; on the device
        an id >= num_ent scores 0.  The scores are exact fp32 dot products with the master entity table for every
        ``prec`` - the logits the sampled-label training step computes, bit for bit - so they match ``predict_all``
        only to the engine's score tolerance (bf16: 1e-2).  Under entity sharding every rank returns the single-GPU
        result (a logit of -0 comes back as +0).  The tensor is a buffer of the (B, C) slot, overwritten by the next
        call with the same B and C (clone it to keep it)."""
        b, c = self._stage_candidates({k: batch[k] for k in ("e1", "rel")}, candidates, with_e2=False)
        self._run_graphed(("cand_score", b.B, c.C), lambda: self._cand_score_device(b, c))
        return c.scores

    def candidate_ranks(self, batch: Dict, candidates, filtered: bool = True):
        """Rank of the gold tail ``batch['e2']`` among given candidates (int [B, C] global ids, -1 = padding), as
        ``filtered_ranks`` ranks it among all entities: rank = 1 + #{j : candidates[b, j] != e2[b], not a known true
        tail, s[b, j] > s[b, e2[b]]}; n_equal counts the ties the same way.  A candidate listed twice counts twice.
        ``filtered=True`` excludes the known true tails ``batch['e2_multi*']`` (ValueError without them);
        ``filtered=False`` excludes only the gold entity itself.  Scores as in ``score_candidates``.  Returns int32
        device tensors (rank, n_equal) [B], buffers of the (B, C) slot, overwritten by the next call with the same B
        and C (clone them to keep them)."""
        self._check_e2(batch["e2"])
        keys = ("e1", "rel", "e2")
        if filtered:
            if not has_known_tails(batch):
                raise ValueError("filtered candidate ranks need the known true tails: e2_multi, or e2_multi_rowptr / "
                                 "e2_multi_col")
            keys += ("e2_multi_rowptr", "e2_multi_col", "e2_multi")
        b, c = self._stage_candidates({k: batch[k] for k in keys if k in batch}, candidates, with_e2=True)
        self._run_graphed(("cand_rank", b.B, c.C, bool(filtered)), lambda: self._cand_rank_device(b, c, filtered))
        return c.rank, c.n_equal

    def _stage_candidates(self, batch, candidates, with_e2):
        on_device = isinstance(candidates, torch.Tensor) and candidates.is_cuda
        if not on_device:
            candidates = np.asarray(candidates)
        if len(candidates.shape) != 2 or candidates.shape[1] < 1 or candidates.shape[0] != len(batch["e1"]):
            raise ValueError("candidates must be [B, C] with C >= 1 and B = len(e1), got %s" % (tuple(candidates.shape),))
        if not on_device and (int(candidates.min()) < -1 or int(candidates.max()) >= self.num_ent):
            raise ValueError("candidate ids must lie in [0, %d) or be -1 (padding)" % self.num_ent)
        b = self.stage_batch(batch)             # e1, rel and the filter bits; e2 travels in the candidate block
        B, C = b.B, int(candidates.shape[1])
        c = _slot(b.cand, C, _CandSlot, self, B, C)
        # each region of the block comes from where its ids live; two host regions travel in one copy
        e2 = batch["e2"] if with_e2 else None
        e2_on_device = isinstance(e2, torch.Tensor) and e2.is_cuda
        if on_device:
            c.cand.copy_(candidates)
        else:
            c.h_np[:B * C] = candidates.reshape(-1)
        if e2 is not None and e2_on_device:
            c.e2.copy_(e2)
        elif e2 is not None:
            c.h_np[B * C:] = np.asarray(e2).reshape(-1)
        host_e2 = e2 is not None and not e2_on_device
        if not on_device and host_e2:
            c.d_ids.copy_(c.h_ids, non_blocking=True)
        elif not on_device:
            c.cand.copy_(c.h_ids[:B * C].view(B, C), non_blocking=True)
        elif host_e2:
            c.e2.copy_(c.h_ids[B * C:], non_blocking=True)
        b.h2d_event.record()               # the next stage_batch waits for this copy before reusing pinned memory
        return b, c

    def _cand_score_device(self, b, c):
        s = self.shard
        self._eval_q(b)
        call("coper_score_candidates", ptr(b.q), ptr(self.ent_emb), ptr(self.pred_bias), ptr(c.cand), b.B, c.C,
             self.ent_emb_size, s.lo, s.hi, ptr(c.scores))
        sharding.exchange_rows(c.scores, self.world, self.group)     # non-owned positions hold exact zeros
        c.scores.masked_fill_(c.cand < 0, float("-inf"))

    def _cand_rank_device(self, b, c, filtered):
        s, d = self.shard, self.ent_emb_size
        self._eval_q(b)
        c.counts.zero_()
        # the gold logit by the same kernel and arithmetic as the candidates it is compared with
        call("coper_score_candidates", ptr(b.q), ptr(self.ent_emb), ptr(self.pred_bias), ptr(c.e2), b.B, 1, d, s.lo,
             s.hi, ptr(c.gold))
        sharding.reduce_gold(c.gold, self.world, self.group)
        bits = (b.bits if self.prec == 0 else b.bitsT) if filtered else None
        call("coper_candidate_rank", ptr(b.q), ptr(self.ent_emb), ptr(self.pred_bias), ptr(c.cand), ptr(c.e2), b.B,
             c.C, d, s.lo, s.hi, ptr(c.gold), ptr(bits), int(self.prec != 0), ptr(c.n_greater), ptr(c.n_equal))
        sharding.reduce_counts(c.n_greater, c.n_equal, self.world, self.group)
        torch.add(c.n_greater, 1, out=c.rank)
