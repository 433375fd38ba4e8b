"""Top-k link prediction on the host: workspace queries, the sharded exchange step (gloo, world 2 and 3) followed by a
NumPy merge under the (score descending, id ascending) order, and the run_cpg argument checks."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from test_sharding_gloo import _free_port


def test_topk_workspace_queries_run_without_gpu():
    from coper_b200 import _lib
    lib = _lib.load()
    for prec in (1, 2, 3):
        assert lib.coper_score1n_topk_workspace_bytes(512, 40943, 200, 10, prec) > 0
        assert lib.coper_score1n_topk_workspace_bytes(512, 40943, 200, 0, prec) == 0
        assert lib.coper_score1n_topk_workspace_bytes(512, 40943, 200, 129, prec) == 0
    assert lib.coper_score1n_topk_workspace_bytes(512, 40943, 200, 10, 0) == 0      # fp32: coper_topk_scores
    assert lib.coper_topk_scores_workspace_bytes(512, 40943, 128) >= 512 * 128 * 8
    assert lib.coper_topk_scores_workspace_bytes(512, 40943, 129) == 0


def np_topk(scores, ids, k):
    """Top k of each row under (score desc, id asc); padding (-inf, -1) entries never win."""
    B = scores.shape[0]
    out_s = np.full((B, k), -np.inf, np.float32)
    out_i = np.full((B, k), -1, np.int64)
    for b in range(B):
        ok = ids[b] >= 0
        s, i = scores[b][ok], ids[b][ok]
        o = np.lexsort((i, -s))[:k]
        out_s[b, :len(o)], out_i[b, :len(o)] = s[o], i[o]
    return out_s, out_i


def _shard_lists(rank, world, B, N, k, seed):
    """Global scores with planted ties; each rank owns a contiguous id range and returns its local top-k."""
    rng = np.random.default_rng(seed)
    S = rng.integers(-20, 20, (B, N)).astype(np.float32) * 0.25          # many exact ties across shards
    per = -(-N // world)
    lo, hi = rank * per, min(N, (rank + 1) * per)
    ids = np.broadcast_to(np.arange(lo, hi), (B, hi - lo))
    ls, li = np_topk(S[:, lo:hi], ids, k)
    return S, ls, li


def _worker(rank, world, port, out_dir):
    from coper_b200 import sharding
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        B, N, k = 9, 301, 12
        S, ls, li = _shard_lists(rank, world, B, N, k, seed=7)
        all_s, all_i = sharding.gather_topk(torch.from_numpy(ls), torch.from_numpy(li), world)
        assert tuple(all_s.shape) == (world, B, k) and all_i.dtype == torch.int64
        out = (torch.empty(world, B, k), torch.empty(world, B, k, dtype=torch.int64))
        all_s2, all_i2 = sharding.gather_topk(torch.from_numpy(ls), torch.from_numpy(li), world, out=out)
        assert torch.equal(all_s, all_s2) and torch.equal(all_i, all_i2)
        cat_s = all_s.permute(1, 0, 2).reshape(B, -1).numpy()
        cat_i = all_i.permute(1, 0, 2).reshape(B, -1).numpy()
        ms, mi = np_topk(cat_s, cat_i, k)
        rs, ri = np_topk(S, np.broadcast_to(np.arange(N), (B, N)), k)
        np.savez(os.path.join(out_dir, "r%d.npz" % rank), ms=ms, mi=mi, rs=rs, ri=ri)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_gather_topk_then_merge_equals_global_topk(world, tmp_path):
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        o = np.load(os.path.join(str(tmp_path), "r%d.npz" % r))
        assert np.array_equal(o["mi"], o["ri"]) and np.array_equal(o["ms"], o["rs"])


def test_gather_topk_without_group_is_the_local_list():
    from coper_b200 import sharding
    s, i = torch.randn(3, 4), torch.arange(12).reshape(3, 4)
    a, b = sharding.gather_topk(s, i, 1)
    assert tuple(a.shape) == (1, 3, 4) and torch.equal(a[0], s) and torch.equal(b[0], i)


@pytest.mark.parametrize("argv", [
    ["--synthetic", "toy", "--predict-topk", "5"],                                   # no checkpoint to predict from
    ["--synthetic", "toy", "--model-load-path", "x.ckpt", "--predict-topk", "0"],
    ["--synthetic", "toy", "--model-load-path", "x.ckpt", "--predict-topk", "129"],
])
def test_run_cpg_rejects_bad_predict_topk(argv):
    from coper_b200 import run_cpg
    with pytest.raises(SystemExit) as e:
        run_cpg.main(argv)
    assert e.value.code == 2
