"""Host-side pieces kept from the reference (no GPU): dataset loaders (qa_cpg/data.py), config flag system
(qa_cpg/configs/*.yaml + run_cpg.py:49-60), entry-point plumbing."""
import os

import numpy as np
import pytest

from coper_b200 import configs, data

TRAIN = [("a", "likes", "b"), ("a", "likes", "c"), ("b", "likes", "c"), ("c", "knows", "a"), ("d", "knows", "a")]
DEV = [("a", "knows", "d"), ("b", "likes", "a")]
TEST = [("d", "likes", "b")]


def _write(tmp_path, name="train"):
    for fn, rows in (("train.txt", TRAIN), ("dev.txt", DEV), ("test.txt", TEST)):
        with open(os.path.join(tmp_path, fn), "w") as fh:
            for r in rows:
                fh.write("\t".join(r) + "\n")


def _loader():
    return data.CountriesS1Loader()          # a _MinervaDataLoader: plain train/dev/test.txt, no archive


def test_loader_classes_and_urls_match_reference_names():
    for name in ("NationsLoader", "UMLSLoader", "KinshipLoader", "WN18RRLoader", "YAGO310Loader", "FB15k237Loader",
                 "CountriesS1Loader", "CountriesS2Loader", "CountriesS3Loader", "WN18Loader", "FB15kLoader",
                 "NELL995Loader"):
        assert hasattr(data, name)
    assert data.WN18RRLoader().dataset_name == "WN18RR" and data.WN18RRLoader().filenames == ["WN18RR.tar.gz"]
    assert data.NELL995Loader(is_test=True).dataset_name == "nell-995-test"
    assert data.FB15kLoader(is_test=True).dataset_name == "FB15ktest"
    assert data.YAGO310Loader().filetypes == ["train", "valid", "test"]
    assert data.YAGO310Loader().add_reverse_per_filetype == [True, False, False]


def test_missing_files_fail_loudly_without_network(tmp_path):
    with pytest.raises(FileNotFoundError) as exc:
        data.WN18RRLoader().maybe_create_tf_record_files(str(tmp_path))
    assert "TimDettmers/ConvE" in str(exc.value)


def test_graph_semantics(tmp_path):
    _write(str(tmp_path))
    ld = _loader()
    ld.maybe_create_tf_record_files(str(tmp_path))
    ents = [l.strip() for l in open(os.path.join(tmp_path, "entities.txt"))]
    rels = [l.strip() for l in open(os.path.join(tmp_path, "relations.txt"))]
    assert ents == ["a", "b", "c", "d"] and ld.num_ent == 4
    assert rels == ["knows", "knows_reverse", "likes", "likes_reverse"] and ld.num_rel == 4     # reverse relations count
    eid, rid = {e: i for i, e in enumerate(ents)}, {r: i for i, r in enumerate(rels)}
    # training samples: one per (e1, rel) key incl. reverse keys, labels = that split's own tails (data.py:482-488)
    it = ld.train_dataset(str(tmp_path), batch_size=100, num_labels=None)
    b = next(it)
    got = {}
    for i in range(len(b["e1"])):
        got[(int(b["e1"][i]), int(b["rel"][i]))] = set(b["e2_multi_col"][b["e2_multi_rowptr"][i]:b["e2_multi_rowptr"][i + 1]])
    assert got[(eid["a"], rid["likes"])] == {eid["b"], eid["c"]}
    assert got[(eid["c"], rid["likes_reverse"])] == {eid["a"], eid["b"]}
    assert got[(eid["a"], rid["knows_reverse"])] == {eid["c"], eid["d"]}
    assert (b["e2"] == -1).all()                                       # train rows carry e2 = -1 (data.py:335,485)
    assert len(got) == 7
    # without inverse relations only the 4 forward keys remain
    b2 = next(ld.train_dataset(str(tmp_path), batch_size=100, include_inv_relations=False, num_labels=None))
    assert len(b2["e1"]) == 4 and all(int(r) in (rid["knows"], rid["likes"]) for r in b2["rel"])
    # eval: one sample per triple; filter = full graph (train + dev + test, both directions); tail-only
    dev = list(ld.eval_dataset(str(tmp_path), "dev", batch_size=10, include_inv_relations=False))
    assert len(dev) == 1 and len(dev[0]["e1"]) == 2
    rows = {(int(e1), int(r), int(e2)): set(dev[0]["e2_multi_col"][dev[0]["e2_multi_rowptr"][i]:dev[0]["e2_multi_rowptr"][i + 1]])
            for i, (e1, r, e2) in enumerate(zip(dev[0]["e1"], dev[0]["rel"], dev[0]["e2"]))}
    assert rows[(eid["b"], rid["likes"], eid["a"])] == {eid["c"], eid["a"]}           # train tail c + dev tail a
    assert rows[(eid["a"], rid["knows"], eid["d"])] == {eid["d"]}
    test = list(ld.eval_dataset(str(tmp_path), "test", batch_size=10, include_inv_relations=False))
    assert len(test[0]["e1"]) == 1 and int(test[0]["e2"][0]) == eid["b"]
    # the dense schema of the reference is the same labels
    d = list(ld.eval_dataset(str(tmp_path), "dev", batch_size=10, include_inv_relations=False, dense=True))[0]
    assert d["e2_multi"].shape == (2, 4) and d["e2_multi"].sum() == 3
    # second loader instance reuses the cache and the id files
    ld2 = _loader()
    ld2.maybe_create_tf_record_files(str(tmp_path))
    assert (ld2.num_ent, ld2.num_rel) == (4, 4)


def test_existing_id_files_are_honoured(tmp_path):
    _write(str(tmp_path))
    with open(os.path.join(tmp_path, "entities.txt"), "w") as fh:
        fh.write("d\nc\nb\na\n")
    ld = _loader()
    ld.maybe_create_tf_record_files(str(tmp_path))
    t = list(ld.eval_dataset(str(tmp_path), "test", batch_size=10, include_inv_relations=False))[0]
    assert int(t["e1"][0]) == 0 and int(t["e2"][0]) == 2                # d -> 0, b -> 2


def test_test_set_cleaning(tmp_path):
    rows_test = TEST + [("zzz", "likes", "b"), ("a", "unseen_rel", "b")]
    _write(str(tmp_path))
    with open(os.path.join(tmp_path, "test.txt"), "w") as fh:
        for r in rows_test:
            fh.write("\t".join(r) + "\n")
    ld = data.NELL995Loader(needs_test_set_cleaning=True)
    ld.maybe_create_tf_record_files(str(tmp_path))
    t = list(ld.eval_dataset(str(tmp_path), "test", batch_size=10, include_inv_relations=False))[0]
    assert len(t["e1"]) == 1                                            # unseen entity / relation questions dropped


def _big_graph(tmp_path, n_ent=60, n_trip=400, seed=0):
    rng = np.random.default_rng(seed)
    rows = {("e%d" % rng.integers(n_ent), "r%d" % rng.integers(3), "e%d" % rng.integers(n_ent)) for _ in range(n_trip)}
    rows = sorted(rows)
    for fn, part in (("train.txt", rows[:-20]), ("dev.txt", rows[-20:-10]), ("test.txt", rows[-10:])):
        with open(os.path.join(tmp_path, fn), "w") as fh:
            for r in part:
                fh.write("\t".join(r) + "\n")


@pytest.mark.parametrize("one_pos", [False, True])
def test_sampled_label_pipelines(tmp_path, one_pos):
    """data.py:228-312: [B, L] lookup ids + labels; negatives are distinct entities, labels are 1 exactly where the
    looked-up id is a positive of the query, positives come first."""
    _big_graph(str(tmp_path))
    ld = _loader()
    L, B = 16, 8
    it = ld.train_dataset(str(tmp_path), batch_size=B, num_labels=L, prop_negatives=3.0,
                          one_positive_label_per_sample=one_pos, prefetch_buffer_size=2)
    c = ld.load_and_preprocess(str(tmp_path))
    key = {(int(a), int(b)): i for i, (a, b) in enumerate(zip(c["train_e1"], c["train_rel"]))}
    for _ in range(5):
        b = next(it)
        assert b["lookup_values"].shape == (B, L) and b["lookup_values"].dtype == np.int32
        assert b["e2_multi"].shape == (B, L) and b["e2_multi"].dtype == np.float32 and (b["e2"] == -1).all()
        for i in range(B):
            r = key[(int(b["e1"][i]), int(b["rel"][i]))]
            pos = set(c["train_col"][c["train_rowptr"][r]:c["train_rowptr"][r + 1]].tolist())
            lk, lab = b["lookup_values"][i], b["e2_multi"][i]
            assert np.array_equal(lab, np.isin(lk, list(pos)).astype(np.float32))
            if one_pos:
                assert int(lk[0]) in pos and len(set(lk[1:].tolist())) == L - 1          # 1 positive + distinct negatives
            else:
                n_needed = int(1.0 / (1.0 + 3.0) * L)
                n_pos = len(pos) if len(pos) <= n_needed else L - min(ld.num_ent, L - n_needed)
                assert set(lk[:n_pos].tolist()) <= pos and len(set(lk[n_pos:].tolist())) == L - n_pos
    with pytest.raises(ValueError):
        ld.train_dataset(str(tmp_path), batch_size=4, num_labels=10 ** 6)


def test_device_sampling_pipeline_and_restatement(tmp_path):
    """device_sampling=True: the loader hands out the CSR id lists + (num_labels, prop_negatives); the sampler the GPU
    kernel implements (NumPy restatement, oracle/dropout_hash.sample_labels) builds rows with the reference's shape:
    positives first, distinct sampled entities, labels == membership (data.py:228-277)."""
    from oracle import dropout_hash as DH
    _big_graph(str(tmp_path))
    ld = _loader()
    L, B, prop = 16, 8, 3.0
    it = ld.train_dataset(str(tmp_path), batch_size=B, num_labels=L, prop_negatives=prop,
                          one_positive_label_per_sample=False, device_sampling=True)
    b = next(it)
    assert b["sample_on_device"] == (L, prop) and b["lookup_values"].shape == (B, 0)
    rowptr, col = b["e2_multi_rowptr"], b["e2_multi_col"]
    n_needed = int(1.0 / (1.0 + prop) * L)
    lk, lab = DH.sample_labels(rowptr, col, ld.num_ent, L, n_needed, seed_dev=12345)
    for i in range(B):
        pos = set(col[rowptr[i]:rowptr[i + 1]].tolist())
        n_pos = len(pos) if len(pos) <= n_needed else L - min(ld.num_ent, L - n_needed)
        assert set(lk[i, :n_pos].tolist()) <= pos and len(set(lk[i, n_pos:].tolist())) == L - n_pos
        assert np.array_equal(lab[i], np.isin(lk[i], list(pos)).astype(np.float32))
    lk2, _ = DH.sample_labels(rowptr, col, ld.num_ent, L, n_needed, seed_dev=12346)
    assert not np.array_equal(lk, lk2)
    # one_positive_label_per_sample keeps the host sampler (a different row expansion, data.py:279-312)
    b1 = next(ld.train_dataset(str(tmp_path), batch_size=B, num_labels=L, prop_negatives=prop,
                               one_positive_label_per_sample=True, device_sampling=True, prefetch_buffer_size=2))
    assert b1["lookup_values"].shape == (B, L) and "sample_on_device" not in b1


def test_shipped_configs():
    cfg = configs.load_config("WN18RR", "cpg")
    assert cfg.model.entity_embedding_size == 200 and cfg.model.relation_embedding_size == 8
    assert cfg.context.context_rel_out == [] and cfg.context.context_rel_conv is None
    assert cfg.training.batch_size == 512 and cfg.training.num_labels == 100 and cfg.eval.eval_steps == 5000
    fb = configs.load_config("FB15k-237", "cpg")
    assert fb.model.relation_embedding_size == 32 and fb.model.batch_norm_momentum == 0.99
    assert fb.training.num_labels == 1000 and fb.training.prop_negatives == 100.0
    um = configs.load_config("umls", "cpg")
    assert um.context.context_rel_out == [64] and um.training.num_labels is None
    assert configs.load_config("WN18RR", "plain").context.context_rel_out is None
    assert configs.load_config("nell-995", "cpg").model.entity_embedding_size % 10 == 0
    assert len(configs.SHIPPED) == 22                                   # one entry per shipped YAML file
    with pytest.raises(KeyError):
        configs.load_config("WN18RR", "nonexistent")


def test_model_descriptors_and_yaml_roundtrip(tmp_path):
    cfg = configs.load_config("FB15k-237", "cpg")
    md = configs.model_descriptors(cfg, 14541, 474)
    assert md["use_negative_sampling"] is True and md["hidden_dropout"] == 0.3 and md["rel_emb_size"] == 32
    cfg.training.num_labels = None
    assert configs.model_descriptors(cfg, 14541, 474)["use_negative_sampling"] is False
    import yaml
    p = os.path.join(tmp_path, "c.yaml")
    yaml.safe_dump({k: dict(v) for k, v in cfg.items()}, open(p, "w"))
    again = configs.load_config(p)
    assert again.model.relation_embedding_size == 32 and again.training.num_labels is None
