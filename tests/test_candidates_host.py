"""Candidate scoring without a GPU: the argument checks of the two C entry points (rejected before anything is
launched), the dispatch of ranking_and_hits on candidate batches, and run_cpg --score-triples' argument and input
checks."""
import logging

import numpy as np
import pytest

from coper_b200 import _lib, build

ERR_INVALID_ARG, ERR_UNSUPPORTED = -1, -3
FAKE = 256               # never dereferenced: every case below is rejected before a launch


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def _score(lib, B=13, C=37, d=200, lo=0, hi=997, ptr=FAKE):
    return lib.coper_score_candidates(ptr, FAKE, FAKE, FAKE, B, C, d, lo, hi, FAKE, None)


def _rank(lib, B=13, C=37, d=200, lo=0, hi=997, entity_major=0, bits=None, e2=FAKE):
    return lib.coper_candidate_rank(FAKE, FAKE, FAKE, FAKE, e2, B, C, d, lo, hi, FAKE, bits, entity_major, FAKE, FAKE,
                                    None)


@pytest.mark.parametrize("kw", [dict(B=0), dict(C=0), dict(B=-1), dict(B=1 << 16, C=1 << 15), dict(d=0),
                                dict(lo=-1), dict(lo=500, hi=500), dict(lo=600, hi=500), dict(hi=1 << 31)])
def test_candidate_calls_reject_bad_arguments(lib, kw):
    assert _score(lib, **kw) == ERR_INVALID_ARG
    assert _rank(lib, **kw) == ERR_INVALID_ARG


def test_candidate_calls_reject_unsupported_width(lib):
    assert _score(lib, d=257) == ERR_UNSUPPORTED
    assert _rank(lib, d=257) == ERR_UNSUPPORTED


def test_candidate_calls_reject_missing_buffers_and_bad_layout(lib):
    assert _score(lib, ptr=None) == ERR_INVALID_ARG
    assert _rank(lib, e2=None) == ERR_INVALID_ARG
    assert _rank(lib, entity_major=2, bits=FAKE) == ERR_INVALID_ARG


# ------------------------------------------------------------------------------------------ ranking_and_hits
class _FakeModel:
    """Records which rank call ranking_and_hits makes; returns fixed ranks."""

    def __init__(self):
        self.calls = []

    def filtered_ranks(self, batch):
        import torch
        self.calls.append(("full", None))
        return torch.full((len(batch["e1"]),), 3, dtype=torch.int32), torch.zeros(len(batch["e1"]), dtype=torch.int32)

    def candidate_ranks(self, batch, candidates, filtered=True):
        import torch
        self.calls.append(("cand", filtered, tuple(candidates.shape)))
        return torch.full((len(batch["e1"]),), 2, dtype=torch.int32), torch.zeros(len(batch["e1"]), dtype=torch.int32)


def test_ranking_and_hits_dispatches_candidate_batches(tmp_path, caplog):
    from coper_b200.metrics import ranking_and_hits
    ids = np.arange(4)
    cand = np.zeros((4, 5), np.int32)
    batches = [
        {"e1": ids, "rel": ids, "e2": ids, "candidates": cand, "e2_multi_rowptr": np.arange(5), "e2_multi_col": ids},
        {"e1": ids, "rel": ids, "e2": ids, "candidates": cand},
        {"e1": ids, "rel": ids, "e2": ids, "e2_multi_rowptr": np.arange(5), "e2_multi_col": ids},
    ]
    m = _FakeModel()
    with caplog.at_level(logging.INFO, logger="coper_b200.metrics"):
        mr, mrr, hits, ranks = ranking_and_hits(m, str(tmp_path), batches, "test", return_ranks=True)
    assert m.calls == [("cand", True, (4, 5)), ("cand", False, (4, 5)), ("full", None)]
    assert ranks.tolist() == [2] * 8 + [3] * 4
    assert hits[1] == 0.0 and hits[3] == 1.0
    assert any("C = 5 given candidates" in r.getMessage() for r in caplog.records)


def test_ranking_and_hits_without_candidates_does_not_mention_them(tmp_path, caplog):
    from coper_b200.metrics import ranking_and_hits
    ids = np.arange(4)
    m = _FakeModel()
    with caplog.at_level(logging.INFO, logger="coper_b200.metrics"):
        ranking_and_hits(m, str(tmp_path), [{"e1": ids, "rel": ids, "e2": ids}], "test")
    assert m.calls == [("full", None)]
    assert not any("candidates" in r.getMessage() for r in caplog.records)


# ------------------------------------------------------------------------------------------ run_cpg --score-triples
def test_run_cpg_score_triples_needs_a_checkpoint():
    from coper_b200 import run_cpg
    with pytest.raises(SystemExit) as e:
        run_cpg.main(["--synthetic", "toy", "--score-triples", "facts.tsv"])
    assert e.value.code == 2


NAMES = (["alice", "bob", "carol"], ["knows", "likes"])


def _write(tmp_path, text):
    p = tmp_path / "facts.tsv"
    p.write_text(text)
    return str(p)


def test_read_triples_maps_names(tmp_path):
    from coper_b200.run_cpg import _read_triples
    path = _write(tmp_path, "alice\tknows\tbob\n\ncarol\tlikes\talice\n")
    e1, rel, e2, cols = _read_triples(path, NAMES, 3, 2)
    assert e1.tolist() == [0, 2] and rel.tolist() == [0, 1] and e2.tolist() == [1, 0]
    assert cols == [["alice", "knows", "bob"], ["carol", "likes", "alice"]]


def test_read_triples_plain_ids(tmp_path):
    from coper_b200.run_cpg import _read_triples
    e1, rel, e2, _ = _read_triples(_write(tmp_path, "0\t1\t2\n2\t0\t1\n"), None, 3, 2)
    assert e1.tolist() == [0, 2] and rel.tolist() == [1, 0] and e2.tolist() == [2, 1]


@pytest.mark.parametrize("text, names, needle", [
    ("alice\tknows\tbob\nalice\tknows\tdave\n", NAMES, ":2: unknown entity name 'dave'"),
    ("alice\thates\tbob\n", NAMES, ":1: unknown relation name 'hates'"),
    ("alice\tknows\n", NAMES, ":1: expected 3 tab-separated columns"),
    ("0\t1\t2\n0\t1\t3\n", None, ":2: entity id 3 out of range"),
    ("0\tx\t2\n", None, ":1: 'x' is not an integer relation id"),
])
def test_read_triples_reports_file_and_line(tmp_path, text, names, needle):
    from coper_b200.run_cpg import _read_triples
    path = _write(tmp_path, text)
    with pytest.raises(SystemExit) as e:
        _read_triples(path, names, 3, 2)
    assert str(e.value.code).startswith(path) and needle in str(e.value.code)
