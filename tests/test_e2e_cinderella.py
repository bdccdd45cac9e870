"""End to end: the reference's UNMODIFIED ComoRAG.index() + try_answer() on its bundled cinderella sample (BASELINE
config 1; entry point main_openai.py:23-25), driven offline by tests/e2e_harness.py (LLM stub, igraph/umap/tiktoken
stand-ins), was run once on the reference's own classes (CPU, fp32 HF encoder + numpy search).  Its trace is committed
(golden/e2e_cinderella_reference.json), and so is what its retrieval methods saw: every store's rows and every probe
with its query row (golden/e2e_cinderella_replay.npz, tests/golden/make_golden_e2e_replay.py).  The tests replay those
probes through the engine's retrieval methods on cuda:0 and compare the retrieved ids / scores of every probe.
"""
import json
import os
import sys
import tempfile

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import e2e_harness as H  # noqa: E402

GOLDEN = os.path.join(HERE, "golden", "e2e_cinderella_reference.json")


def golden_view():
    return H.retrieval_view(json.load(open(GOLDEN)))


def test_llm_stub_covers_every_prompt_family():
    sysm = lambda s: [{"role": "system", "content": s}]
    ner = json.loads(H.llm_reply(sysm("Your task is to extract named entities from the given paragraph.") +
                                 [{"role": "user", "content": "Cinderella went to the Palace with the Prince."}]))
    assert ner["named_entities"][:3] == ["Cinderella", "Palace", "Prince"]
    tri = json.loads(H.llm_reply(sysm("Your task is to construct an RDF graph") + [{"role": "user", "content":
                     "Paragraph:\n```\nx\n```\n\n" + json.dumps({"named_entities": ["A", "B"]})}]))
    assert ["A", "appears with", "B"] in tri["triples"]
    qa = H.llm_reply(sysm("qa") + [{"role": "user", "content": "### Detail Chunks\nabc\n\nQuestion: q\nThought: "}])
    assert qa.split("### Final Answer")[1].strip() == "*"
    qa2 = H.llm_reply(sysm("qa") + [{"role": "user", "content": "### Historical Information\nx\n\nQuestion: q\nThought: "}])
    assert qa2.split("### Final Answer")[1].strip() == "Cinderella"
    probes = json.loads(H.llm_reply(sysm("You are an expert in multi-turn retrieval-oriented probe generation.") +
                                    [{"role": "user", "content": "Original Query:\nHow did the prince find her?\n\nContext:\n"}]))
    assert sorted(probes) == ["probe_1", "probe_2"]


def test_igraph_stand_in_pagerank_is_a_distribution():
    g = H._Graph()
    g.add_vertices(4, attributes={"name": list("abcd")})
    g.add_edges([("a", "b"), ("b", "c"), ("c", "d")], attributes={"weight": [1.0, 2.0, 1.0]})
    p = g.personalized_pagerank(vertices=range(4), damping=0.5, reset=[1, 0, 0, 0])
    assert abs(sum(p) - 1.0) < 1e-9 and p[0] > p[1] > p[2] > p[3]


def test_recorded_reference_inputs_reproduce_the_committed_trace():
    """The recorded store rows and query rows, put through the reference's retrieval arithmetic (the oracle's
    restatement), give the committed trace: the replay fixture pins the reference side of the comparison."""
    rec = H.load_replay()
    gold = json.load(open(GOLDEN))
    out = H.replay_reference(rec)
    assert {k: sorted(v) for k, v in out["stores"].items()} == {k: sorted(v) for k, v in gold["stores"].items()}
    assert set(out["trace"]) == set(gold["trace"]) == set(rec["queries"].tolist())
    summary = H.compare_traces(H.retrieval_view(gold), out, raw_tol=0.0, floor_tol=5e-4)
    assert not summary["problems"], summary["problems"]
    assert summary["queries"] == len(gold["trace"]) == 12
    # the char-iteration bug (ComoRAG.py:470, 909-935): each tri_retrieve encoded len(query) single characters twice
    assert gold["query_encodes"]["encoded_texts"] > 20 * len(gold["trace"])


def _count_device_calls():
    from comorag_b200 import index as crag_index
    calls = {"scores": 0, "rank": 0, "topk": 0}
    real = (crag_index.DenseIndex.scores_device, crag_index.DenseIndex.rank_device, crag_index.DenseIndex.search_device)

    def counting(name, fn):
        def inner(self, *a, **kw):
            calls[name] += 1
            return fn(self, *a, **kw)
        return inner
    crag_index.DenseIndex.scores_device = counting("scores", real[0])
    crag_index.DenseIndex.rank_device = counting("rank", real[1])
    crag_index.DenseIndex.search_device = counting("topk", real[2])

    def restore():
        (crag_index.DenseIndex.scores_device, crag_index.DenseIndex.rank_device, crag_index.DenseIndex.search_device) = real
    return calls, restore


def _replay(arm):
    rec = H.load_replay()
    calls, restore = _count_device_calls()
    try:
        with tempfile.TemporaryDirectory() as tmp:
            got = H.replay_engine(rec, arm, tmp)
    finally:
        restore()
    return rec, got, calls


@pytest.mark.gpu
def test_search_half_replay_on_the_device_matches_the_reference_rankings():
    """arm "shim_search": the reference's own fp32 rows feed OUR stores, and the fact / passage / summary / timeline
    searches of every probe run on the device kernels through the methods install() binds onto ComoRAG.  Only the
    bf16 storage of rows and queries separates the two arms: raw inner products may move by <= 4e-3, i.e. normalised
    scores by that over the result's raw range, and rankings must be consistent within the measured deviation."""
    rec, got, calls = _replay("shim_search")
    summary = H.compare_traces(golden_view(), got, raw_tol=4e-3)
    assert not summary["problems"], summary["problems"]
    n = len(rec["queries"])
    assert summary["queries"] == n >= 9
    # every tri_retrieve went through a retrieval wave: per wave one score-all pass over each of the fact / passage /
    # summary shards and one fused top-k pass over the timeline shard; per probe two device rankings
    waves, served = got["wave_stats"]["waves"], got["wave_stats"]["queries"]
    assert 1 <= waves <= served == n
    assert calls["scores"] >= 3 * waves and calls["rank"] >= 2 * served and calls["topk"] >= waves


@pytest.mark.gpu
def test_shim_retrieval_replay_retrieves_what_the_reference_retrieves():
    import torch
    rec, got, calls = _replay("shim")
    # the GPU encoder is bf16 against the reference's fp32 HF model (parity bar: embedding max-abs error <= 1e-2, i.e.
    # raw inner products of unit vectors within ~3e-2); this synthetic 2-layer checkpoint packs all texts into a
    # narrow cone, so the raw ranges that normalise the scores are small and the normalised deviations large.
    summary = H.compare_traces(golden_view(), got, raw_tol=3e-2)
    assert not summary["problems"], summary["problems"]
    n = len(rec["queries"])
    assert summary["queries"] == n >= 9
    waves, served = got["wave_stats"]["waves"], got["wave_stats"]["queries"]
    assert 1 <= waves <= served == n
    assert calls["scores"] >= 3 * waves and calls["rank"] >= 2 * served and calls["topk"] >= waves
    # the per-character encode waste is gone: one encoded text per tri_retrieve instead of 2 * len(query) + 4
    gold = json.load(open(GOLDEN))
    assert got["query_encodes"]["encoded_texts"] <= n + 16 * 3
    assert gold["query_encodes"]["encoded_texts"] > 5 * got["query_encodes"]["encoded_texts"]
    torch.cuda.synchronize()
