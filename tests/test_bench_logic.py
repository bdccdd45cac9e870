"""bench.py's own checker and bookkeeping (CPU): the float64 ranking it compares the timed step against, the mismatch
counter with its near-tie rule, and the shard / exchange sizing it relies on."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import bench  # noqa: E402
from oracle import search_oracle as so  # noqa: E402


def test_reference_topk_f64_equals_the_numpy_oracle():
    g = torch.Generator().manual_seed(0)
    corpus = torch.nn.functional.normalize(torch.randn(3000, 64, generator=g), dim=1).bfloat16()
    q = torch.nn.functional.normalize(torch.randn(5, 64, generator=g), dim=1).bfloat16()
    ids, scores = bench.reference_topk_f64(corpus, q, 12, row_offset=1000, chunk=700)
    want_i, want_s, _, _ = so.topk_exact(corpus.float().numpy(), q.float().numpy(), 12)
    np.testing.assert_array_equal(ids.numpy(), want_i + 1000)
    np.testing.assert_allclose(scores.numpy(), want_s, atol=1e-12)
    # a shard shorter than kk is padded with (-1, -inf)
    ids2, sc2 = bench.reference_topk_f64(corpus[:5], q, 8, row_offset=0)
    assert (ids2[:, 5:] == -1).all() and torch.isinf(sc2[:, 5:]).all()


def test_mismatch_counter_exact_and_near_tie_rules():
    want_ids = np.array([[10, 11, 12, 13, 14, 15]])
    want_sc = np.array([[0.9, 0.8, 0.8 - 1e-7, 0.7, 0.6, 0.6 - 1e-7]])     # ranks 1-2 tie, ranks 4-5 tie (5 is past k)
    k = 5
    assert bench.count_id_mismatches(np.array([[10, 11, 12, 13, 14]]), want_ids, want_sc, k) == 0
    assert bench.count_id_mismatches(np.array([[10, 12, 11, 13, 14]]), want_ids, want_sc, k) == 0     # swap inside a tie
    assert bench.count_id_mismatches(np.array([[10, 11, 12, 13, 15]]), want_ids, want_sc, k) == 0     # tie reaching past k
    assert bench.count_id_mismatches(np.array([[11, 10, 12, 13, 14]]), want_ids, want_sc, k) > 0      # a real inversion
    assert bench.count_id_mismatches(np.array([[10, 11, 12, 13, 99]]), want_ids, want_sc, k) > 0      # a wrong row


def test_shard_bounds_and_exchange_buffer_sizes():
    from comorag_b200 import _native
    from comorag_b200.dist import shard_bounds
    for world in (1, 2, 4, 8):
        offs = shard_bounds(10_000_000, world)
        assert offs[0] == 0 and offs[-1] == 10_000_000 and max(np.diff(offs)) - min(np.diff(offs)) <= 1
    lib = _native.load()
    sizes = [lib.crag_exchange_buffer_bytes(w) for w in (1, 2, 8, 16)]
    assert all(s > 0 and s % 256 == 0 for s in sizes) and sizes == sorted(sizes)
    assert lib.crag_exchange_buffer_bytes(0) == 0 and lib.crag_exchange_buffer_bytes(17) == 0
    # one rank's slot holds 128 ids + 128 scores + (min, max): the buffer covers 2 parities x world x 32 queries of them
    assert sizes[2] >= 2 * 8 * 32 * (128 * 12 + 8)


def test_synthetic_vocab_and_texts_tokenise_one_token_per_word():
    vocab = bench.synthetic_vocab(1000)
    assert len(vocab) == 1000 and vocab[:5] == ["[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]"]
    texts = bench.synthetic_texts(3, 20, seed=1, vocab_size=1000)
    assert all(len(t.split()) == 20 and all(w in set(vocab) for w in t.split()) for t in texts)


def test_both_arms_print_the_same_config_object():
    """`bench.py` and `bench.py --impl reference` must describe the SAME workload (the driver compares the two
    `config` objects); rank 0's row count is the one comorag_b200.dist.shard_bounds gives."""
    import bench
    from comorag_b200.dist import shard_bounds
    for rows, world in ((10_000_000, 1), (10_000_000, 8), (1_000_003, 4)):
        cfg = bench.workload_config(rows, 1024, 32, 10, world)
        offs = shard_bounds(rows, world)
        assert cfg["rows_per_rank"] == offs[1] - offs[0]
        assert cfg["index_rows"] == rows and cfg["queries_per_step"] == 32 and cfg["k"] == 10
        assert f"over {world} GPU(s)" in cfg["workload"] and "L2" in cfg["l2"]
        assert cfg == bench.workload_config(rows, 1024, 32, 10, world)
    src = open(bench.__file__).read()
    assert src.count('"config": workload_config(') == 2      # our arm and the reference arm, nothing hand-written beside it


def test_dump_outputs_writes_float_arrays(tmp_path):
    ids = np.array([[3, 1 << 40]], dtype=np.int64)
    scores = np.array([[0.5, 0.25]], dtype=np.float32)
    bench.dump_outputs(str(tmp_path / "out"), {"ids": ids, "scores": scores})
    got_ids, got_scores = np.load(tmp_path / "out" / "ids.npy"), np.load(tmp_path / "out" / "scores.npy")
    assert got_ids.dtype == np.float64 and (got_ids.astype(np.int64) == ids).all()
    assert got_scores.dtype == np.float32 and (got_scores == scores).all()
