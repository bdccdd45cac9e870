"""Record what the reference's retrieval methods saw during its cinderella run, so the end-to-end comparison
(tests/test_e2e_cinderella.py) can replay every probe against the engine without the reference tree.

    COMORAG_REFERENCE=<ComoRAG checkout> python tests/golden/make_golden_e2e_replay.py

Runs the reference's unmodified ComoRAG.index() + try_answer() under tests/e2e_harness.py (the same run that produced
e2e_cinderella_reference.json) and writes tests/golden/e2e_cinderella_replay.npz:
  <ns>_keys / <ns>_texts / <ns>_emb   row order, texts and the reference's fp32 embeddings of every store the loop
                                      searched (chunk, entity, fact, summary, timeline)
  queries / query_emb                 every probe string the loop retrieved for, and the reference encoder's row for it
  epi_top_k                           the top_k the loop passed to get_similar_summaries
Before writing, the recorded rows are checked to reproduce the committed trace with the reference's own arithmetic.
"""
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import e2e_harness as H  # noqa: E402

OUT = os.path.join(HERE, "e2e_cinderella_replay.npz")
STORES = {"chunk": "ver_embedding_store", "entity": "entity_embedding_store", "fact": "fact_embedding_store",
          "summary": "sem_embedding_store", "timeline": "level_store"}


def capture(rag, batch_encode):
    out = {"epi_top_k": int(rag.global_config.qa_epi_top_k)}
    for ns, attr in STORES.items():
        store = getattr(rag, attr)
        out[ns + "_keys"] = np.array(store.get_all_ids())
        out[ns + "_texts"] = np.array(store.texts)
        out[ns + "_emb"] = np.asarray(store.embeddings, dtype=np.float32).reshape(len(store.texts), -1)
    return out


def main():
    root = H.find_reference_root()
    if root is None:
        raise SystemExit("set COMORAG_REFERENCE to a ComoRAG checkout (with dataset/cinderella)")
    with tempfile.TemporaryDirectory() as tmp:
        run = H.run_cinderella("reference", tmp, root, capture=capture)
    rec = run["captured"]
    queries = sorted(run["trace"])
    # the reference's BGE model prefixes its own instruction whatever the caller passes, so one row per probe
    from src.comorag.utils.config_utils import BaseConfig
    import src.comorag.embedding_model.BGEEmbedding as ref_bge
    model = ref_bge.BGEEmbeddingModel(global_config=BaseConfig(embedding_model_name=H.CKPT, embedding_batch_size=4,
                                                               embedding_max_seq_len=512),
                                      embedding_model_name=H.CKPT)
    rec["queries"] = np.array(queries)
    rec["query_emb"] = np.concatenate([model.batch_encode(q, norm=True) for q in queries]).astype(np.float32)

    gold = json.load(open(os.path.join(HERE, "e2e_cinderella_reference.json")))
    replayed = H.replay_reference(rec)
    summary = H.compare_traces(H.retrieval_view(gold), replayed, raw_tol=0.0, floor_tol=5e-4)
    assert not summary["problems"], summary["problems"]
    assert summary["queries"] == len(gold["trace"])
    np.savez_compressed(OUT, **rec)
    print(f"wrote {OUT} ({os.path.getsize(OUT)} bytes, {len(queries)} probes); replay vs committed trace: {summary}")


if __name__ == "__main__":
    main()
