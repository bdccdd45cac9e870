"""Test-side harness that runs the reference's UNMODIFIED `ComoRAG.index()` + `try_answer()` offline (SURVEY.md section 4):

  * a localhost OpenAI-compatible `/v1/chat/completions` stub with deterministic canned replies for every prompt family
    the loop sends (NER, triples, summaries, QA, probes, memory/node fusion, the DSPy fact filter);
  * stand-ins for modules this image lacks: `igraph` (a small Graph over python lists + a power-iteration personalised
    PageRank), `umap` (deterministic PCA projection), and `tiktoken.get_encoding` (whitespace token counter; the real
    one downloads its BPE table);
  * a recorder around the four retrieval entry points so a run leaves a trace {query: rankings / scores}.

The same harness drives both arms -- the reference's own classes on CPU and the comorag_b200 shim on cuda:0 -- so
whatever the stand-ins approximate, they approximate identically for both.  Nothing in here is product code; nothing
in comorag_b200/ imports it.  Running the loop needs a reference checkout, named by $COMORAG_REFERENCE; the tests replay
what such a run recorded (see "replay" below) and need no checkout.
"""
from __future__ import annotations

import json
import os
import re
import sys
import threading
import types
from http.server import BaseHTTPRequestHandler, ThreadingHTTPServer
from typing import Any, Dict, List, Optional

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CKPT = os.path.join(ROOT, "tests", "golden", "bge-tiny-synth")


def find_reference_root() -> Optional[str]:
    cand = os.environ.get("COMORAG_REFERENCE")
    if cand and os.path.isdir(os.path.join(cand, "src", "comorag")) and \
            os.path.isdir(os.path.join(cand, "dataset", "cinderella")):
        return cand
    return None


# ------------------------------------------------------------------------------------------------ LLM stub
_STOP = {"the", "and", "that", "with", "from", "this", "were", "have", "what", "when", "then", "they", "them", "there",
         "into", "your", "which", "about", "will", "would", "their", "said", "been", "before", "after", "where"}


def _words(text: str) -> List[str]:
    return re.findall(r"[A-Za-z']+", text)


def _entities(passage: str, limit: int = 8) -> List[str]:
    seen: List[str] = []
    for w in re.findall(r"\b[A-Z][a-z]{3,}\b", passage):
        if w.lower() not in _STOP and w not in seen:
            seen.append(w)
    for w in sorted({w.lower() for w in _words(passage) if len(w) > 6 and w.lower() not in _STOP}):
        if len(seen) >= limit:
            break
        if w not in seen:
            seen.append(w)
    return seen[:limit]


def _bag_summary(text: str, n: int = 30) -> str:
    counts: Dict[str, int] = {}
    for w in _words(text.lower()):
        if len(w) > 3 and w not in _STOP:
            counts[w] = counts.get(w, 0) + 1
    top = sorted(counts.items(), key=lambda kv: (-kv[1], kv[0]))[:n]
    return "Summary: " + " ".join(w for w, _ in top)


def llm_reply(messages: List[Dict[str, str]]) -> str:
    system = messages[0]["content"] if messages and messages[0]["role"] == "system" else ""
    user = messages[-1]["content"]
    if system.startswith("Your task is to extract named entities"):
        return json.dumps({"named_entities": _entities(user)})
    if system.startswith("Your task is to construct an RDF"):
        m = re.search(r"\{\s*\"named_entities\".*\}", user, re.S)
        ents = json.loads(m.group())["named_entities"] if m else []
        triples = [[a, "appears with", b] for a, b in zip(ents, ents[1:])] + [[e, "is part of", "the story"] for e in ents[:3]]
        return json.dumps({"triples": triples})
    if "fact_before_filter" in system or "[[ ## fact_before_filter ## ]]" in user:
        m = re.search(r"\[\[ ## fact_before_filter ## \]\]\n(.*?)\n\n", user, re.S)
        facts = json.loads(m.group(1))["fact"] if m else []
        keep = sorted(facts)[: min(3, len(facts))]            # order-independent choice
        return "[[ ## fact_after_filter ## ]]\n" + json.dumps({"fact": keep}) + "\n\n[[ ## completed ## ]]"
    if "retrieval-oriented probe generation" in system:
        q = re.search(r"Original Query:\n(.*?)\n\nContext:", user, re.S)
        ents = [w for w in _words(q.group(1) if q else user) if len(w) > 3 and w.lower() not in _STOP][:3]
        return json.dumps({f"probe_{i + 1}": f"What does the story say about {e}?" for i, e in enumerate(ents)})
    if "expert narrative analyst" in system:       # memory_fusion
        q = re.search(r"Questions:\n(.*?)\n\nContent:\n(.*)\n\nYour Response:", user, re.S)
        return "- Key Finding: " + _bag_summary(q.group(2) if q else user, 12)
    if "narrative synthesis specialist" in system:  # node_fusion
        return "Fused: " + _bag_summary(user, 12)
    if user.startswith("Write a summary of the following"):
        return _bag_summary(user.split(":", 1)[1])
    if user.rstrip().endswith("Thought:"):          # rag_qa_*: force one probe cycle, then answer
        if "### Historical Information" not in user:
            return "The context is not sufficient yet.\n### Final Answer\n*"
        return "The notes answer it.\n### Final Answer\nCinderella"
    return "OK"


class _Handler(BaseHTTPRequestHandler):
    def log_message(self, *a):   # quiet
        pass

    def do_POST(self):
        body = json.loads(self.rfile.read(int(self.headers.get("Content-Length", "0"))) or b"{}")
        text = llm_reply(body.get("messages", []))
        payload = json.dumps({
            "id": "stub", "object": "chat.completion", "created": 0, "model": body.get("model", "stub"),
            "choices": [{"index": 0, "message": {"role": "assistant", "content": text}, "finish_reason": "stop"}],
            "usage": {"prompt_tokens": 1, "completion_tokens": 1, "total_tokens": 2}}).encode()
        self.send_response(200)
        self.send_header("Content-Type", "application/json")
        self.send_header("Content-Length", str(len(payload)))
        self.end_headers()
        self.wfile.write(payload)


class LLMStub:
    def __enter__(self):
        self.server = ThreadingHTTPServer(("127.0.0.1", 0), _Handler)
        self.server.daemon_threads = True
        self.thread = threading.Thread(target=self.server.serve_forever, daemon=True)
        self.thread.start()
        self.url = f"http://localhost:{self.server.server_address[1]}/v1"
        return self

    def __exit__(self, *exc):
        self.server.shutdown()
        self.server.server_close()


# ------------------------------------------------------------------------------------------------ module stand-ins
class _Vertex:
    def __init__(self, g, i):
        self._g, self.index = g, i

    def __getitem__(self, k):
        return self._g._vattr[k][self.index]

    def attributes(self):
        return {k: v[self.index] for k, v in self._g._vattr.items()}


class _VertexSeq:
    def __init__(self, g):
        self._g = g

    def __call__(self):
        return self

    def __len__(self):
        return self._g._n

    def __iter__(self):
        return (_Vertex(self._g, i) for i in range(self._g._n))

    def __getitem__(self, k):
        if isinstance(k, str):
            if k not in self._g._vattr:
                raise KeyError(k)
            return list(self._g._vattr[k])
        return _Vertex(self._g, k)

    def attribute_names(self):
        return list(self._g._vattr)


class _EdgeSeq:
    def __init__(self, g):
        self._g = g

    def __call__(self):
        return self

    def __len__(self):
        return len(self._g._edges)


class _Graph:
    """The slice of igraph.Graph that ComoRAG.py touches (ComoRAG.py:161-182, 628-654, 779-841, 890, 1001, 1092)."""

    def __init__(self, directed=False):
        self.directed = directed
        self._n = 0
        self._vattr: Dict[str, list] = {}
        self._edges: List[tuple] = []
        self._weights: List[float] = []

    @property
    def vs(self):
        return _VertexSeq(self)

    @property
    def es(self):
        return _EdgeSeq(self)

    def vcount(self):
        return self._n

    def ecount(self):
        return len(self._edges)

    def add_vertices(self, n, attributes=None):
        attributes = attributes or {}
        for k in set(self._vattr) | set(attributes):
            col = self._vattr.setdefault(k, [None] * self._n)
            col.extend(attributes.get(k, [None] * n))
        self._n += n

    def add_edges(self, edges, attributes=None):
        name_to_idx = {nm: i for i, nm in enumerate(self._vattr.get("name", []))}
        w = (attributes or {}).get("weight", [1.0] * len(edges))
        for (a, b), wt in zip(edges, w):
            self._edges.append((name_to_idx[a] if isinstance(a, str) else a, name_to_idx[b] if isinstance(b, str) else b))
            self._weights.append(float(wt))

    def write_graphml(self, path):
        with open(path + ".json", "w") as f:
            json.dump({"n": self._n, "vattr": self._vattr, "edges": self._edges, "weights": self._weights}, f)

    @classmethod
    def Read_GraphML(cls, path):
        raise FileNotFoundError(path)      # the harness always starts from a fresh save_dir

    def personalized_pagerank(self, vertices=None, damping=0.85, directed=False, weights=None, reset=None,
                              implementation=None):
        n = self._n
        W = np.zeros((n, n), dtype=np.float64)
        for (a, b), wt in zip(self._edges, self._weights):
            W[a, b] += wt
            W[b, a] += wt
        out = W.sum(axis=1)
        r = np.asarray(reset, dtype=np.float64)
        r = r / r.sum() if r.sum() > 0 else np.full(n, 1.0 / n)
        P = np.divide(W, out[:, None], out=np.zeros_like(W), where=out[:, None] > 0)
        p = r.copy()
        for _ in range(200):
            dangling = p[out == 0].sum()
            p_new = damping * (P.T @ p + dangling * r) + (1 - damping) * r
            if np.abs(p_new - p).sum() < 1e-14:
                p = p_new
                break
            p = p_new
        idx = list(vertices) if vertices is not None else list(range(n))
        return [float(p[i]) for i in idx]


class _UMAP:
    """Deterministic stand-in: centre + PCA to n_components (the reference only needs *a* low-dimensional layout for
    its GMM, cluster_utils.py:191-211)."""

    def __init__(self, n_neighbors=15, n_components=2, metric="cosine", random_state=None, **kw):
        self.n_components = n_components

    def fit_transform(self, X):
        if self.n_components < 1:
            raise ValueError("n_components must be greater than 0")   # as umap-learn does; the caller falls back
        X = np.asarray(X, dtype=np.float64)
        X = X - X.mean(axis=0, keepdims=True)
        u, s, vt = np.linalg.svd(X, full_matrices=False)
        k = min(self.n_components, vt.shape[0])
        Y = u[:, :k] * s[:k]
        for j in range(k):                    # fix the sign so tiny input changes cannot mirror an axis
            if Y[np.argmax(np.abs(Y[:, j])), j] < 0:
                Y[:, j] = -Y[:, j]
        return np.round(Y, 3)                 # coarse grid: robust to the 1e-3 differences between the two arms


class _WordEncoding:
    def encode(self, text):
        return text.split()


def install_stand_ins() -> None:
    if "igraph" not in sys.modules:
        ig = types.ModuleType("igraph")
        ig.Graph = _Graph
        sys.modules["igraph"] = ig
    if "umap" not in sys.modules:
        um = types.ModuleType("umap")
        um.UMAP = _UMAP
        sys.modules["umap"] = um
    import tiktoken
    tiktoken.get_encoding = lambda name: _WordEncoding()


# ------------------------------------------------------------------------------------------------ the run
def _h(text: str) -> str:
    """Texts are recorded by a short content hash (keeps the committed trace small)."""
    import hashlib
    return hashlib.md5(text.encode()).hexdigest()[:16]


def _json_safe(x: Any) -> Any:
    if isinstance(x, np.ndarray):
        return x.tolist()
    if isinstance(x, (np.floating, np.integer)):
        return x.item()
    return x


def run_cinderella(arm: str, workdir: str, ref_root: str, max_loops: int = 1, questions: Optional[int] = None,
                   capture=None) -> Dict:
    """arm = "reference": the reference's own classes on CPU (fp32 HF encoder, numpy search);
    arm = "shim": comorag_b200.install() first, then the SAME unmodified ComoRAG.py (needs cuda:0);
    arm = "shim_search": install(encoder=False): reference encoder, engine stores + device search (needs cuda:0).
    `capture(rag, batch_encode)`, if given, runs after try_answer and its result is returned under "captured".
    Returns {"trace": {...}, "solutions": [...], "encodes": int, "kernel_search_calls": int}."""
    sys.dont_write_bytecode = True
    if ref_root not in sys.path:
        sys.path.insert(0, ref_root)
    install_stand_ins()
    os.environ.setdefault("OPENAI_API_KEY", "stub")
    import src.comorag  # noqa: F401
    main = sys.modules["src.comorag.ComoRAG"]
    from src.comorag.utils.config_utils import BaseConfig
    import src.comorag.embedding_model as ref_em
    import src.comorag.embedding_model.BGEEmbedding as ref_bge

    if arm == "shim":
        import comorag_b200.install as crag
        crag.install("src.comorag")
    if arm == "shim_search":       # the reference's fp32 CPU encoder, our stores + device search under ComoRAG.py
        import comorag_b200.install as crag
        crag.install("src.comorag", encoder=False)
    if arm != "shim":
        # `accelerate` is absent: drop device_map from the HF init params (SURVEY.md section 8c, shim 2)
        if not getattr(ref_bge.BGEEmbeddingModel, "_harness_patched", False):
            _orig_init = ref_bge.BGEEmbeddingModel._init_embedding_config

            def _init(self, _orig_init=_orig_init):
                _orig_init(self)
                self.embedding_config.model_init_params.pop("device_map", None)
            ref_bge.BGEEmbeddingModel._init_embedding_config = _init
            ref_bge.BGEEmbeddingModel._harness_patched = True

    data = os.path.join(ref_root, "dataset", "cinderella", "cinderella_1")
    docs = [json.loads(l)["contents"] for l in open(os.path.join(data, "corpus.jsonl")) if l.strip()]
    queries = [json.loads(l)["question"] for l in open(os.path.join(data, "qas.jsonl")) if l.strip()]
    if questions:
        queries = queries[:questions]

    trace: Dict[str, Dict] = {}
    lock = threading.Lock()
    counters = {"encodes": 0, "encoded_texts": 0}
    cls = main.ComoRAG

    def record(kind, query, value):
        with lock:
            trace.setdefault(query, {})[kind] = value

    wrapped = {}
    tools: Dict[str, Any] = {}

    def raw_range(self, matrix, query) -> Optional[float]:
        """max - min of the RAW inner products behind a min-max-normalised result (harness-side: the tolerance on
        normalised scores is a raw-score error bound divided by this range)."""
        enc = tools.get("encode")
        if enc is None:
            return None
        E = np.asarray(matrix, dtype=np.float32)
        if E.ndim != 2 or E.shape[0] == 0:
            return None
        raw = E @ np.asarray(enc(query), dtype=np.float32).reshape(-1)
        return float(raw.max() - raw.min())

    def wrap(name, fn):
        orig = getattr(cls, name)
        wrapped[name] = orig

        def inner(self, *a, **kw):
            out = orig(self, *a, **kw)
            fn(self, out, *a, **kw)
            return out
        setattr(cls, name, inner)

    # rows are recorded by key: the stores' ROW ORDER depends on thread completion order (as_completed loops at
    # openie_openai.py:206-226 and ComoRAG.py:1166-1176), their contents do not
    def rec_facts(self, out, query):
        record("fact_scores", query, dict(zip(self.fact_node_keys, np.asarray(out, dtype=np.float64).tolist())))
        record("fact_range", query, raw_range(self, self.fact_embeddings, query))
    wrap("get_fact_scores", rec_facts)
    wrap("dense_passage_retrieval", lambda self, out, query, need_cluster=False: record(
        "sem" if need_cluster else "ver",
        query, {"ids": [self.summary_node_keys[i] if need_cluster else self.passage_node_keys[i] for i in np.asarray(out[0]).tolist()],
                "scores": np.asarray(out[1], dtype=np.float64).tolist(),
                "range": raw_range(self, self.summary_embeddings if need_cluster else self.passage_embeddings, query)}))
    wrap("graph_search_with_fact_entities", lambda self, out, *a, **kw: record(
        "ppr", kw.get("query", a[0] if a else None),
        {"ids": [self.passage_node_keys[i] for i in np.asarray(out[0]).tolist()],
         "scores": np.asarray(out[1], dtype=np.float64).tolist()}))
    wrap("tri_retrieve", lambda self, out, query=None, memory_pool=None, **kw: record(
        "docs", query, {k: [_h(t) for t in v] for k, v in out[0].items()}))
    orig_gss = main.get_similar_summaries

    def gss(query, level_store, embedding_model, top_k=3, **kw):
        texts, scores = orig_gss(query=query, level_store=level_store, embedding_model=embedding_model, top_k=top_k, **kw)
        rng = None
        if tools.get("encode") is not None and len(level_store.get_all_ids()):
            E = np.asarray(level_store.get_embeddings(level_store.get_all_ids()), dtype=np.float32)
            raw = E @ np.asarray(tools["encode"](query), dtype=np.float32).reshape(-1)
            rng = float(raw.max() - raw.min())
        record("epi", query, {"texts": [_h(t) for t in texts], "scores": [float(s) for s in scores], "range": rng})
        return texts, scores
    main.get_similar_summaries = gss

    try:
        with LLMStub() as llm:
            cfg = BaseConfig(llm_base_url=llm.url, llm_name="stub-llm", llm_api_key="stub", dataset="cinderella",
                             embedding_model_name=CKPT, embedding_batch_size=4, embedding_max_seq_len=512,
                             need_cluster=True, output_dir=os.path.join(workdir, "result"),
                             save_dir=os.path.join(workdir, "outputs"), max_meta_loop_max_iterations=max_loops,
                             is_mc=False, max_tokens_ver=2000, max_tokens_sem=2000, max_tokens_epi=2000)
            rag = cls(global_config=cfg)
            model = rag.embedding_model
            orig_be = model.batch_encode

            def counting_batch_encode(texts, **kw):
                with lock:
                    counters["encodes"] += 1
                    counters["encoded_texts"] += 1 if isinstance(texts, str) else len(texts)
                return orig_be(texts, **kw)
            model.batch_encode = counting_batch_encode
            tools["encode"] = lambda text: orig_be(text)      # harness-side encodes do not count
            rag.index(docs)
            index_encodes = dict(counters)
            solutions = rag.try_answer(queries)
            stores = {
                "chunk": rag.ver_embedding_store.get_all_ids(), "entity": rag.entity_embedding_store.get_all_ids(),
                "fact": rag.fact_embedding_store.get_all_ids(), "summary": rag.sem_embedding_store.get_all_ids(),
                "timeline": rag.level_store.get_all_ids(),
            }
            n_edges = rag.graph.ecount()
            captured = capture(rag, orig_be) if capture is not None else None
            wave = getattr(rag, "_crag_wave", None)
            wave_stats = dict(wave.stats) if wave is not None else None
            if wave is not None:
                wave.close()
    finally:
        for name, original in wrapped.items():
            setattr(cls, name, original)
        main.get_similar_summaries = orig_gss
    return {"arm": arm, "wave_stats": wave_stats if arm != "reference" else None, "trace": trace, "answers": [getattr(s, "answer", None) for s in solutions], "stores": stores,
            "graph_edges": n_edges, "index_encodes": index_encodes,
            "query_encodes": {k: counters[k] - index_encodes[k] for k in counters}, "queries": queries,
            "captured": captured}


# ------------------------------------------------------------------------------------------------ comparison
def ranking_consistent(ref_ids: List, ref_scores: List[float], got_ids: List, got_scores: List[float], slack: float):
    """Both rankings order the same items; positions may differ only among items whose REFERENCE scores are within
    `slack` of each other (the two arms' scores differ by the encoder's bf16 error).  Returns (ok, message)."""
    if sorted(ref_ids) != sorted(got_ids):
        return False, f"different item sets: {set(ref_ids) ^ set(got_ids)}"
    ref_s = dict(zip(ref_ids, ref_scores))
    for pos, (a, b) in enumerate(zip(ref_ids, got_ids)):
        if a != b and abs(ref_s[a] - ref_s[b]) > slack:
            return False, f"rank {pos}: reference {a} ({ref_s[a]:.4f}) vs {b} ({ref_s[b]:.4f}), slack {slack:.4f}"
    return True, ""


def compare_traces(ref: Dict, got: Dict, raw_tol: float = 4e-3, floor_tol: float = 1e-3) -> Dict:
    """The shim arm must have retrieved what the reference arm retrieved, query by query.  Scores are min-max
    normalised ((s - min) / (max - min), misc_utils.py:141-150), so a raw inner-product error e shows up as e / range:
    the allowed deviation of a result is floor_tol + 2 * raw_tol / (the reference's raw range of that result)
    (raw_tol: 4e-3 covers bf16 storage of unit rows and queries; the bf16 ENCODER adds its embedding error on top).
    Rankings are then checked for consistency within twice the MEASURED deviation of each query.
    Returns a report {"queries", "max_score_dev", "max_ppr_dev", "problems": [...]} -- no problems is a pass."""
    problems: List[str] = []
    for ns in ref["stores"]:
        if sorted(ref["stores"][ns]) != sorted(got["stores"][ns]):
            problems.append(f"{ns} store contents differ between the arms")
    if set(ref["trace"]) != set(got["trace"]):
        problems.append(f"different probe sets: {sorted(set(ref['trace']) ^ set(got['trace']))}")
    worst, worst_ppr, checked = 0.0, 0.0, 0
    for query, r in ref["trace"].items():
        g = got["trace"].get(query)
        if g is None or set(r) != set(g):
            problems.append(f"{query!r}: recorded kinds differ")
            continue
        if set(r["fact_scores"]) != set(g["fact_scores"]):
            problems.append(f"{query!r}: fact sets differ")
            continue
        def allowed(rng):
            return floor_tol + (2 * raw_tol / rng if rng else 1.0)

        fkeys = sorted(r["fact_scores"])
        fr = np.asarray([r["fact_scores"][f] for f in fkeys])
        fg = np.asarray([g["fact_scores"][f] for f in fkeys])
        dev = float(np.abs(fr - fg).max()) if fr.size else 0.0
        if dev > allowed(r.get("fact_range")):
            problems.append(f"{query!r} facts: normalised scores differ by {dev:.4f} > {allowed(r.get('fact_range')):.4f}")
        for kind in ("ver", "sem"):
            rs, gs = dict(zip(r[kind]["ids"], r[kind]["scores"])), dict(zip(g[kind]["ids"], g[kind]["scores"]))
            if set(rs) != set(gs):
                problems.append(f"{query!r} {kind}: different item sets")
                continue
            d = max((abs(rs[i] - gs[i]) for i in rs), default=0.0)
            if d > allowed(r[kind].get("range")):
                problems.append(f"{query!r} {kind}: normalised scores differ by {d:.4f} > {allowed(r[kind].get('range')):.4f}")
            dev = max(dev, d)
        re_, ge_ = dict(zip(r["epi"]["texts"], r["epi"]["scores"])), dict(zip(g["epi"]["texts"], g["epi"]["scores"]))
        if set(re_) == set(ge_):
            d = max((abs(re_[i] - ge_[i]) for i in re_), default=0.0)
            if d > allowed(r["epi"].get("range")):
                problems.append(f"{query!r} epi: normalised scores differ by {d:.4f} > {allowed(r['epi'].get('range')):.4f}")
            dev = max(dev, d)
        worst = max(worst, dev)
        slack = 2 * dev + 1e-6
        # facts: the linking_top_k candidates (ComoRAG.py:475)
        k = min(5, fr.size)
        top_r, top_g = np.argsort(fr)[-k:][::-1].tolist(), np.argsort(fg)[-k:][::-1].tolist()
        for a in set(top_r) ^ set(top_g):
            kth = fr[top_r[-1]]
            if abs(fr[a] - kth) > slack:
                problems.append(f"{query!r}: fact {fkeys[a]} in one top-{k} only, gap {abs(fr[a] - kth):.4f} > {slack:.4f}")
        for kind in ("ver", "sem"):
            ok, msg = ranking_consistent(r[kind]["ids"], r[kind]["scores"], g[kind]["ids"], g[kind]["scores"], slack)
            if not ok:
                problems.append(f"{query!r} {kind}: {msg}")
        if ("ppr" in r) != ("ppr" in g):
            problems.append(f"{query!r}: only one arm went through the graph search")
        elif "ppr" in r:      # the graph search's final passage ranking (PPR over weights built from the scores above)
            pr, pg = dict(zip(r["ppr"]["ids"], r["ppr"]["scores"])), dict(zip(g["ppr"]["ids"], g["ppr"]["scores"]))
            pdev = max(abs(pr[i] - pg[i]) for i in pr)
            worst_ppr = max(worst_ppr, pdev)
            ok, msg = ranking_consistent(r["ppr"]["ids"], r["ppr"]["scores"], g["ppr"]["ids"], g["ppr"]["scores"], 2 * pdev + 1e-9)
            if not ok:
                problems.append(f"{query!r} ppr: {msg} (dev {pdev:.4f})")
        ok, msg = ranking_consistent(r["epi"]["texts"], r["epi"]["scores"], g["epi"]["texts"], g["epi"]["scores"], slack)
        if not ok:
            problems.append(f"{query!r} epi: {msg}")
        # what tri_retrieve hands to the memory pool (after the corpus-order re-sort): identical text lists
        for part in ("veridical", "episodic", "semantic") if "docs" in r else ():
            if sorted(r["docs"][part]) != sorted(g["docs"][part]):
                problems.append(f"{query!r}: {part} docs differ")
        checked += 1
    if ref.get("answers") != got.get("answers"):
        problems.append("final answers differ")
    return {"queries": checked, "max_score_dev": worst, "max_ppr_dev": worst_ppr, "problems": problems}


# ------------------------------------------------------------------------------------------------ replay
# The reference tree is not part of this repository.  tests/golden/make_golden_e2e_replay.py ran the loop above on the
# reference once and stored what its retrieval methods saw: every store's rows (texts, keys, the reference encoder's
# fp32 embeddings) and every probe string with its query row.  Replaying those probes reproduces the fact / passage /
# summary / timeline part of the committed trace without the reference.
REPLAY = os.path.join(ROOT, "tests", "golden", "e2e_cinderella_replay.npz")
STORE_NAMES = ("chunk", "entity", "fact", "summary", "timeline")
REPLAYED_KINDS = ("fact_scores", "fact_range", "ver", "sem", "epi")


def load_replay(path: str = REPLAY) -> Dict:
    with np.load(path) as z:
        rec = {k: z[k] for k in z.files}
    rec["epi_top_k"] = int(rec["epi_top_k"])
    return rec


def retrieval_view(run: Dict) -> Dict:
    """The stores and the REPLAYED_KINDS of every probe of a run (the part a replay can reproduce)."""
    return {"stores": run["stores"],
            "trace": {q: {k: v for k, v in t.items() if k in REPLAYED_KINDS} for q, t in run["trace"].items()}}


def _entry(rec, q, facts, ver, sem, epi) -> Dict:
    def rng(ns):
        raw = rec[ns + "_emb"] @ np.asarray(q, dtype=np.float32).reshape(-1)
        return float(raw.max() - raw.min())
    keys = {ns: rec[ns + "_keys"].tolist() for ns in ("fact", "chunk", "summary")}
    return {"fact_scores": dict(zip(keys["fact"], np.asarray(facts, dtype=np.float64).tolist())),
            "fact_range": rng("fact"),
            "ver": {"ids": [keys["chunk"][i] for i in np.asarray(ver[0]).tolist()],
                    "scores": np.asarray(ver[1], dtype=np.float64).tolist(), "range": rng("chunk")},
            "sem": {"ids": [keys["summary"][i] for i in np.asarray(sem[0]).tolist()],
                    "scores": np.asarray(sem[1], dtype=np.float64).tolist(), "range": rng("summary")},
            "epi": {"texts": [_h(t) for t in epi[0]], "scores": [float(s) for s in epi[1]], "range": rng("timeline")}}


def replay_reference(rec: Dict) -> Dict:
    """The reference's retrieval arithmetic (oracle/search_oracle.py restates it) on the recorded rows, on the CPU."""
    from oracle import search_oracle as so
    trace = {}
    for query, q in zip(rec["queries"].tolist(), rec["query_emb"]):
        q = q[None, :]
        ei, es = so.similar_summaries(rec["timeline_emb"], q, rec["epi_top_k"])
        trace[query] = _entry(rec, q, so.fact_scores(rec["fact_emb"], q), so.dense_passage_retrieval(rec["chunk_emb"], q),
                              so.dense_passage_retrieval(rec["summary_emb"], q),
                              ([rec["timeline_texts"][i] for i in ei.tolist()], es))
    return {"trace": trace, "stores": {ns: rec[ns + "_keys"].tolist() for ns in STORE_NAMES}}


class RecordedEncoder:
    """Hands out the reference encoder's recorded rows: store texts when called without an instruction (store
    inserts), probe rows when called with one (query encodes)."""
    instruction_is_forced = True
    global_config = None

    def __init__(self, rec: Dict):
        self.embedding_dim = int(rec["query_emb"].shape[1])
        self._texts = {str(t): e for ns in STORE_NAMES for t, e in zip(rec[ns + "_texts"], rec[ns + "_emb"])}
        self._queries = {str(t): e for t, e in zip(rec["queries"], rec["query_emb"])}

    def batch_encode(self, texts, **kw) -> np.ndarray:
        rows = self._queries if "instruction" in kw else self._texts
        texts = [texts] if isinstance(texts, str) else texts
        return np.stack([rows[t] for t in texts]).astype(np.float32)


def replay_engine(rec: Dict, arm: str, workdir: str) -> Dict:
    """The engine's side of the loop's retrieval, probe by probe, through the methods install() binds onto ComoRAG
    (comorag_b200.comorag_methods) in tri_retrieve's order, three probes in flight as the loop's question threads do.
    arm = "shim_search": the recorded reference rows go into engine stores (device search only);
    arm = "shim": the engine's bf16 encoder on the synthetic checkpoint encodes the store texts and the probes.
    Needs cuda:0.  Returns {"trace", "stores", "wave_stats", "query_encodes"}."""
    from concurrent.futures import ThreadPoolExecutor
    from comorag_b200 import comorag_methods as cm
    from comorag_b200.embedding_store import EmbeddingStore
    from comorag_b200.retrieval import get_similar_summaries

    cfg = types.SimpleNamespace(embedding_model_name=CKPT, embedding_batch_size=4, embedding_max_seq_len=512,
                                need_cluster=True, qa_epi_top_k=rec["epi_top_k"])
    if arm == "shim":
        from comorag_b200.embedding_model import BGEEmbeddingModel
        model = BGEEmbeddingModel(global_config=cfg, embedding_model_name=CKPT)
    elif arm == "shim_search":
        model = RecordedEncoder(rec)
    else:
        raise ValueError(arm)
    stores = {}
    for ns in STORE_NAMES:
        keys = rec[ns + "_keys"].tolist()
        store = EmbeddingStore(model, os.path.join(workdir, ns), 4, keys[0].rsplit("-", 1)[0])
        store.insert_strings([str(t) for t in rec[ns + "_texts"]])
        stores[ns] = store
    counters = {"encodes": 0, "encoded_texts": 0}
    lock = threading.Lock()
    orig_be = model.batch_encode

    def counting_batch_encode(texts, **kw):
        with lock:
            counters["encodes"] += 1
            counters["encoded_texts"] += 1 if isinstance(texts, str) else len(texts)
        return orig_be(texts, **kw)
    model.batch_encode = counting_batch_encode

    graph = _Graph()
    names = rec["entity_keys"].tolist() + rec["chunk_keys"].tolist()
    graph.add_vertices(len(names), attributes={"name": names})
    rag = types.SimpleNamespace(global_config=cfg, embedding_model=model, graph=graph, level_store=stores["timeline"],
                                ver_embedding_store=stores["chunk"], entity_embedding_store=stores["entity"],
                                fact_embedding_store=stores["fact"], sem_embedding_store=stores["summary"])
    cm.prepare_retrieval_objects(rag)

    def tri_retrieve(query):
        cm.get_query_embeddings(rag, query)
        facts = cm.get_fact_scores(rag, query)
        ver = cm.dense_passage_retrieval(rag, query)
        sem = cm.dense_passage_retrieval(rag, query, need_cluster=True)
        epi = get_similar_summaries(query=query, level_store=rag.level_store, embedding_model=model,
                                    top_k=rec["epi_top_k"])
        return facts, ver, sem, epi

    queries = rec["queries"].tolist()
    with ThreadPoolExecutor(max_workers=3) as ex:
        results = list(ex.map(tri_retrieve, queries))
    wave = getattr(rag, "_crag_wave", None)
    wave_stats = dict(wave.stats) if wave is not None else None
    if wave is not None:
        wave.close()
    trace = {q: _entry(rec, q_emb, *res) for q, q_emb, res in zip(queries, rec["query_emb"], results)}
    return {"trace": trace, "stores": {ns: s.get_all_ids() for ns, s in stores.items()}, "wave_stats": wave_stats,
            "query_encodes": counters}
