"""comorag_b200.install rebinds the hot-path names inside a ComoRAG package.  The package here is a stand-in written by
the test: the module layout and the `from ... import` bindings of the reference's src/comorag that install() relies
on (ComoRAG.py:21-35, utils/timeline_utils.py), with empty bodies."""
import sys

STANDIN = {
    "__init__.py": "from .ComoRAG import ComoRAG\n",
    "embedding_model/__init__.py": (
        "from .BGEEmbedding import BGEEmbeddingModel\n"
        "def _get_embedding_model_class(embedding_model_name):\n"
        "    return BGEEmbeddingModel\n"),
    "embedding_model/BGEEmbedding.py": "class BGEEmbeddingModel:\n    pass\n",
    "embedding_store.py": "class EmbeddingStore:\n    pass\n",
    "rerank.py": "class DSPyFilter:\n    pass\n",
    "utils/__init__.py": "",
    "utils/embed_utils.py": (
        "def retrieve_knn(*a, **kw):\n    pass\n"
        "def get_similar_summaries(*a, **kw):\n    pass\n"),
    "utils/timeline_utils.py": "from ..embedding_store import EmbeddingStore\n",
    "ComoRAG.py": (
        "from .embedding_model import _get_embedding_model_class\n"
        "from .embedding_store import EmbeddingStore\n"
        "from .rerank import DSPyFilter\n"
        "from .utils.embed_utils import retrieve_knn, get_similar_summaries\n"
        "from .utils import timeline_utils\n"
        "class ComoRAG:\n"
        "    def prepare_retrieval_objects(self): pass\n"
        "    def get_query_embeddings(self, queries): pass\n"
        "    def get_fact_scores(self, query): pass\n"
        "    def dense_passage_retrieval(self, query, need_cluster=False): pass\n"),
}


def test_install_rebinds_names_package_wide(tmp_path, monkeypatch):
    pkg = "comorag_standin"
    for rel, text in STANDIN.items():
        path = tmp_path / pkg / rel
        path.parent.mkdir(parents=True, exist_ok=True)
        path.write_text(text)
    monkeypatch.syspath_prepend(str(tmp_path))
    monkeypatch.setattr(sys, "dont_write_bytecode", True)
    try:
        __import__(pkg)  # its __init__ imports ComoRAG.py, which binds the names with `from ... import`
        ref_main = sys.modules[pkg + ".ComoRAG"]   # the package attribute of that name is the class, not the module

        import comorag_b200.install as crag
        from comorag_b200 import comorag_methods as cm
        from comorag_b200.embedding_model import BGEEmbeddingModel, _get_embedding_model_class
        from comorag_b200.embedding_store import EmbeddingStore
        from comorag_b200.retrieval import get_similar_summaries, retrieve_knn
        counts = crag.install(pkg)
        assert counts["EmbeddingStore"] >= 3 and counts["_get_embedding_model_class"] >= 2
        assert ref_main.EmbeddingStore is EmbeddingStore
        assert ref_main._get_embedding_model_class is _get_embedding_model_class
        assert ref_main.get_similar_summaries is get_similar_summaries
        assert ref_main.retrieve_knn is retrieve_knn
        tl = sys.modules[pkg + ".utils.timeline_utils"]
        assert tl.EmbeddingStore is EmbeddingStore
        assert ref_main._get_embedding_model_class("BAAI/bge-large-en-v1.5") is BGEEmbeddingModel
        for name, fn in cm.METHODS.items():
            assert ref_main.ComoRAG.__dict__[name] is fn
        assert ref_main.DSPyFilter.__module__.startswith(pkg)      # LLM filter untouched unless rerank=True
        crag.install(pkg, rerank=True)
        assert ref_main.DSPyFilter.__module__ == "comorag_b200.rerank"
        crag.uninstall_search(pkg)
        assert ref_main.ComoRAG.get_fact_scores.__module__ == pkg + ".ComoRAG"
    finally:
        for name in [m for m in sys.modules if m == pkg or m.startswith(pkg + ".")]:
            del sys.modules[name]
