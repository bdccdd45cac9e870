#!/usr/bin/env python
"""bench.py -- the hot path of BASELINE.json on B200: brute-force IP top-10 over a 10M x 1024 bf16 index
(queries/sec) and BGE-large index-build encode (chunks/sec).

    python bench.py [--gpus N --steps K --warmup W]            # our arm, one JSON line on stdout
    python bench.py --impl reference [...]                     # the reference's CPU path, same metric
    torchrun --nproc-per-node N bench.py --gpus N ...          # N > 1: one rank per GPU (launched by the driver)

A "step" is one pass of the search hot path over one batch of 32 synthetic probe queries (config 5's probe
batch) against the whole index: N=1 holds all 10M rows on one GPU (20.5 GB bf16); at N>1 the SAME 10M rows are
row-sharded over the ranks ("strong" scaling: total work fixed).  A step is ONE CUDA-graph launch holding the shard
scan kernel and the fused finalize kernel -- at N>1 the finalize kernel also pushes the rank's top-k record into
every peer's buffer over NVLink and merges all ranks' records (crag_search_finalize_exchange), or, when symmetric
memory is unavailable, scan + finalize + one NCCL all-gather + merge kernel.
`value` = queries/sec with queries already in HBM; `e2e` = the same through the public host API
(ShardedIndex.search: pinned fp32 queries -> H2D -> search -> D2H of ids/scores/minmax, every step).
After the timed region the step's ids are checked against a float64 ranking of the same bf16 rows (`parity`); a
mismatch fails the run.  The `encode` object times the index-build encoder (BGE-large shape, random-init weights,
32 chunks x 512 tokens per rank per step; data-parallel, no collective) plus a mixed-length profile and the
tokenizer rate.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "queries/sec"
UNIT = "queries/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=10_000_000, help="total index rows (BASELINE: 10M)")
    ap.add_argument("--dim", type=int, default=1024)
    ap.add_argument("--nq", type=int, default=32, help="probe queries per step")
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--encode-chunks", type=int, default=32, help="chunks per encode step per rank")
    ap.add_argument("--encode-len", type=int, default=512)
    ap.add_argument("--encode-steps", type=int, default=5)
    ap.add_argument("--no-encode", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch the step's kernels one by one instead of one CUDA graph")
    ap.add_argument("--cpu-budget-s", type=float, default=20.0, help="CPU baseline sample budget (seconds of queries)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed search step returned (ids, scores, minmax) and the last timed "
                         "encode step's embeddings to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """DIR/<name>.npy in float32 / float64 (int64 ids as float64, exact below 2**53), so that two builds run with the
    same arguments -- hence the same seeded inputs -- can be compared output by output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32 if a.dtype == np.float32 else np.float64))


def workload_config(rows: int, dim: int, nq: int, k: int, world: int) -> dict:
    """The `config` object of BOTH arms' JSON lines: what is computed, nothing about how.  It depends on the command
    line and the GPU count only, so `bench.py` and `bench.py --impl reference` print the same object for the same
    flags (the driver compares them); what each arm's step consists of is said under `implementation` (ours) and
    `sample` (the reference arm's bounded sample of the step)."""
    base, rem = divmod(int(rows), int(world))        # comorag_b200.dist.shard_bounds: rank 0 owns base + (1 if rem) rows
    rows_rank0 = base + (1 if rem else 0)
    return {"workload": f"{rows}x{dim} bf16 index, brute-force IP top-{k}, {nq} probe queries per step, "
                        f"row-sharded over {world} GPU(s)",
            "index_rows": rows, "rows_per_rank": rows_rank0, "dim": dim, "queries_per_step": nq, "k": k,
            "l2": f"inputs larger than L2 ({rows_rank0 * dim * 2 / 1e9:.2f} GB shard per rank vs 126 MB)"}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def scan_traffic(rows: int, dim: int, nq: int, k: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of one scan launch from the committed `ncu --set full` capture
    (profiles/search_traffic.json), if one exists for exactly this shard shape; else None."""
    p = os.path.join(ROOT, "profiles", "search_traffic.json")
    if not os.path.exists(p):
        return None
    for e in json.load(open(p)):
        if (e["rows"], e["dim"], e["nq"], e["k"]) == (rows, dim, nq, k):
            return e["dram_bytes"]
    return None


# ------------------------------------------------------------------------------------------ clocks sampler
class ClockSampler:
    """nvidia-smi sampled every 100 ms while the timed region runs (B200_PROFILING.md recipe)."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1])); power.append(float(parts[2]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        load = [c for c in sm if c > 0.5 * (mx[0] if mx else 1)] or sm
        return {"sm_mhz": load[len(load) // 2] if load else None, "sm_max_mhz": mx[0] if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------ the reference's modules
def find_reference_root():
    """A ComoRAG checkout named by $COMORAG_REFERENCE, if any; without one the CPU arms time the oracle port."""
    cand = os.environ.get("COMORAG_REFERENCE")
    if cand and os.path.isdir(os.path.join(cand, "src", "comorag")):
        return cand
    return None


def import_reference():
    """The reference's own classes (CPU): ComoRAG (for its dense_passage_retrieval), BGEEmbeddingModel, EmbeddingStore.
    Two harness shims (SURVEY.md 8c): empty `igraph` / `umap` modules so the package imports, and `device_map` dropped
    from the HF init params (`accelerate` is absent).  Returns None when no reference tree is present."""
    root = find_reference_root()
    if root is None:
        return None
    import types
    sys.dont_write_bytecode = True
    if root not in sys.path:
        sys.path.insert(0, root)
    for m in ("igraph", "umap"):
        sys.modules.setdefault(m, types.ModuleType(m))
    try:
        from src.comorag.ComoRAG import ComoRAG
        from src.comorag.embedding_model.BGEEmbedding import BGEEmbeddingModel
        from src.comorag.embedding_store import EmbeddingStore
        from src.comorag.utils.config_utils import BaseConfig
    except Exception as e:   # a missing third-party module on this box: report, use the port
        sys.stderr.write(f"[bench] reference import failed ({e!r}); using the oracle port\n")
        return None

    class OracleBGE(BGEEmbeddingModel):
        def _init_embedding_config(self):
            super()._init_embedding_config()
            self.embedding_config.model_init_params.pop("device_map", None)

    return types.SimpleNamespace(root=root, ComoRAG=ComoRAG, OracleBGE=OracleBGE, EmbeddingStore=EmbeddingStore,
                                 BaseConfig=BaseConfig)


# ------------------------------------------------------------------------------------------ CPU search arm
class CpuSearch:
    """The reference's per-query CPU search -- dense_passage_retrieval, ComoRAG.py:950-967: np.dot(E, q.T) ->
    min_max_normalize -> np.argsort[::-1] over ALL rows -- on this host, one query at a time as the reference does,
    over an fp32 matrix of the FULL config shape.  Nothing is extrapolated: a timed query does the whole
    full_rows x dim arithmetic.  When the full matrix fits in RAM it is one [full_rows, dim] array and the reference's
    own method runs on it (kind "reference" if its modules import, else the oracle port); otherwise the matrix is
    streamed as `slabs` passes over one resident slab (distinct memory is not needed for the arithmetic) and the
    port evaluates the same expression slab by slab before the single min-max + argsort over all scores."""

    def __init__(self, full_rows: int, dim: int, ref=None):
        import numpy as np
        import torch
        try:
            import psutil
            free = psutil.virtual_memory().available
        except Exception:
            free = 32 << 30
        need = full_rows * dim * 4
        slab_rows = full_rows
        while slab_rows * dim * 4 * 1.6 > free * 0.7 and slab_rows > 100_000:
            slab_rows = (slab_rows + 1) // 2
        self.slabs = -(-full_rows // slab_rows)
        self.slab_rows, self.full_rows, self.dim = slab_rows, full_rows, dim
        t0 = time.time()
        self.mat = unit_rows_host(slab_rows, dim, seed=1234)
        self.q = torch.nn.functional.normalize(torch.randn(32, dim, generator=torch.Generator().manual_seed(4321)), dim=1).numpy()
        self.gen_s = time.time() - t0
        self.need_bytes = need
        self.kind = "port"
        self._ref_self = None
        if ref is not None and self.slabs == 1:
            import types
            self._ref_fn = ref.ComoRAG.dense_passage_retrieval       # the reference's own method, unbound
            self._ref_self = types.SimpleNamespace(query_to_embedding={"passage": {}}, passage_embeddings=self.mat,
                                                   embedding_model=None)
            self.kind = "reference"
        self.i = 0

    def one_query(self) -> float:
        import numpy as np
        from oracle import search_oracle
        q = self.q[self.i % 32: self.i % 32 + 1]
        self.i += 1
        t0 = time.perf_counter()
        if self._ref_self is not None:
            key = f"q{self.i}"
            self._ref_self.query_to_embedding["passage"][key] = q
            ids, sc = self._ref_fn(self._ref_self, key)
        elif self.slabs == 1:
            ids, sc = search_oracle.dense_passage_retrieval(self.mat, q)
        else:
            scores = np.empty(self.full_rows, dtype=np.float32)
            for s in range(self.slabs):
                r0 = s * self.slab_rows
                n = min(self.slab_rows, self.full_rows - r0)
                scores[r0:r0 + n] = np.squeeze(np.dot(self.mat[:n], q.T))
            scores = search_oracle.min_max_normalize(scores)
            ids = np.argsort(scores)[::-1]
            sc = scores[ids.tolist()]
        dt = time.perf_counter() - t0
        assert len(ids) == self.full_rows
        return dt

    def describe(self, times) -> dict:
        import numpy as np
        import torch
        try:
            from threadpoolctl import threadpool_info
            blas_threads = max([i.get("num_threads", 1) for i in threadpool_info() if i.get("user_api") == "blas"] or [1])
        except Exception:
            blas_threads = torch.get_num_threads()
        med = float(np.median(times))
        return {"value": 1.0 / med, "unit": UNIT, "cores": os.cpu_count(), "threads": blas_threads, "kind": self.kind,
                "extrapolated": False, "slabs": self.slabs,
                "per_query_s": {"min": float(min(times)), "median": med, "max": float(max(times))},
                "sample": f"{len(times)} single queries, each over the full fp32 [{self.full_rows}, {self.dim}] matrix"
                          + (f" streamed as {self.slabs} passes over a resident [{self.slab_rows}, {self.dim}] slab" if self.slabs > 1 else "")
                          + f" (np.dot + min-max + full argsort per query, {blas_threads} BLAS threads; matrix generation {self.gen_s:.0f} s not timed)"}


def unit_rows_host(rows: int, dim: int, seed: int):
    """Seeded N(0,1) rows, L2-normalised, fp32 [rows, dim] in host memory; generated (and first-touched) by a thread
    pool -- numpy's generators release the GIL -- because one thread takes minutes for the 41 GB of the 10M-row config."""
    import numpy as np
    from concurrent.futures import ThreadPoolExecutor
    out = np.empty((rows, dim), dtype=np.float32)
    n_threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    blk = max(4096, -(-rows // (4 * n_threads)))

    def fill(i):
        s0 = i * blk
        n = min(blk, rows - s0)
        x = np.random.default_rng(seed + i).standard_normal((n, dim), dtype=np.float32)
        x /= np.linalg.norm(x, axis=1, keepdims=True)
        out[s0:s0 + n] = x

    with ThreadPoolExecutor(max_workers=n_threads) as ex:
        list(ex.map(fill, range(-(-rows // blk))))
    return out


def cpu_search_baseline(full_rows: int, dim: int, budget_s: float, ref=None):
    cs = CpuSearch(full_rows, dim, ref)
    cs.one_query()   # warm
    times, t0 = [], time.time()
    while (time.time() - t0 < budget_s and len(times) < 32) or len(times) < 2:
        times.append(cs.one_query())
    return cs.describe(times)


# ------------------------------------------------------------------------------------------ CPU encode arm
def synthetic_vocab(size: int = 30522):
    specials = ["[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]"]
    return specials + [f"w{i}" for i in range(size - len(specials))]


def synthetic_texts(n: int, words: int, seed: int, vocab_size: int = 30522):
    import numpy as np
    rng = np.random.default_rng(seed)
    ids = rng.integers(0, vocab_size - 5, size=(n, words))
    return [" ".join(f"w{j}" for j in row) for row in ids]


def cpu_encode_baseline(ref, n_chunks: int, seq_len: int):
    """SURVEY.md 8d (i): the reference's index-build encode on the host cores.  With the reference's modules present:
    its own BGEEmbeddingModel (fp32 HF BertModel of the bge-large shape, random init) driven by its own
    EmbeddingStore.insert_strings on n_chunks synthetic ~seq_len-token chunks, embedding_batch_size 32.  Otherwise the
    port: one HF BertModel forward + the oracle's mean pooling + normalise."""
    import tempfile
    import torch
    from transformers import BertConfig, BertModel
    from comorag_b200.encoder import EncoderConfig
    cfg = EncoderConfig.bge_large()
    hf_cfg = BertConfig(hidden_size=cfg.hidden_size, num_hidden_layers=cfg.num_hidden_layers,
                        num_attention_heads=cfg.num_attention_heads, intermediate_size=cfg.intermediate_size,
                        vocab_size=cfg.vocab_size)
    if ref is not None:
        from transformers import BertTokenizerFast
        with tempfile.TemporaryDirectory() as tmp:
            ckpt = os.path.join(tmp, "bge-large-synth")     # "bge-" in the name selects BGEEmbeddingModel in the reference's factory
            os.makedirs(ckpt)
            torch.manual_seed(0)
            BertModel(hf_cfg).save_pretrained(ckpt, safe_serialization=True)
            vocab = synthetic_vocab(cfg.vocab_size)
            BertTokenizerFast(vocab={w: i for i, w in enumerate(vocab)}, do_lower_case=True).save_pretrained(ckpt)
            rcfg = ref.BaseConfig(embedding_model_name=ckpt, embedding_batch_size=32, embedding_max_seq_len=512)
            model = ref.OracleBGE(global_config=rcfg, embedding_model_name=ckpt)
            # the instruction prefix costs ~15 word pieces; seq_len - 24 words keep every chunk at <= 512 tokens
            texts = synthetic_texts(n_chunks + 2, max(seq_len - 24, 8), seed=7, vocab_size=cfg.vocab_size)
            store = ref.EmbeddingStore(model, os.path.join(tmp, "chunk_embeddings"), 32, "chunk")
            store.insert_strings(texts[:2])                   # warm (thread pools, allocator)
            t0 = time.perf_counter()
            store.insert_strings(texts[2:])
            dt = time.perf_counter() - t0
            assert len(store.get_all_ids()) == n_chunks + 2
        return {"value": n_chunks / dt, "unit": "chunks/s", "cores": os.cpu_count(), "threads": torch.get_num_threads(),
                "kind": "reference",
                "sample": f"the reference's EmbeddingStore.insert_strings -> BGEEmbeddingModel.batch_encode (fp32 HF BertModel, bge-large "
                          f"shape, random init) on {n_chunks} synthetic chunks of ~{seq_len} tokens, batch 32, incl. tokenizer + parquet write ({dt:.1f} s)"}
    from oracle.encoder_oracle import mean_pooling
    hf = BertModel(hf_cfg, add_pooling_layer=False).eval()
    ids = torch.randint(1000, cfg.vocab_size, (n_chunks, seq_len))
    mask = torch.ones_like(ids)
    with torch.no_grad():
        hf(input_ids=ids[:1, :64], attention_mask=mask[:1, :64])
        t0 = time.perf_counter()
        for s0 in range(0, n_chunks, 32):
            out = hf(input_ids=ids[s0:s0 + 32], attention_mask=mask[s0:s0 + 32]).last_hidden_state
            torch.nn.functional.normalize(mean_pooling(out, mask[s0:s0 + 32]), dim=1)
        dt = time.perf_counter() - t0
    return {"value": n_chunks / dt, "unit": "chunks/s", "cores": os.cpu_count(), "threads": torch.get_num_threads(),
            "kind": "port", "sample": f"HF BertModel fp32 forward + mean pool + normalise of {n_chunks} x {seq_len} tokens in batches of 32 ({dt:.1f} s)"}


# ------------------------------------------------------------------------------------------ reference arm
def run_reference(args):
    """--impl reference: the reference's own CPU path for the same metric and config.  A step is a bounded sample of
    the 32-query step: ONE query scored against the full 10M x 1024 fp32 matrix (the reference scores one query at a
    time anyway); `ms_per_step` is that measured time, `value` = 1 / it.  Nothing is extrapolated."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t_all = time.time()
    # torchrun exports OMP_NUM_THREADS=1; the reference arm is meant to use every host thread it can.  numpy / torch
    # have not been imported yet in this process, so the BLAS pools still honour the environment.
    n_threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[var] = str(n_threads)
    ref = import_reference()
    cs = CpuSearch(args.rows, args.dim, ref)
    for _ in range(max(args.warmup, 1)):
        cs.one_query()
    t0 = time.perf_counter()
    times = [cs.one_query() for _ in range(args.steps)]
    wall = time.perf_counter() - t0
    base = cs.describe(times)
    ms_per_step = wall / args.steps * 1e3
    value = 1e3 / ms_per_step
    base["value"] = value
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": max(args.warmup, 1), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.rows, args.dim, args.nq, args.k, max(int(args.gpus), 1)),
            "sample": f"the reference's CPU path (ComoRAG.dense_passage_retrieval: per-query np.dot + min-max + full argsort over all "
                      f"{args.rows} fp32 rows, host memory, no sharding); a timed step = 1 query, a bounded sample of the "
                      f"{args.nq}-query step (the reference scores one query at a time anyway); value = queries/s, not extrapolated",
            "queries_per_timed_step": 1,
            "cpu_baseline": base,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.time() - t_all}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ our arm
def make_shard(rows: int, dim: int, seed: int, device):
    """Seeded unit-norm rows rounded to bf16, generated on the device in slabs (SURVEY.md 8d)."""
    import torch
    out = torch.empty((rows, dim), dtype=torch.bfloat16, device=device)
    g = torch.Generator(device=device).manual_seed(seed)
    slab = 1 << 19
    for s in range(0, rows, slab):
        n = min(slab, rows - s)
        x = torch.randn((n, dim), generator=g, device=device, dtype=torch.float32)
        out[s:s + n] = torch.nn.functional.normalize(x, dim=1).to(torch.bfloat16)
    return out


def reference_topk_f64(corpus, queries, kk: int, row_offset: int, chunk: int = 1 << 18):
    """float64 ranking of this rank's bf16 rows on the device (checker, not product): the kk best (score desc, id asc)
    per query as (global ids int64 [nq, kk], scores float64 [nq, kk])."""
    import torch
    nq, dev = queries.shape[0], corpus.device
    q = queries.double()
    best_s = torch.empty((nq, 0), dtype=torch.float64, device=dev)
    best_i = torch.empty((nq, 0), dtype=torch.int64, device=dev)
    for s0 in range(0, corpus.shape[0], chunk):
        blk = corpus[s0:s0 + chunk].double()
        sc = q @ blk.T
        ids = torch.arange(s0, s0 + blk.shape[0], device=dev, dtype=torch.int64).expand(nq, -1) + row_offset
        cs, ci = torch.cat([best_s, sc], 1), torch.cat([best_i, ids], 1)
        o1 = torch.argsort(ci, dim=1, stable=True)
        cs, ci = torch.gather(cs, 1, o1), torch.gather(ci, 1, o1)
        o2 = torch.argsort(cs, dim=1, descending=True, stable=True)[:, :kk]
        best_s, best_i = torch.gather(cs, 1, o2), torch.gather(ci, 1, o2)
    pad = kk - best_s.shape[1]
    if pad > 0:
        best_s = torch.cat([best_s, torch.full((nq, pad), float("-inf"), dtype=torch.float64, device=dev)], 1)
        best_i = torch.cat([best_i, torch.full((nq, pad), -1, dtype=torch.int64, device=dev)], 1)
    return best_i, best_s


def count_id_mismatches(got_ids, want_ids, want_scores, k: int, tie: float = 2e-6) -> int:
    """got_ids [nq, k] vs the float64 ranking want_* [nq, kk > k].  Ranks whose float64 scores are closer than `tie`
    (indistinguishable under any fp32 summation order) are compared as sets; a group reaching past rank k accepts
    any of its members."""
    import numpy as np
    bad = 0
    for q in range(got_ids.shape[0]):
        j = 0
        while j < k:
            e = j
            while e + 1 < want_ids.shape[1] and want_scores[q, e] - want_scores[q, e + 1] < tie:
                e += 1
            group = set(want_ids[q, j:e + 1].tolist())
            hi = min(e, k - 1)
            got = got_ids[q, j:hi + 1].tolist()
            if e < k:
                bad += 0 if set(got) == group else len(group ^ set(got)) // 2 or 1
            else:
                bad += sum(1 for g in got if g not in group)
            j = hi + 1
    return int(bad)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from comorag_b200 import _native
    from comorag_b200.dist import ShardedIndex, shard_bounds
    from comorag_b200.index import DenseIndex

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (ours) needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # keep stdout to the single JSON line: NCCL's banner / debug output goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    lib = _native.load()
    peaks = load_peaks()
    use_graph = not args.no_graph

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- index: the same 10M rows at every N, row-sharded (strong scaling)
    offs = shard_bounds(args.rows, world)
    my_rows = offs[rank + 1] - offs[rank]
    corpus = make_shard(my_rows, args.dim, 1234 + rank, dev)
    index = ShardedIndex(DenseIndex.from_tensor(corpus, row_offset=offs[rank]))
    gq = torch.Generator().manual_seed(4321)
    q_host = torch.nn.functional.normalize(torch.randn(args.nq, args.dim, generator=gq), dim=1).pin_memory()
    q_dev = q_host.to(dev).to(torch.bfloat16).contiguous()
    st = torch.cuda.current_stream(dev)
    session = index.session(args.nq, args.k, use_graph) if world > 1 else index.local.session(args.nq, args.k, use_graph)
    session.queries.copy_(q_dev)

    def step_device():
        return session.run(session.queries)

    def step_e2e():
        # the public host entry point: pinned fp32 queries -> H2D -> bf16 -> search -> D2H of (ids, scores, minmax)
        if world > 1:
            return index.search(q_host, args.k)
        q = index.local.prepare_queries(q_host)
        session.run(q)
        return session.record.cpu()   # ids | scores | minmax in one packed D2H; .cpu() synchronises

    for _ in range(max(args.warmup, 3)):
        step_device()
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(st)
    for _ in range(args.steps):
        step_device()
    e1.record(st)
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    ms_per_step = ms_total / args.steps
    value = args.nq / ms_per_step * 1e3
    got_ids = session.ids.clone()
    got_scores = session.scores.clone()
    got_minmax = session.minmax.clone() if args.dump_outputs else None
    if index.peer is not None:
        index.peer.check()

    # ---- parity of the timed step's answer: float64 ranking of the same bf16 rows, merged over ranks by (score, id)
    kk = args.k + 8
    loc_i, loc_s = reference_topk_f64(corpus, q_dev, kk, offs[rank])
    if world > 1:
        all_i = [torch.empty_like(loc_i) for _ in range(world)]
        all_s = [torch.empty_like(loc_s) for _ in range(world)]
        dist.all_gather(all_i, loc_i)
        dist.all_gather(all_s, loc_s)
        ci, cs = torch.cat(all_i, 1), torch.cat(all_s, 1)
        o1 = torch.argsort(ci, dim=1, stable=True)
        cs, ci = torch.gather(cs, 1, o1), torch.gather(ci, 1, o1)
        o2 = torch.argsort(cs, dim=1, descending=True, stable=True)[:, :kk]
        loc_s, loc_i = torch.gather(cs, 1, o2), torch.gather(ci, 1, o2)
    mism = count_id_mismatches(got_ids.cpu().numpy(), loc_i.cpu().numpy(), loc_s.cpu().numpy(), args.k)
    score_err = float((got_scores.double() - loc_s[:, :args.k]).abs().max().item())
    mism = int(max_over_ranks(float(mism)))
    parity = {"checked": True, "queries": args.nq, "k": args.k, "mismatches": mism, "max_score_err": score_err,
              "against": "float64 ranking of the same bf16 rows on the device, merged over ranks by (score desc, id asc); "
                         "ranks closer than 2e-6 compared as sets"}

    # ---- roofline of the dominant kernel: the shard scan, timed in the SAME loop as a full step (alternating), with
    # CUDA events on its stream
    ws_bytes = lib.crag_search_workspace_bytes(args.nq, args.k)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    scan_ms, step_ms = [], []
    for i in range(args.steps + 3):
        a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        a.record(st)
        step_device()
        b.record(st)
        rc = lib.crag_search_scan(corpus.data_ptr(), my_rows, args.dim, corpus.stride(0), q_dev.data_ptr(), args.nq, args.k,
                                  ws.data_ptr(), ws_bytes, st.cuda_stream)
        c.record(st)
        _native.check(rc, "crag_search_scan")
        torch.cuda.synchronize()
        if i >= 3:
            step_ms.append(a.elapsed_time(b))
            scan_ms.append(b.elapsed_time(c))
    scan_avg = sum(scan_ms) / len(scan_ms)
    algo_bytes = float(my_rows) * args.dim * 2
    achieved = algo_bytes / scan_avg / 1e6  # GB/s

    # ---- e2e through the host API
    for _ in range(3):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_value = args.nq * args.steps / e2e_s
    h2d = args.nq * args.dim * 4
    d2h = args.nq * args.k * (8 + 4) + args.nq * 2 * 4

    # ---- SURVEY.md 8d's second data set (one GPU only: no collectives inside a try block): planted neighbours
    # x_j = normalise(q + 0.3 * noise) with |noise| = 1 (cosine to the query ~ 0.96, far above the ~0.16 of the best
    # random row), 64 rows per query, written over the LAST tiles of the shard -- a corpus whose best rows all sit at
    # the end of the row order.  Same session, same graph: timing + float64 parity again.
    planted = None
    if world == 1 and my_rows >= 1_000_000:
        try:
            gp = torch.Generator(device=dev).manual_seed(777)
            per = 64
            tail = q_dev.float().repeat_interleave(per, dim=0) + (0.3 / args.dim ** 0.5) * torch.randn((args.nq * per, args.dim), generator=gp, device=dev)
            corpus[my_rows - tail.shape[0]:] = torch.nn.functional.normalize(tail, dim=1).to(torch.bfloat16)
            for _ in range(3):
                step_device()
            pa, pb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            pa.record(st)
            for _ in range(args.steps):
                step_device()
            pb.record(st)
            torch.cuda.synchronize()
            p_ms = pa.elapsed_time(pb) / args.steps
            p_ids = session.ids.clone()
            w_i, w_s = reference_topk_f64(corpus, q_dev, kk, offs[rank])
            p_mism = count_id_mismatches(p_ids.cpu().numpy(), w_i.cpu().numpy(), w_s.cpu().numpy(), args.k)
            in_tail = float((p_ids >= offs[rank] + my_rows - tail.shape[0]).float().mean().item())
            planted = {"what": f"{per} planted neighbours per query (normalise(q + 0.3 unit noise), cosine ~0.96) in the last {tail.shape[0]} rows of the shard",
                       "ms_per_step": p_ms, "vs_random_corpus": p_ms / ms_per_step, "mismatches": int(p_mism),
                       "fraction_of_topk_in_planted_rows": in_tail}
        except Exception as e:   # reported, never fatal: the headline numbers above are already measured
            planted = {"error": repr(e)[:300]}

    # ---- encode (index build): data-parallel, every rank encodes its own batch
    encode = None
    if not args.no_encode:
        encode, enc_out = bench_encode(args, world, rank, dev, st, peaks, barrier, max_over_ranks)

    # the sampler has been running through every GPU-timed phase above (search value, scan roofline, e2e, encode)
    clocks = sampler.stop() if rank == 0 else None
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ref = import_reference()
        cpu = cpu_search_baseline(args.rows, args.dim, args.cpu_budget_s, ref)
        if encode is not None:
            try:
                encode["cpu_baseline"] = cpu_encode_baseline(ref, 64, args.encode_len)
            except Exception as e:  # transformers missing etc.: report, do not fake
                encode["cpu_baseline"] = {"unavailable": repr(e)[:300]}

    if rank == 0 and args.dump_outputs:
        outputs = {"search_ids": got_ids.cpu().numpy(), "search_scores": got_scores.float().cpu().numpy(),
                   "search_minmax": got_minmax.float().cpu().numpy()}
        if encode is not None:
            outputs["encode_embeddings"] = enc_out.cpu().numpy()
        dump_outputs(args.dump_outputs, outputs)

    if rank == 0:
        if world == 1 or index.exchange_mode == "peer":
            kernels = ["search_topk_kernel", "merge_topk_kernel" if world == 1 else "finalize_exchange_kernel"]
        else:
            kernels = ["search_topk_kernel", "merge_topk_kernel", "ncclAllGather (library)", "merge_topk_kernel"]
            use_graph = False
        ours_per_step = sum(1 for kname in kernels if "library" not in kname)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": workload_config(args.rows, args.dim, args.nq, args.k, world),
            "implementation": {"step": ("one CUDA graph: " if use_graph else "") + " + ".join(kernels),
                               "exchange": index.exchange_mode},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": args.steps * ours_per_step,
            "parity": parity,
            "planted_neighbours": planted,
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": achieved / peaks["hbm_gbs"], "traffic": scan_traffic(my_rows, args.dim, args.nq, args.k),
                         "peak_source": peaks["source"],
                         "kernel": "search_topk_kernel", "algorithmic_bytes_per_launch": algo_bytes,
                         "kernel_ms": scan_avg, "step_ms_same_loop": sum(step_ms) / len(step_ms)},
            "cpu_baseline": cpu,
            "encode": encode,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        del session
        index.close()
        torch.cuda.synchronize()
        dist.destroy_process_group()
    if mism != 0:
        raise SystemExit(f"bench.py: {mism} id mismatches against the float64 ranking -- the timed path returned wrong ids")


def bench_encode(args, world, rank, dev, st, peaks, barrier, max_over_ranks):
    import numpy as np
    import torch
    from comorag_b200.encoder import BertEncoderB200, EncoderConfig
    from comorag_b200.index import DenseIndex
    cfg = EncoderConfig.bge_large()
    enc = BertEncoderB200.random_init(cfg, seed=0, device=dev)
    n, L = args.encode_chunks, args.encode_len
    gi = torch.Generator().manual_seed(99 + rank)
    ids_host = torch.randint(1000, cfg.vocab_size, (n * L,), generator=gi, dtype=torch.int32).pin_memory()
    cu_host = (torch.arange(n + 1, dtype=torch.int32) * L).pin_memory()
    ids_dev, cu_dev = ids_host.to(dev), cu_host.to(dev)
    out = torch.empty((n, cfg.hidden_size), dtype=torch.float32, device=dev)
    for _ in range(3):
        enc.forward_packed(ids_dev, cu_dev, L, out_f32=out)
    barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for _ in range(args.encode_steps):
        enc.forward_packed(ids_dev, cu_dev, L, out_f32=out)
    b.record(st)
    barrier()
    out_last = out.clone()      # the last timed encode step's embeddings (later phases reuse `out`)
    enc_ms = max_over_ranks(a.elapsed_time(b)) / args.encode_steps
    chunks_s = world * n / enc_ms * 1e3
    flops = cfg.flops_per_chunk(L) * n
    enc_tflops = flops / enc_ms / 1e9

    # e2e index build: token ids from pinned host memory, K3 writes the bf16 rows straight into the corpus shard,
    # the fp32 rows (what EmbeddingStore keeps / writes to parquet) come back to the host
    shard = DenseIndex(cfg.hidden_size, device=dev, capacity=n * (args.encode_steps + 1))
    shard_rows = shard._buf
    barrier()
    t0 = time.perf_counter()
    for s in range(args.encode_steps):
        rows = shard_rows[s * n:(s + 1) * n]
        enc.forward_packed(ids_host.to(dev, non_blocking=True), cu_host.to(dev, non_blocking=True), L, out_f32=out, out_bf16=rows)
        out.cpu()
    e2e_enc_s = max_over_ranks(time.perf_counter() - t0)
    assert float(shard_rows[: n * args.encode_steps].float().norm(dim=1).min()) > 0.99   # the shard rows were written

    # mixed-length profile L ~ U[32, 512] (SURVEY.md 8d): the varlen packing has no padding waste to hide
    rng = np.random.default_rng(5 + rank)
    lens = rng.integers(32, L + 1, size=2 * n)
    cu_m = torch.from_numpy(np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)).to(dev)
    ids_m = torch.randint(1000, cfg.vocab_size, (int(lens.sum()),), generator=gi, dtype=torch.int32).to(dev)
    out_m = torch.empty((2 * n, cfg.hidden_size), dtype=torch.float32, device=dev)
    for _ in range(2):
        enc.forward_packed(ids_m, cu_m, int(lens.max()), out_f32=out_m)
    barrier()
    a2, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a2.record(st)
    for _ in range(args.encode_steps):
        enc.forward_packed(ids_m, cu_m, int(lens.max()), out_f32=out_m)
    b2.record(st)
    barrier()
    mix_ms = max_over_ranks(a2.elapsed_time(b2)) / args.encode_steps
    mix_flops = float(sum(cfg.flops_per_chunk(int(x)) for x in lens))
    mixed = {"chunks": int(2 * n), "tokens": int(lens.sum()), "length_profile": f"U[32, {L}]", "ms_per_step": mix_ms,
             "chunks_per_s": world * 2 * n / mix_ms * 1e3, "tokens_per_s": world * float(lens.sum()) / mix_ms * 1e3,
             "tflops": mix_flops / mix_ms / 1e9, "frac_of_sustained_peak": mix_flops / mix_ms / 1e9 / peaks["bf16_tflops_sustained"]}

    # short probe batch (ComoRAG's query pattern): 32 probes x ~24 tokens through the CUDA-graph path
    probes = [[101] + rng.integers(1000, cfg.vocab_size, size=22).tolist() + [102] for _ in range(32)]
    for _ in range(3):
        enc.encode_token_lists(probes)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(20):
        enc.encode_token_lists(probes)
    torch.cuda.synchronize()
    probe_ms = (time.perf_counter() - t0) / 20 * 1e3

    # tokenizer rate (host, HF fast tokenizer over a synthetic 30522-word vocabulary): reported, not part of chunks/s
    tok = None
    if rank == 0:
        try:
            from transformers import BertTokenizerFast
            tk = BertTokenizerFast(vocab={w: i for i, w in enumerate(synthetic_vocab(cfg.vocab_size))}, do_lower_case=True)
            texts = synthetic_texts(256, L - 2, seed=3, vocab_size=cfg.vocab_size)
            tk(texts[:8], truncation=True, max_length=L)
            t0 = time.perf_counter()
            enc_ids = tk(texts, truncation=True, max_length=L)["input_ids"]
            dt = time.perf_counter() - t0
            tok = {"chunks_per_s": len(texts) / dt, "tokens_per_s": sum(len(x) for x in enc_ids) / dt,
                   "what": "transformers BertTokenizerFast (Rust), one batched call over 256 synthetic 512-token chunks, host threads as configured"}
        except Exception as e:
            tok = {"unavailable": repr(e)[:200]}
    launches_per_fwd = 2 + cfg.num_hidden_layers * 7
    del enc
    return {"metric": "encode chunks/sec", "value": chunks_s, "unit": "chunks/s", "ms_per_step": enc_ms,
            "config": {"workload": f"bge-large-en-v1.5 shape (1024-d, 24 layers), {n} chunks x {L} tokens per rank per step, random-init bf16 weights",
                       "scaling": "weak (data-parallel, no collective)"},
            "dtype": "bf16",
            "e2e": {"value": world * n * args.encode_steps / e2e_enc_s, "unit": "chunks/s",
                    "h2d_bytes_per_step": n * L * 4 + (n + 1) * 4, "d2h_bytes_per_step": n * cfg.hidden_size * 4,
                    "what": "pinned token ids -> H2D -> forward -> bf16 rows written into the corpus shard by the pooling kernel + fp32 rows D2H"},
            "roofline": {"bound": "tensor", "achieved": enc_tflops, "peak": peaks["bf16_tflops_sustained"],
                         "unit": "TFLOP/s", "frac": enc_tflops / peaks["bf16_tflops_sustained"], "traffic": None,
                         "peak_source": peaks["source"] + " (sustained)", "flops_per_chunk": cfg.flops_per_chunk(L)},
            "mixed_length": mixed,
            "probe_batch": {"probes": 32, "tokens_each": 24, "ms": probe_ms, "probes_per_s": 32 / probe_ms * 1e3,
                            "what": "encode_token_lists through the captured CUDA graph (768-token bucket), host call to result on device"},
            "tokenizer": tok,
            "gpu_launches": args.encode_steps * launches_per_fwd}, out_last


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
