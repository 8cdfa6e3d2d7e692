"""The reference's OWN acceptance harness (bench/bench.py, unmodified, SURVEY §2 item 19) driven on top of the
ssd_b200 host engine through the `ssd` compat shim — on CPU, with the device runner replaced by a deterministic test
double.  The calls that harness makes into the engine (the model and the kwargs of `create_llm_kwargs`, the
`llm.config.max_num_seqs` / `llm.scheduler.max_num_seqs` pokes of its sweep path, the METRICS reset, the prompts and
SamplingParams handed to `generate()`) were recorded from a run of the unmodified harness into
tests/golden/reference_bench_calls.json (oracle/gen_harness_golden.py); the tests replay them through `import ssd.paths`,
`from ssd import LLM, SamplingParams`, `from ssd.engine.llm_engine import METRICS`, and check `generate()`'s return
value and the scheduler / block-manager bookkeeping under random accept lengths."""
import importlib
import json
import os
import sys
import types

import numpy as np

CALLS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_bench_calls.json")

V = 128256


def _next(tok: int) -> int:
    """The fake target model: a fixed permutation-like map; greedy decoding follows it exactly."""
    return (tok * 31 + 7) % V


class FakeRunner:
    """Stands in for PairRunner: the target's greedy next token is _next(last); the draft agrees most of the time."""

    def __init__(self, K):
        self.K = K
        self.rng = np.random.default_rng(0)
        self.calls = {"prefill": 0, "spec_step": 0, "decode": 0}
        self.max_batch_seen = 0

    def prefill(self, which, tokens, block_table, start=0, temp=0.0, want_sample=True, chunk=64, seed=0):
        self.calls["prefill"] += 1
        assert len(block_table) * 256 >= len(tokens), "prefill without enough KV blocks"
        return _next(tokens[-1]) if want_sample else None

    def prefill_many(self, which, tokens, block_tables, starts, temps=None, want_sample=True, chunk=256, seed=0):
        out = [self.prefill(which, t, bt, start=s, want_sample=want_sample) for t, bt, s in zip(tokens, block_tables, starts)]
        return out if want_sample else None

    def forward_tokens(self, which, ids, ctx_len, block_tables, temps=None, want_sample=True, seed=0):
        self.calls["decode"] += 1
        return [_next(x[-1]) for x in ids]

    def spec_step(self, ctx_len, recovery, bt_target, bt_draft, temps_t, temps_q, seed=0):
        self.calls["spec_step"] += 1
        B, K = len(ctx_len), self.K
        self.max_batch_seen = max(self.max_batch_seen, B)
        toks = np.zeros((B, K + 1), dtype=np.int64)
        nacc = np.zeros(B, dtype=np.int32)
        rec = np.zeros(B, dtype=np.int64)
        for b in range(B):
            for t in (bt_target[b], bt_draft[b]):
                assert len(t) * 256 >= ctx_len[b] + K + 1, "look-ahead KV slots were not reserved"
            n = int(self.rng.integers(0, K + 1))
            cur = recovery[b]
            toks[b, 0] = cur
            for j in range(K):
                cur = _next(cur) if j < n else (_next(cur) + 1) % V  # first wrong token at position n
                toks[b, j + 1] = cur
            nacc[b] = n
            last = toks[b, n]
            rec[b] = _next(int(last))
        return toks, nacc, rec

    def close(self):
        pass


def _make_hf_cache(root):
    from ssd_b200 import synth
    for repo, shape, role in (("models--meta-llama--Llama-3.1-8B-Instruct", "llama-3.1-8b", "target"),
                              ("models--meta-llama--Llama-3.2-1B-Instruct", "llama-3.2-1b", "draft")):
        snap = os.path.join(root, repo, "snapshots")
        os.makedirs(snap, exist_ok=True)
        made = synth.make_model_dir(snap, shape, role)
        os.rename(made, os.path.join(snap, "synthetic"))


def engine_env(tmp_path, monkeypatch):
    """SSD_HF_CACHE with the synthetic Llama 8B / 1B pair, the `ssd` compat shim, a wandb stub and FakeRunner in place
    of the device runner.  Returns {"runner", "config"}, filled when the engine is built."""
    monkeypatch.setenv("SSD_HF_CACHE", str(tmp_path))
    monkeypatch.setenv("SSD_DATASET_DIR", str(tmp_path / "datasets"))
    _make_hf_cache(str(tmp_path))
    import ssd_b200.paths as P
    importlib.reload(P)
    import ssd_b200.compat as compat
    compat.install()
    wandb = types.ModuleType("wandb")
    wandb.init = wandb.log = wandb.finish = lambda *a, **k: None
    monkeypatch.setitem(sys.modules, "wandb", wandb)
    fake = {}

    def fake_build_runner(config, tp_size=1, tp_rank=0, device=None, finalize=True):
        config.num_kvcache_blocks = 256
        fake["runner"] = FakeRunner(config.speculate_k)
        fake["config"] = config
        return fake["runner"], types.SimpleNamespace(num_kvcache_blocks=256)

    import ssd_b200.loader as loader
    monkeypatch.setattr(loader, "build_runner", fake_build_runner)
    return fake


def spy_engine(monkeypatch, cache_dir):
    """Records every LLMEngine construction and generate() call: the calls as made (paths relative to `cache_dir`), and
    what generate() returned."""
    import dataclasses

    import ssd_b200.engine.llm_engine as eng
    calls, captured = {"runs": []}, {"runs": []}
    orig_init, orig_generate = eng.LLMEngine.__init__, eng.LLMEngine.generate
    rel = lambda p: os.path.relpath(p, cache_dir) if isinstance(p, str) and p.startswith(str(cache_dir)) else p

    def spy_init(self, model, **kwargs):
        calls["model"], calls["llm_kwargs"] = rel(model), {k: rel(v) for k, v in kwargs.items()}
        orig_init(self, model, **kwargs)

    def spy_generate(self, prompts, sampling_params, use_tqdm=True, stream_callback=None):
        calls["runs"].append({"config_max_num_seqs": self.config.max_num_seqs,
                              "scheduler_max_num_seqs": self.scheduler.max_num_seqs, "prompts": [list(p) for p in prompts],
                              "sampling_params": [dataclasses.asdict(sp) for sp in sampling_params]})
        outs, metrics = orig_generate(self, prompts, sampling_params, use_tqdm=False, stream_callback=stream_callback)
        captured["runs"].append((prompts, outs, {k: (list(v) if isinstance(v, list) else v) for k, v in metrics.items()}))
        return outs, metrics

    monkeypatch.setattr(eng.LLMEngine, "__init__", spy_init)
    monkeypatch.setattr(eng.LLMEngine, "generate", spy_generate)
    return calls, captured


def _run_bench(tmp_path, monkeypatch, name):
    """Replay the recorded calls of the reference harness run `name` in the order it made them."""
    with open(CALLS) as f:
        rec = json.load(f)[name]
    fake = engine_env(tmp_path, monkeypatch)
    _, captured = spy_engine(monkeypatch, tmp_path)
    import ssd.paths  # noqa: F401
    from ssd import LLM, SamplingParams
    from ssd.engine.llm_engine import METRICS
    path = lambda p: os.path.join(ssd.paths.HF_CACHE_DIR, p) if p else p
    llm = LLM(path(rec["model"]), **{**rec["llm_kwargs"], "draft": path(rec["llm_kwargs"]["draft"])})
    for run in rec["runs"]:
        llm.config.max_num_seqs = run["config_max_num_seqs"]
        llm.scheduler.max_num_seqs = run["scheduler_max_num_seqs"]
        for k, v in METRICS.items():
            if isinstance(v, list):
                v.clear()
            else:
                METRICS[k] = 0
        llm.generate(run["prompts"], [SamplingParams(**sp) for sp in run["sampling_params"]])
    return captured, fake


def test_reference_bench_py_runs_unmodified_on_the_engine(tmp_path, monkeypatch):
    captured, fake = _run_bench(tmp_path, monkeypatch, "spec")
    cfg = fake["config"]
    assert cfg.speculate and cfg.speculate_k == 6 and cfg.jit_speculate and cfg.kvcache_block_size == 256
    assert cfg.max_num_seqs == 2 and cfg.max_model_len == 8192
    (prompts, outs, metrics), = captured["runs"]
    assert len(outs) == 5
    for p, o in zip(prompts, outs):
        want, cur = [], p[-1]
        for _ in range(60):
            cur = _next(cur)
            want.append(cur)
        assert o["token_ids"] == want, "speculative bookkeeping changed the greedy continuation"
    lens = metrics["accepted_suffix_lens_with_recovery"]
    assert lens and all(1 <= x <= 7 for x in lens)
    assert metrics["decode_total_tokens"] == sum(lens) and metrics["prefill_total_tokens"] == 5 * 40
    r = fake["runner"]
    assert r.max_batch_seen == 2 and r.calls["prefill"] == 2 * 5          # target + draft prefill per sequence
    assert r.calls["spec_step"] <= len(lens) <= 2 * r.calls["spec_step"]  # one suffix per running sequence per step


def test_reference_bench_py_sweep_and_autoregressive(tmp_path, monkeypatch):
    captured, fake = _run_bench(tmp_path, monkeypatch, "sweep")
    assert not fake["config"].speculate
    assert len(captured["runs"]) == 2
    for prompts, outs, metrics in captured["runs"]:
        assert [len(o["token_ids"]) for o in outs] == [20, 20, 20]
        assert metrics["decode_total_tokens"] > 0 and not metrics["accepted_suffix_lens_with_recovery"]
