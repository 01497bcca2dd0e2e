"""The whole draft -> retrieve -> verify iteration as ONE CUDA-graph launch with a device-side loop — this repo's replacement for
the reference's `utils/graph_infer.py` runtime (GraphInferenceEngine :129-194: gamma+3 draft graphs + one verify graph, replayed
one by one from `utils/decoding.py:163-223` with a host synchronisation after every sampled token, :186,193,203).

    parent graph = [pre] -> WHILE (n < gamma) { draft forward (gamma rows) -> draft sample -> retrieval verify forward ->
                   accept / resample / bookkeeping } -> [post: full-KV verify (gamma+2 rows) -> accept walk + residual resample ->
                   seq_len / retrieval-tail / draft-window maintenance -> results to pinned host memory]

`pre`, `body` and `post` are stream captures of the engine's own forwards (kept as cudaGraph_t); `tf_loop_graph_build` joins them
with a CUDA conditional WHILE node whose condition a kernel sets from the device-side `n` (csrc/loop_graph.cu).  Per outer
iteration the host launches one graph and reads one small record: tokens produced, accept counts, the new sequence length.

What differs from the step-wise loop (`decoding.TriForceRun`), and why results are still the same token for token:
  * the draft forward always runs gamma rows (gamma+3 for the window refresh) and the full-KV verify always gamma+2 rows; rows
    beyond the valid ones hold placeholder ids, are causally invisible to the valid rows, and their K/V slots are overwritten or
    rolled back — every kernel of the stack is row-independent, so the valid rows are bit-identical;
  * random numbers come from a counter-based Philox stream on the device (no torch generator inside a graph the host does not
    replay); `PhiloxNoise` feeds the very same draws to the step-wise loop, and `tests/test_device_loop_gpu.py` checks that both
    loops then emit identical tokens and counts (the step-wise loop itself replays the reference's golden traces).
"""
from __future__ import annotations

import ctypes
from typing import List, Optional

import torch

from . import _C, ops
from .sampling import norm_logits


class PhiloxNoise:
    """Noise source over the device Philox stream (`state` int64[2] = {seed, next draw}): same interface as rng.TorchNoise /
    rng.CounterNoise, so `decoding.TriForceRun` can consume exactly the draws the device loop consumes."""

    def __init__(self, device, seed: int = 0, state: Optional[torch.Tensor] = None):
        self.device = device
        self.state = state if state is not None else torch.tensor([int(seed), 0], dtype=torch.int64, device=device)

    def exponential_into(self, out: torch.Tensor) -> torch.Tensor:
        return ops.philox_fill(self.state, 1, out)

    def uniform_into(self, out: torch.Tensor) -> torch.Tensor:
        return ops.philox_fill(self.state, 0, out)

    def mark(self):
        return None

    def uniform_block_into(self, out: torch.Tensor) -> torch.Tensor:
        return ops.philox_fill(self.state, 0, out)  # ONE draw, element i = the uniform of the i-th examined token

    def rewind(self, mark, used: int) -> None:  # the block is one draw of the stream whatever part of it was examined
        return None


def _capture_kept(fn, mempool, warmups: int = 2):
    """Warm up `fn` on a side stream, then capture it into a CUDAGraph that keeps its cudaGraph_t (not instantiated by torch)."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(warmups):
            fn()
        s.synchronize()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph(keep_graph=True)
    before = ops.COUNTER.n
    with torch.cuda.graph(g, pool=mempool):
        fn()
    g.tf_kernels = ops.COUNTER.n - before
    return g


class DeviceLoop:
    """One outer TriForce iteration per `launch()`.  Built on a `GraphInferenceEngine` (its models, caches and memory pool)."""

    def __init__(self, graph_engine, gamma: int, temperature: float, top_p: float, eos: int = -1, strict_less: bool = True,
                 max_new: int = 1024):
        self.ge = graph_engine
        eng = self.eng = graph_engine.engine
        dev = self.dev = eng.model.device
        V = self.V = eng.model.config.vocab_size
        self.gamma, self.temperature, self.top_p = gamma, temperature, top_p
        self.rng = torch.zeros(2, dtype=torch.int64, device=dev)  # {seed, next draw} of the Philox stream (baked into the graphs)
        g = gamma
        self.st = torch.zeros(8, dtype=torch.int32, device=dev)
        self.verify_tokens = torch.full((1, g + 1), 100, dtype=torch.int64, device=dev)
        self.position_ids = torch.zeros((1, g + 1), dtype=torch.int64, device=dev)
        self.first_token = torch.zeros(1, dtype=torch.int64, device=dev)
        self.out_ids = torch.zeros(g + 2, dtype=torch.int64, device=dev)
        self.spec_probs = torch.zeros((g + 2, V), dtype=torch.float32, device=dev)
        self.full_ids = torch.full((1, g + 2), 100, dtype=torch.int64, device=dev)
        self.res = torch.zeros(16, dtype=torch.int32, device=dev)
        self.tokens = torch.zeros(g + 3, dtype=torch.int64, device=dev)
        self.pass_tokens = torch.full((1, g + 3), 100, dtype=torch.int64, device=dev)
        self.res_host = torch.zeros(16, dtype=torch.int32).pin_memory()
        self.tokens_host = torch.zeros(g + 3, dtype=torch.int64).pin_memory()
        kv, gc, dc = eng.kv_cache, eng.graph_cache, eng.draft_cache
        max_new = min(max_new, gc.max_budget)

        def draft_rows(ids):  # [1, R] ids -> probabilities of all R rows (the per-offset graphs of graph_infer.py:136-150 in one)
            R = ids.shape[-1]
            logits = eng.draft(input_ids=ids, kv_cache=dc, graph_cache=dc, gamma_offset=R - 1).logits
            return norm_logits(logits[0], temperature=temperature, top_k=-1, top_p=top_p)

        def pre():
            ops.loop_begin(self.st, self.verify_tokens, self.first_token, g, kv.seq_len_dev, self.position_ids)

        def body():
            dp = draft_rows(self.verify_tokens[:, :g])
            ops.loop_draft_sample(dp, self.st, self.rng, self.verify_tokens)
            vp = eng.model_verify(input_ids=self.verify_tokens, position_ids=self.position_ids, probs=True, temperature=temperature, top_p=top_p)
            ops.loop_middle_accept(dp, vp, self.verify_tokens, self.rng, g, self.st, self.out_ids, self.spec_probs)

        def post():
            ops.loop_prepare_full(self.st, self.out_ids, self.first_token, self.full_ids)
            logits = eng.model.forward_target(self.full_ids, kv, None, None, spec=False, use_device_len=True)
            probs = norm_logits(logits[0], temperature=temperature, top_k=-1, top_p=top_p)
            self.full_probs = probs  # [gamma+2, V]; the captured graph rewrites it on every launch
            ops.loop_verify(probs, self.spec_probs, self.out_ids, self.st, self.rng, strict_less, eos, self.first_token, self.res, self.tokens,
                            self.pass_tokens, kv.seq_len_dev)
            gc.update_graph_cache(kv, use_device_len=True, max_new=max_new)
            draft_rows(self.pass_tokens)  # refresh the draft window with the tokens of this step (decoding.py:137)
            ops.window_slide_dev(dc.key_store, dc.value_store, dc.start_size, self.res[8:9], dc.start_size, dc.recent_size)
            self.res_host.copy_(self.res, non_blocking=True)
            self.tokens_host.copy_(self.tokens, non_blocking=True)

        # warm-ups run the pieces eagerly: give them a consistent state, then put the caches' lengths back
        saved_len = kv.seq_len
        kv.sync_seq_len_to_device()
        pool = graph_engine.mempool or torch.cuda.graphs.graph_pool_handle()
        rng_saved = self.rng.clone()
        self._graphs = [_capture_kept(pre, pool), _capture_kept(body, pool), _capture_kept(post, pool)]
        self.rng.copy_(rng_saved)
        kv.seq_len = saved_len
        kv._dev_mirror = -1
        kv.sync_seq_len_to_device()
        self.kernels_per_inner = self._graphs[1].tf_kernels + 1
        self.kernels_fixed = self._graphs[0].tf_kernels + self._graphs[2].tf_kernels
        exec_out = ctypes.c_void_p()
        _C.check(_C.lib().tf_loop_graph_build(ctypes.c_void_p(self._graphs[0].raw_cuda_graph()), ctypes.c_void_p(self._graphs[1].raw_cuda_graph()),
                                              ctypes.c_void_p(self._graphs[2].raw_cuda_graph()), self.st.data_ptr(), g, ctypes.byref(exec_out)),
                 "tf_loop_graph_build")
        self._exec = exec_out

    @classmethod
    def for_engine(cls, graph_engine, gamma, temperature, top_p, eos=-1, strict_less=True, max_new=1024) -> "DeviceLoop":
        """One captured loop per engine and sampling setup (capturing costs seconds and graph-pool memory)."""
        key = (gamma, float(temperature), float(top_p), int(eos), bool(strict_less), int(max_new))
        cache = graph_engine.__dict__.setdefault("_device_loops", {})
        if key not in cache:
            cache[key] = cls(graph_engine, gamma, temperature, top_p, eos=eos, strict_less=strict_less, max_new=max_new)
        return cache[key]

    def set_first_token(self, token: int):
        self.first_token.fill_(int(token))

    def launch(self):
        """Enqueue one outer iteration (no host synchronisation)."""
        _C.check(_C.lib().tf_loop_graph_launch(self._exec, _C.stream_ptr()), "tf_loop_graph_launch")

    def read(self):
        """Wait for the launched iteration and return (result record, tokens it produced)."""
        torch.cuda.current_stream().synchronize()
        r = self.res_host.tolist()
        return r, self.tokens_host[:r[0]].tolist()

    def __del__(self):
        try:
            if getattr(self, "_exec", None):
                _C.lib().tf_loop_graph_destroy(self._exec)
        except Exception:
            pass


class DeviceLoopRun:
    """`decoding.TriForceRun` on the device loop: same attributes (`n`, `generated`, `acceptance_rate`, …), `step()` = one graph
    launch + one read-back."""

    def __init__(self, tokenizer, graph_engine, gamma=4, top_k=-1, top_p=0.9, temperature=0.6, seed: int = 0, strict_less=True,
                 max_new: int = 1024):
        from .decoding import TriForceRun
        self.ge, self.eng = graph_engine, graph_engine.engine
        self.dev = self.eng.model.device
        self.gamma = gamma
        self.eos = tokenizer.eos_token_id if tokenizer is not None and tokenizer.eos_token_id is not None else -1
        self.loop = DeviceLoop.for_engine(graph_engine, gamma, temperature, top_p, eos=self.eos, strict_less=strict_less, max_new=max_new)
        self.loop.rng.copy_(torch.tensor([int(seed), 0], dtype=torch.int64))  # restart the stream
        self.noise = PhiloxNoise(self.dev, state=self.loop.rng)
        # the prompt phase (prefill, retrieval build, draft prefill, first token) is the step-wise loop's, on the same noise stream
        self._host = TriForceRun(tokenizer, graph_engine, gamma=gamma, top_k=top_k, top_p=top_p, temperature=temperature, noise=self.noise,
                                 strict_less=strict_less)
        self.n = 0
        self.generated: List[int] = []
        self.accepted_count = self.draft_count = self.resample_count = self.target_sample_count = 0
        self.inner_iterations = self.inner_accepts = 0
        self.steps = 0
        self.next_token: Optional[int] = None
        self.h2d_bytes = self.d2h_bytes = 0
        self.records: List[list] = []

    @torch.inference_mode()
    def prefill(self, input_ids, skip_target_prefill: bool = False):
        tok = self._host.prefill(input_ids, skip_target_prefill=skip_target_prefill)
        self.generated = [tok]
        self.next_token = tok
        kv = self.eng.kv_cache
        kv.sync_seq_len_to_device()
        self.loop.set_first_token(tok)
        self.h2d_bytes += 8
        return tok

    @torch.inference_mode()
    def step(self) -> int:
        self.loop.launch()
        r, toks = self.loop.read()
        produced, count, rejected, g2, examined, hit_eos, inner, inner_acc, shift, new_len = r[:10]
        kv = self.eng.kv_cache
        kv.seq_len = new_len
        kv._dev_mirror = new_len
        self.records.append(r[:10])
        self.steps += 1
        self.n += produced
        self.generated.extend(toks)
        self.accepted_count += count
        self.draft_count += g2 - ((g2 - count) if hit_eos else 0)
        self.resample_count += 1 if rejected else 0
        self.target_sample_count += 1 if (not rejected and count == g2) else 0
        self.inner_iterations += inner
        self.inner_accepts += inner_acc
        self.next_token = toks[-1] if toks else self.next_token
        self.d2h_bytes += 16 * 4 + (self.gamma + 3) * 8
        ops.COUNTER.n += self.loop.kernels_fixed + inner * self.loop.kernels_per_inner
        return produced

    @property
    def acceptance_rate(self) -> float:
        return self.accepted_count / max(self.draft_count, 1)
