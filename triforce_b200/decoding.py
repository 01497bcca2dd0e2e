"""The speculative-decoding loops of the reference's `utils/decoding.py` — `Autoregressive` (:14-37), `TriForce`
(:41-160), `Middle_Spec` (:163-223) and their tensor-parallel twins (:230-495) — with the same signatures and return
values, on the fused kernels:

  * every multinomial is `argmax(p / Exp(1))` on the device (`tf_sample_argmax`), the draft token never visits the host;
  * one inner decision (accept test + the multinomial that follows + bookkeeping of ids / proposal rows / slot
    update) is ONE kernel (`tf_middle_accept`); the host reads back a single int per inner iteration (the reference
    synchronises three times: decoding.py:186,193,203);
  * the outer accept walk and the residual / bonus resample are two kernels (`tf_verify_accept`, `tf_verify_resample`).

Random numbers come from a *noise source* (triforce_b200.rng): `TorchNoise` consumes torch's Philox stream in the
reference's call order; tests replay committed `CounterNoise` streams.  `trace`, when given, receives the same
("sample" | "rand" | "middle" | "target_in", value) events the golden fixtures were recorded with.
"""
from __future__ import annotations

import time
from typing import List, Optional

import numpy as np
import torch

from . import ops
from .rng import TorchNoise
from .sampling import norm_logits


class _LoopBuffers:
    """Device scratch of the loops, allocated once per engine."""

    def __init__(self, device, gamma: int, V: int):
        self.gamma, self.V = gamma, V
        self.verify_tokens = torch.empty((1, gamma + 1), dtype=torch.int64, device=device)
        self.state = torch.zeros(8, dtype=torch.int32, device=device)
        self.out_ids = torch.zeros(gamma + 2, dtype=torch.int64, device=device)
        self.spec_probs = torch.zeros((gamma + 2, V), dtype=torch.float32, device=device)
        self.expo = torch.empty(V, dtype=torch.float32, device=device)
        self.expo2 = torch.empty(V, dtype=torch.float32, device=device)
        self.uniform = torch.empty(1, dtype=torch.float32, device=device)
        self.uniforms = torch.empty(gamma + 2, dtype=torch.float32, device=device)
        self.res = torch.zeros(4, dtype=torch.int32, device=device)
        self.out_token = torch.zeros(1, dtype=torch.int64, device=device)
        self.pass_tokens = torch.zeros((1, gamma + 3), dtype=torch.int64, device=device)
        self.gen = torch.zeros(gamma + 2, dtype=torch.int64, device=device)


def _buffers(graph_engine, gamma: int) -> _LoopBuffers:
    V = graph_engine.engine.model.config.vocab_size
    b = getattr(graph_engine, "_loop_buffers", None)
    if b is None or b.gamma != gamma or b.V != V:
        b = _LoopBuffers(graph_engine.engine.model.device, gamma, V)
        graph_engine._loop_buffers = b
    return b


def _sample_token(probs_row: torch.Tensor, noise, expo: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    noise.exponential_into(expo)
    return ops.sample_argmax(probs_row, expo, out=out)


@torch.inference_mode()
def Autoregressive(tokenizer, graph_engine, input_ids, max_len=256, top_k=-1, top_p=0.9, temperature=0.6, verbose=False,
                   noise=None, trace=None, return_tokens=False):
    eng = graph_engine.engine
    noise = noise or TorchNoise(eng.model.device)
    buf = _buffers(graph_engine, graph_engine.gamma or 1)
    eng.kv_cache.reset()
    logits = graph_engine.inference(input_ids=input_ids)
    if verbose:
        eng.kv_cache.print_status()
    next_token = _sample_token(norm_logits(logits[:, -1, :], temperature=temperature, top_k=top_k, top_p=top_p), noise, buf.expo)
    tokens = [next_token]
    n = 0
    torch.cuda.synchronize()
    time1 = time.time()
    while n < max_len:
        logits = graph_engine.decode_step(next_token)
        next_token = _sample_token(norm_logits(logits[:, -1, :], temperature=temperature, top_k=top_k, top_p=top_p), noise, buf.expo)
        tokens.append(next_token)
        n += 1
    torch.cuda.synchronize()
    time2 = time.time()
    if trace is not None or return_tokens:
        toks = [int(t.item()) for t in tokens]
        if trace is not None:
            trace.extend(("sample", t) for t in toks)
        if return_tokens:
            return n / (time2 - time1), toks
    return n / (time2 - time1)


@torch.inference_mode()
def Middle_Spec(next_token, graph_engine, gamma, verbose, tokenizer, noise=None, trace=None):
    """Draft (68M + StreamingLLM) → retrieval-cache verify, decoding.py:163-223.
    Returns (ids [python ints, first = next_token], proposal rows [k, V] device tensor, acceptance rate)."""
    eng = graph_engine.engine
    dev = eng.model.device
    noise = noise or TorchNoise(dev)
    buf = _buffers(graph_engine, gamma)
    first = int(next_token.item()) if torch.is_tensor(next_token) else int(next_token)
    buf.verify_tokens.fill_(100)
    buf.verify_tokens[0, 0] = first
    buf.state.zero_()
    seq_len = eng.kv_cache.seq_len
    position_ids = torch.arange(seq_len, seq_len + gamma + 1, device=dev).unsqueeze(0)
    n = 0
    while n < gamma:
        speculation_prob = graph_engine.graph_draft_inference(input_ids=buf.verify_tokens[:, :n + 1], gamma_offset=n)
        _sample_token(speculation_prob, noise, buf.expo, out=buf.verify_tokens[0, n + 1:n + 2])
        if trace is not None:
            trace.append(("sample", int(buf.verify_tokens[0, n + 1].item())))
        verify_prob = graph_engine.graph_verify(input_ids=buf.verify_tokens, position_ids=position_ids)
        noise.uniform_into(buf.uniform)
        noise.exponential_into(buf.expo2)
        k_before = None
        if trace is not None:
            k_before = int(buf.state[1].item())
        ops.middle_accept(speculation_prob, verify_prob, buf.verify_tokens, buf.uniform, buf.expo2, gamma, buf.state,
                          buf.out_ids, buf.spec_probs)
        st = buf.state.tolist()  # the one host sync of the inner iteration
        n = st[0]
        if trace is not None:
            trace.append(("rand", float(buf.uniform.item())))
            trace.append(("sample", int(buf.out_ids[st[1] - 1].item())))
    k = st[1]
    buf.last_inner_iterations = st[4]
    ids = [first] + buf.out_ids[:k].tolist()
    if trace is not None:
        trace.append(("middle", list(ids)))
    acceptance_rate = st[3] / max(st[4], 1)
    return ids, buf.spec_probs[:k], acceptance_rate


class TriForceRun:
    """Step-wise form of `TriForce` (decoding.py:41-160): `prefill()` = :44-62, `step()` = one pass of the :70-141 loop.
    `TriForce(...)` below drives it; `bench.py` drives it directly to time exactly K steps."""

    def __init__(self, tokenizer, graph_engine, gamma=4, top_k=-1, top_p=0.9, temperature=0.6, noise=None, trace=None,
                 strict_less=True, pad_full_verify: bool = False):
        self.ge = graph_engine
        self.eng = graph_engine.engine
        self.dev = self.eng.model.device
        self.gamma, self.top_k, self.top_p, self.temperature = gamma, top_k, top_p, temperature
        self.noise = noise or TorchNoise(self.dev)
        self.trace = trace
        self.tokenizer = tokenizer
        self.strict_less = strict_less
        # pad the full-KV verify to gamma+2 rows (placeholder ids, causally invisible to the real rows, rolled back afterwards):
        # what the device loop (device_loop.py) always does — used to compare the two loops bit for bit
        self.pad_full_verify = pad_full_verify
        self.buf = _buffers(graph_engine, gamma)
        self.eos = tokenizer.eos_token_id if tokenizer is not None and tokenizer.eos_token_id is not None else -1
        self.resample_count = self.accepted_count = self.target_sample_count = self.draft_count = 0
        self.acc_rate_middle_list: List[float] = []
        self.n = 0
        self.generated: List[int] = []
        self.next_token: Optional[int] = None
        self.inner_iterations = 0
        self.h2d_bytes = self.d2h_bytes = 0

    @torch.inference_mode()
    def prefill(self, input_ids, skip_target_prefill: bool = False):
        eng, ge, trace = self.eng, self.ge, self.trace
        if not skip_target_prefill:
            eng.kv_cache.reset()
        eng.graph_cache.reset()
        eng.draft_cache.reset()
        if not skip_target_prefill:
            ge.inference(input_ids=input_ids[:, :-1])
        else:  # bench.py: the prompt's KV is already in HBM from an earlier prefill; roll the length back to P-1
            eng.kv_cache.seq_len = input_ids.shape[1] - 1
        if trace is not None:
            trace.append(("target_in", [int(input_ids[0, -1])]))
        logits = ge.inference(input_ids=input_ids[:, -1:])
        ge.graph_draft_prefill(input_ids=input_ids)
        self.next_token = int(_sample_token(norm_logits(logits[:, -1, :], temperature=self.temperature, top_k=self.top_k,
                                                        top_p=self.top_p), self.noise, self.buf.expo).item())
        if trace is not None:
            trace.append(("sample", self.next_token))
        self.generated = [self.next_token]
        return self.next_token

    @torch.inference_mode()
    def step(self) -> int:
        """One outer iteration; returns the number of tokens it produced."""
        eng, ge, buf, trace, noise, gamma = self.eng, self.ge, self.buf, self.trace, self.noise, self.gamma
        n_before = self.n
        next_token = self.next_token
        # speculative decoding for draft (68m) and retrieval 7b model
        ids, speculation_probs, acc_rate_middle = Middle_Spec(next_token, ge, gamma, False, self.tokenizer, noise=noise, trace=trace)
        self.acc_rate_middle_list.append(acc_rate_middle)
        generated_ids = ids[1:]
        gamma2 = len(generated_ids)
        self.draft_count += gamma2
        self.inner_iterations += buf.last_inner_iterations
        self.d2h_bytes += buf.last_inner_iterations * 32 + 8 * gamma2

        # speculative decoding retrieval 7b model and target model
        pad = (gamma + 2 - len(ids)) if self.pad_full_verify else 0
        verify_tokens = torch.tensor([ids + [100] * pad], dtype=torch.int64, device=self.dev)
        self.h2d_bytes += 8 * len(ids)
        if trace is not None:
            trace.append(("target_in", list(ids)))
        logits = ge.inference(input_ids=verify_tokens)
        if pad:
            eng.kv_cache.seq_len -= pad  # the padding rows were appended too: roll them back at once
        probs = norm_logits(logits[0], temperature=self.temperature, top_k=self.top_k, top_p=self.top_p)
        self.full_probs = probs[:len(ids)]  # the target's distribution at the verified rows, kept for inspection

        gen_dev = verify_tokens[0, 1:]
        mark = noise.mark()
        noise.uniform_block_into(buf.uniforms[:gamma2])
        ops.verify_accept(probs, speculation_probs, gen_dev, gamma2, buf.uniforms, self.strict_less, self.eos, next_token, buf.res,
                          buf.pass_tokens)
        count, rejected, examined, hit_eos = buf.res.tolist()  # host sync: the walk's outcome drives the RNG order
        noise.rewind(mark, examined)  # the reference draws one rand(1) per EXAMINED token only
        if trace is not None:
            trace.extend(("rand", float(u)) for u in buf.uniforms[:examined].tolist())
        draws_token = bool(rejected) or count == gamma2
        if draws_token:
            noise.exponential_into(buf.expo)
        ops.verify_resample(probs, speculation_probs, gen_dev, gamma2, buf.expo, buf.res, buf.out_token, buf.pass_tokens)
        pred_token_idx = int(buf.out_token.item())
        self.d2h_bytes += 16 + 8
        if trace is not None and draws_token:
            trace.append(("sample", pred_token_idx))

        self.accepted_count += count
        self.n += count
        self.generated.extend(generated_ids[:count])
        if hit_eos:
            self.draft_count -= gamma2 - count
        if rejected:
            self.resample_count += 1
            self.n += 1
            self.generated.append(pred_token_idx)

        # update 7b cache
        eng.kv_cache.seq_len -= (gamma2 - count)
        ge.update_graph_cache()

        if count == gamma2:
            self.target_sample_count += 1
            self.n += 1
            self.generated.append(pred_token_idx)
            count += 1

        # update cache for 68m
        ge.graph_draft_inference(input_ids=buf.pass_tokens[:, :gamma2 + 2], gamma_offset=gamma2 + 1)
        current_seq_len = eng.draft_cache.start_size + eng.draft_cache.recent_size + count
        eng.draft_cache.evict_for_spec(current_seq_len)

        self.next_token = pred_token_idx
        return self.n - n_before

    @property
    def acceptance_rate(self) -> float:
        return self.accepted_count / max(self.draft_count, 1)

    def stats(self, seconds: float) -> dict:
        return dict(tokens=self.generated, n=self.n, seconds=seconds, accepted_count=self.accepted_count,
                    draft_count=self.draft_count, resample_count=self.resample_count,
                    target_sample_count=self.target_sample_count,
                    acc_rate_middle=float(np.mean(self.acc_rate_middle_list)) if self.acc_rate_middle_list else 0.0,
                    avg_tokens=self.acceptance_rate * self.gamma, outer_iterations=len(self.acc_rate_middle_list))


@torch.inference_mode()
def TriForce(tokenizer, graph_engine, input_ids, gamma=4, max_len=256, top_k=-1, top_p=0.9, temperature=0.6, verbose=False,
             file_path=None, dataset=None, spec_args=None, noise=None, trace=None, stats=None, strict_less=True):
    eng = graph_engine.engine
    run = TriForceRun(tokenizer, graph_engine, gamma=gamma, top_k=top_k, top_p=top_p, temperature=temperature, noise=noise,
                      trace=trace, strict_less=strict_less)
    run.prefill(input_ids)
    if verbose:
        eng.kv_cache.print_status()
        eng.graph_cache.print_status()
        eng.draft_cache.print_status()
    torch.cuda.synchronize()
    time1 = time.time()
    while run.n < max_len:
        run.step()
    torch.cuda.synchronize()
    time2 = time.time()
    n = run.n
    acceptance_rate = run.acceptance_rate
    avg_tokens = acceptance_rate * gamma
    if verbose:
        print(f"Use {time2 - time1} sec to generate {n} tokens (now {eng.kv_cache.seq_len} tokens), Tokens/s: {n / (time2 - time1)}", flush=True)
        print(f"accepted rate {acceptance_rate}, avg generated tokens {avg_tokens}")
    if stats is not None:
        stats.update(run.stats(time2 - time1))
    if file_path is not None:
        header = "target,acceptance_rate,token/s,avg_tokens,prefill,gen_len,dataset,acc_rate_middle,latency\n"
        entry = (f"{eng.model.config._name_or_path},{acceptance_rate},{n / (time2 - time1)},{avg_tokens},{input_ids.shape[1]},{n},"
                 f"{dataset},{np.array(run.acc_rate_middle_list).mean()},{(time2 - time1) / n}\n")
        if spec_args is not None:
            for k_, v_ in spec_args.items():
                header = header.replace("\n", f",{k_}\n")
                entry = entry.replace("\n", f",{v_}\n")
        from .misc import log_csv
        log_csv(file_path, header, entry)
    return acceptance_rate, n / (time2 - time1)


# ---- tensor-parallel twins (decoding.py:230-495) ---------------------------------------------------------------------
def sample_dist(probs, noise=None):
    """decoding.py:230-239 samples on rank 0 and broadcasts (+barrier).  Here every rank draws the same token from its
    identically seeded stream — the probabilities are bit-identical after the all-reduce — so nothing is communicated."""
    from .sampling import sample
    return sample(probs, noise=noise)


@torch.inference_mode()
def Baseline_Dist(tokenizer, graph_engine, input_ids, max_len=256, top_k=-1, top_p=0.9, temperature=0.6, verbose=False, local_rank=0,
                  noise=None):
    """decoding.py:243-287: returns (ms per token, generated tokens [1, max_len]).  `graph_engine` is a DistributedLlama."""
    llm = graph_engine
    noise = noise or TorchNoise(llm.device)
    llm.reset()
    logits = llm.prefill(input_ids=input_ids)
    expo = torch.empty(llm.vocab_size, dtype=torch.float32, device=llm.device)
    next_token = _sample_token(norm_logits(logits[:, -1, :], temperature=temperature, top_k=top_k, top_p=top_p), noise, expo)
    gen_tokens = torch.zeros((input_ids.size(0), max_len), dtype=torch.long, device=input_ids.device)
    n = 0
    torch.cuda.synchronize()
    time1 = time.time()
    while n < max_len:
        logits = llm.graph_engine.decode_step(next_token) if llm.graph_engine is not None else llm.inference(next_token.reshape(1, 1))
        next_token = _sample_token(norm_logits(logits[:, -1, :], temperature=temperature, top_k=top_k, top_p=top_p), noise, expo)
        gen_tokens[:, n] = next_token.squeeze()
        n += 1
    torch.cuda.synchronize()
    time2 = time.time()
    return 1000 * (time2 - time1) / n, gen_tokens


@torch.inference_mode()
def Middle_Spec_Dist(next_token, llm, gamma, verbose, tokenizer, noise=None, trace=None):
    return Middle_Spec(next_token, llm.graph_engine, gamma, verbose, tokenizer, noise=noise, trace=trace)


@torch.inference_mode()
def TriForce_Dist(tokenizer, llm, input_ids, gamma=4, max_len=256, top_k=-1, top_p=0.9, temperature=0.6, verbose=False, file_path=None,
                  dataset=None, spec_args=None, noise=None, trace=None, stats=None):
    """decoding.py:291-428: returns (avg accepted tokens, seconds per token).  Differences kept from the reference's TP
    variant: the outer accept test is `r <= min(1, p/q)` (:354) and generation stops at an EOS token (:384-392).
    Known, documented deviations from the reference's TP loop (harmless for the shipped scripts, which use top_k = -1):
    the prefill sample honours the caller's `top_k` (the reference hard-codes -1 there, :304); when the step's next token is EOS
    the reference breaks BEFORE the KV rollback / retrieval-tail update / draft refresh of that step (:382-392) while this loop
    finishes `step()` first (the caches are reset by the next call either way)."""
    run = TriForceRun(tokenizer, llm.graph_engine, gamma=gamma, top_k=top_k, top_p=top_p, temperature=temperature, noise=noise,
                      trace=trace, strict_less=False)
    run.prefill(input_ids)
    torch.cuda.synchronize()
    time1 = time.time()
    while run.n < max_len:
        run.step()
        if tokenizer is not None and run.next_token == tokenizer.eos_token_id:
            break
    torch.cuda.synchronize()
    time2 = time.time()
    if stats is not None:
        stats.update(run.stats(time2 - time1))
    return run.acceptance_rate * gamma, (time2 - time1) / max(run.n, 1)
