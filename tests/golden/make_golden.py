#!/usr/bin/env python
"""Generates the committed golden fixtures in this directory FROM THE REFERENCE ITSELF (run where a checkout of the
reference is at $TRIFORCE_REFERENCE_ROOT, see `oracle/ref_harness.py`).  Usage:  python tests/golden/make_golden.py [which ...]

The reference ships no tests or golden vectors (SURVEY.md §4), so these fixtures — outputs of the reference's own
Python (`models/cache.py`, `utils/sampling.py`, `utils/decoding.py`, `models/modeling_llama*.py`) executed on CPU under
the shims documented in `oracle/ref_harness.py` — are what pins `oracle/triforce_oracle.py`.  Inputs are regenerated
from PCG64 seeds by the tests (see `tests/golden_inputs.py`), so only outputs are stored.

Files written:
  retrieval_build.npz   reference RetrievalCache.init_graph_cache: fp16 chunk scores, raw torch.topk indices, cache rows
  sampling.npz          reference norm_logits / max_fn on seeded logits
  forward.npz           reference target forward: last-token logits after a chunked prefill, retrieval-verify logits
  e2e_<cfg>.json        event traces (every sample / rand / Middle_Spec return / target input) of TriForce first and
                        second call (the draft-cache reset quirk, SURVEY §7 hard part 3) and of Autoregressive
  tree_512.json         the reference's SpecTree rounds over the 512-node tree
  reference_tree_512.json   the reference's tree/512.pt (roots, branches, Successors, depth; mask rows as packed bits)
  reference_cli_flags.json  every flag of the reference's test/*.py entry points with its default
  pg19_sample/, dataset_gs.npz   24 PG-19 books cut to 2000 characters, and the reference's get_dataset('gs') on them
"""
from __future__ import annotations

import json
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.abspath(os.path.join(HERE, "..", ".."))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))

from oracle import ref_harness as rh  # noqa: E402
from oracle import triforce_oracle as orc  # noqa: E402
from triforce_b200.config import named_config  # noqa: E402
from triforce_b200.rng import CounterNoise  # noqa: E402
from triforce_b200.synth import numpy_state_dict, numpy_prompt  # noqa: E402
import golden_inputs as gi  # noqa: E402


class _ShapeModel:
    """Just enough of an HF model for the reference cache constructors (cache.py:25-33,131-139)."""

    def __init__(self, L, H, d):
        self.config = type("C", (), dict(hidden_size=H * d, num_key_value_heads=H, num_attention_heads=H,
                                         num_hidden_layers=L))()
        w = type("W", (), dict(dtype=torch.float16))()
        attn = type("A", (), dict(q_proj=type("Q", (), dict(weight=w))()))()
        self.model = type("M", (), dict(layers=[type("Lyr", (), dict(self_attn=attn))()]))()
        self.device = torch.device("cpu")


def make_retrieval_build():
    ref = rh.load_reference()
    out = {}
    for case in gi.RETRIEVAL_CASES:
        name, H, d, P, chunk, budget, seed = case
        K, V, q = gi.retrieval_inputs(case)
        m = _ShapeModel(1, H, d)
        kv = ref.cache.FlashSimpleCache(m, P + 8)
        kv.key_cache[0, 0, :P] = torch.from_numpy(K)
        kv.value_cache[0, 0, :P] = torch.from_numpy(V)
        kv.seq_len = P
        rc = ref.cache.RetrievalCache(m, max_budget=budget, prefill=P, chunk_size=chunk, gamma=4)
        rec = {}
        orig_torch = ref.cache.torch

        class _Proxy:
            def __getattr__(self, n):
                return getattr(orig_torch, n)

            @staticmethod
            def topk(x, k, dim=-1, **kw):
                v, i = orig_torch.topk(x, k=k, dim=dim, **kw)
                rec["scores_rest"] = x.clone()
                rec["idx_rest"] = i.clone()
                return v, i

        ref.cache.torch = _Proxy()
        try:
            rc.init_graph_cache(kv, torch.from_numpy(q).reshape(1, 1, H, d), 0)
        finally:
            ref.cache.torch = orig_torch
        scores_rest = rec["scores_rest"][0].numpy()  # [H, chunks-1] fp16 (chunk 0 excluded by the reference slice)
        idx = rec["idx_rest"][0].numpy().astype(np.int32) + 1  # raw torch.topk order, shifted like cache.py:160
        out[f"{name}.scores_rest"] = scores_rest
        out[f"{name}.topk_idx_rest"] = idx
        rk = rc.key_cache[0, 0, :budget].numpy()
        rv = rc.value_cache[0, 0, :budget].numpy()
        # store a digest of the gathered rows instead of megabytes: per-(slot-chunk, head) sums in fp64
        out[f"{name}.retrK_digest"] = rk.astype(np.float64).reshape(budget // chunk, chunk, H, d).sum((1, 3))
        out[f"{name}.retrV_digest"] = rv.astype(np.float64).reshape(budget // chunk, chunk, H, d).sum((1, 3))
        # cross-check the oracle while we are here
        oK, oV, oidx, osc = orc.retrieval_build(K, V, q, P, chunk, budget)
        ulp_diff = (osc[:, 1:].view(np.int16).astype(np.int32) - scores_rest.view(np.int16).astype(np.int32))
        frac = float((ulp_diff != 0).mean())
        same_set = all(set(oidx[h, 1:]) == set(idx[h]) for h in range(H))
        print(f"[retrieval_build:{name}] oracle-vs-reference score mismatch frac={frac:.5f} "
              f"max|ulp|={np.abs(ulp_diff).max()} same top-k set={same_set}")
        out[f"{name}.oracle_score_mismatch_frac"] = np.float64(frac)
    np.savez_compressed(os.path.join(HERE, "retrieval_build.npz"), **out)


def make_sampling():
    ref = rh.load_reference()
    out = {}
    for case in gi.SAMPLING_CASES:
        name = case[0]
        logits = gi.sampling_logits(case)
        T, top_p = case[4], case[5]
        probs = ref.sampling.norm_logits(torch.from_numpy(logits.copy()), temperature=T, top_k=-1, top_p=top_p).numpy()
        out[f"{name}.probs"] = probs.astype(np.float32)
        o = orc.norm_logits(logits.copy(), T, -1, top_p)
        print(f"[sampling:{name}] kept ref={int((probs > 0).sum())} oracle={int((o > 0).sum())} "
              f"mask mismatches={int(((probs > 0) != (o > 0)).sum())} max|dp|={np.abs(o - probs).max():.3e}")
        p, q = gi.residual_pair(case)
        out[f"{name}.max_fn"] = ref.sampling.max_fn(torch.from_numpy(p - q)).numpy()
    np.savez_compressed(os.path.join(HERE, "sampling.npz"), **out)


def _models(case):
    ts, ds = named_config(case["target"]), named_config(case["draft"])
    tsd = numpy_state_dict(ts, case["target_seed"])
    dsd = numpy_state_dict(ds, case["draft_seed"])
    target, draft = rh.build_reference_models(ts, ds, tsd, dsd)
    return ts, ds, tsd, dsd, target, draft


def make_forward():
    case = gi.FORWARD_CASE
    ts, ds, tsd, dsd, target, draft = _models(case)
    P, B, c, g = case["prefill"], case["budget"], case["chunk"], case["gamma"]
    ge = rh.build_reference_engine(target, draft, P, 32, B, c, g, case["temperature"], case["top_p"])
    ids = numpy_prompt(P, seed=case["prompt_seed"])
    with torch.inference_mode():
        ge.engine.kv_cache.reset(); ge.engine.graph_cache.reset(); ge.engine.draft_cache.reset()
        ge.inference(input_ids=ids[:, :-1])
        logits_last = ge.inference(input_ids=ids[:, -1:])[0, -1].numpy()
        vt = torch.from_numpy(np.asarray(case["verify_tokens"], dtype=np.int64))[None]
        pos = torch.arange(P, P + g + 1)[None]
        vlogits = ge.engine.model_verify(input_ids=vt, position_ids=pos, probs=False)[0].numpy()
        # full-KV verify of the same rows (non-spec path, graph_cache given but q_len > 1 so no rebuild)
        flogits = ge.inference(input_ids=vt)[0].numpy()
        # draft: prefill then one speculative step of 3 tokens
        ge.graph_draft_prefill(input_ids=ids)
        dlogits = ge.engine.draft_run(input_ids=vt[:, :3], gamma_offset=2, probs=False)[0].numpy()
    rot = target.model.layers[0].self_attn.rotary_emb
    np.savez_compressed(os.path.join(HERE, "forward.npz"),
                        logits_last=logits_last.astype(np.float16), verify_logits=vlogits.astype(np.float16),
                        full_verify_logits=flogits.astype(np.float16), draft_logits=dlogits.astype(np.float16),
                        yarn_cos_rows=rot.cos_cached[:: 97].numpy(), yarn_sin_rows=rot.sin_cached[:: 97].numpy())
    assert np.array_equal(logits_last.astype(np.float16).astype(np.float32), logits_last)
    print("[forward] wrote logits; |logits| max", np.abs(logits_last).max())


def make_e2e():
    ref = rh.load_reference()
    tok = rh.TokenizerStub()
    only = os.environ.get("GOLDEN_E2E_ONLY")  # regenerate one case: GOLDEN_E2E_ONLY=plain [GOLDEN_NOISE_SEED=n]
    for case in gi.E2E_CASES:
        if only and case["name"] != only:
            continue
        if os.environ.get("GOLDEN_NOISE_SEED"):
            case = dict(case, noise_seed=int(os.environ["GOLDEN_NOISE_SEED"]))
        t0 = time.time()
        ts, ds, tsd, dsd, target, draft = _models(case)
        P, B, c, g, gen = case["prefill"], case["budget"], case["chunk"], case["gamma"], case["gen_len"]
        T, top_p = case["temperature"], case["top_p"]
        ge = rh.build_reference_engine(target, draft, P, gen + 16, B, c, g, T, top_p)
        ids = numpy_prompt(P, seed=case["prompt_seed"])
        ot = orc.LlamaOracle(ts, {k: v.numpy() for k, v in tsd.items()}, False)
        od = orc.LlamaOracle(ds, {k: v.numpy() for k, v in dsd.items()}, True)
        rot = target.model.layers[0].self_attn.rotary_emb
        rd = draft.model.layers[0].self_attn.rotary_emb
        ot.set_tables(rot.cos_cached.numpy(), rot.sin_cached.numpy())
        od.set_tables(rd.cos_cached.numpy().astype(np.float16), rd.sin_cached.numpy().astype(np.float16))
        eng = orc.EngineOracle(ot, od, P, gen + 16, B, c, g, T, top_p)
        record = dict(case=case, calls=[])
        for call in range(2):
            trace = []
            with rh.traced_random(CounterNoise(case["noise_seed"]), trace), rh.traced_calls(ge, trace):
                acc, _ = ref.decoding.TriForce(tok, ge, ids, gamma=g, max_len=gen, top_k=-1, top_p=top_p, temperature=T)
            res = orc.triforce(eng, ids.numpy(), g, gen, CounterNoise(case["noise_seed"]))
            same = 0
            for a, b in zip(trace, res["trace"]):
                if a[0] != b[0] or a[1] != b[1]:
                    break
                same += 1
            record["calls"].append(dict(trace=[[e[0], e[1]] for e in trace], acceptance_rate=acc,
                                        oracle_matching_prefix=same, events=len(trace)))
            print(f"[e2e:{case['name']}] call {call}: acceptance {acc:.4f}, events {len(trace)}, "
                  f"oracle matches first {same} events ({time.time() - t0:.1f}s)")
        # autoregressive baseline trace (decoding.py:14-37)
        trace = []
        with rh.traced_random(CounterNoise(case["noise_seed"]), trace):
            ref.decoding.Autoregressive(tok, ge, ids, max_len=case["ar_len"], top_k=-1, top_p=top_p, temperature=T)
        eng.kv_cache.reset()
        otoks = orc.autoregressive(eng, ids.numpy(), case["ar_len"], CounterNoise(case["noise_seed"]))
        rtoks = [e[1] for e in trace if e[0] == "sample"]
        record["autoregressive"] = dict(tokens=rtoks, oracle_equal=(rtoks == otoks))
        print(f"[e2e:{case['name']}] AR tokens equal to oracle: {rtoks == otoks}")
        with open(os.path.join(HERE, f"e2e_{case['name']}.json"), "w") as f:
            json.dump(record, f)


def make_tree():
    """Sequoia tree path: the reference's SpecTree (utils/SpecTree_TP.py) on the functional reference layers, see
    oracle/ref_tree_harness.py.  Stores every round's 512 tree tokens, accepted tokens and random draws."""
    from oracle import ref_tree_harness as th
    from triforce_b200.spectree import load_grow_map
    case = gi.TREE_CASE
    ts = named_config(case["target"])
    sd = numpy_state_dict(ts, case["target_seed"])
    P, B, c, T = case["prefill"], case["budget"], case["chunk"], case["tree_size"]
    eng = th.RefTreeEngine(ts, sd, P, 64, B, c, T)
    ref = th.load_tree_reference()
    gm = load_grow_map(str(T))
    calls, gather = th.build_sampling(gm, case["temperature"])
    noise = CounterNoise(case["noise_seed"])
    trace, rounds = [], []
    with th.traced_tree_random(noise, trace):
        st = ref.spectree.SpecTree(engine=eng, temperature=case["temperature"], top_p=case["top_p"], max_length=P + 64, grow_map=gm,
                                   residual_graph=th.get_residual, sampling_callables=calls, sample_gather_indices=gather,
                                   tokenizer=None, vocab_size=ts.vocab_size)
        ids = numpy_prompt(P, seed=case["prompt_seed"])[0]
        nt = st.prefill(prefix=ids)
        first = int(nt.reshape(-1)[0])
        for r in range(case["rounds"]):
            mark = len(trace)
            st.construct_grow_map(next_token=nt)
            tree_tokens = st.verify_tokens.tolist()
            seq_before = eng.kv_cache.seq_len
            nt, acc, toks = st.verify()
            rounds.append(dict(tree_tokens=tree_tokens, acc_count=int(acc), accept_tokens=[] if nt is None else [int(x) for x in toks.tolist()],
                               seq_len_before=int(seq_before), seq_len_after=int(eng.kv_cache.seq_len),
                               events=[[e[0], e[1]] for e in trace[mark:]]))
            print(f"[tree] round {r}: acc_count {acc}, accepted {rounds[-1]['accept_tokens']}")
            if nt is None:
                break
            nt = nt.unsqueeze(0)
    with open(os.path.join(HERE, "tree_512.json"), "w") as f:
        json.dump(dict(case=case, first_token=first, rounds=rounds), f)


def make_reference_tree():
    """The reference's tree/512.pt, re-encoded as JSON (the 512 x 512 0/1 mask as one packed-bits hex string per row)."""
    g = torch.load(os.path.join(rh.REF_ROOT, "tree", "512.pt"), weights_only=False)
    mask = g["mask"].numpy()
    assert set(np.unique(mask).tolist()) <= {0, 1}
    out = dict(size=int(g["size"]), roots=g["roots"], branches=g["branches"], Successors=g["Successors"],
               depth=[int(x) for x in g["depth"].tolist()], mask_rows=[np.packbits(row.astype(np.uint8)).tobytes().hex() for row in mask])
    with open(os.path.join(HERE, "reference_tree_512.json"), "w") as f:
        json.dump(out, f)


def make_cli_flags():
    """Every `add_argument('--flag', ...)` of the reference's three entry points: its default as written there, or store_true."""
    import re
    out = {}
    for entry in ("on_chip", "offloading_TP", "offloading_seqouia"):
        flags = []
        for flag, rest in re.findall(r"add_argument\('--(\w+)'(.*?)\)\n", open(os.path.join(rh.REF_ROOT, "test", entry + ".py")).read()):
            m = re.search(r"default=([^,)]+)", rest)
            flags.append([flag, m.group(1).strip().strip("'").strip('"') if m else None, "store_true" in rest])
        out[entry] = flags
    with open(os.path.join(HERE, "reference_cli_flags.json"), "w") as f:
        json.dump(out, f, indent=1)


def make_dataset():
    """A PG-19 sample (the first 12 books of each of the reference's jsonl files, files in sorted order, every book cut to its
    first 2000 characters) and the reference's own `get_dataset('gs')` on it with the byte tokenizer of tests/test_dataset_cpu.py.
    The reference reads the files through `datasets.load_dataset("json", data_files=[...], split="train")`; that package is
    stood in for by the rows of the given files in order (what the json builder yields for one-object-per-line files)."""
    import importlib.util
    import shutil
    import tempfile
    import types
    from test_dataset_cpu import ByteTokenizer

    src = os.path.join(rh.REF_ROOT, "data", "pg19")
    rows = []
    for name in sorted(os.listdir(src)):
        with open(os.path.join(src, name), encoding="utf-8") as f:
            books = [json.loads(line)["text"] for line in f if line.strip()]
        rows += [b[:2000] for b in books[:12]]
    sample_dir = os.path.join(HERE, "pg19_sample")
    os.makedirs(sample_dir, exist_ok=True)
    with open(os.path.join(sample_dir, "pg19-sample.json"), "w", encoding="utf-8") as f:
        for t in rows:
            f.write(json.dumps({"text": t}) + "\n")

    def load_dataset(kind, data_files, split):
        assert kind == "json" and split == "train"
        out = []
        for p in data_files:
            with open(p, encoding="utf-8") as f:
                out += [json.loads(line) for line in f if line.strip()]
        return out

    shim = types.ModuleType("datasets")
    shim.load_dataset = load_dataset
    saved, cwd = sys.modules.get("datasets"), os.getcwd()
    sys.modules["datasets"] = shim
    try:
        spec = importlib.util.spec_from_file_location("ref_dataset", os.path.join(rh.REF_ROOT, "data", "dataset.py"))
        ref = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(ref)
        with tempfile.TemporaryDirectory() as tmp:
            os.makedirs(os.path.join(tmp, "data", "pg19"))
            shutil.copy(os.path.join(sample_dir, "pg19-sample.json"), os.path.join(tmp, "data", "pg19"))
            os.chdir(tmp)  # the reference opens "data/pg19/" relative to the working directory
            got = ref.get_dataset("gs", tokenizer=ByteTokenizer())
    finally:
        os.chdir(cwd)
        if saved is None:
            sys.modules.pop("datasets")
        else:
            sys.modules["datasets"] = saved
    assert len(got) == 20 and all(t.dtype == torch.long and t.dim() == 2 and t.shape[0] == 1 for t in got)
    ids = torch.cat([t[0] for t in got]).numpy()
    assert ids.min() >= 0 and ids.max() < 2 ** 16
    np.savez_compressed(os.path.join(HERE, "dataset_gs.npz"), ids=ids.astype(np.uint16),
                        lengths=np.array([t.shape[1] for t in got], dtype=np.int64))


if __name__ == "__main__":
    which = sys.argv[1:] or ["retrieval", "sampling", "forward", "e2e", "tree", "reference_tree", "cli_flags", "dataset"]
    with torch.inference_mode():
        if "retrieval" in which:
            make_retrieval_build()
        if "sampling" in which:
            make_sampling()
        if "forward" in which:
            make_forward()
        if "e2e" in which:
            make_e2e()
        if "tree" in which:
            make_tree()
    if "reference_tree" in which:
        make_reference_tree()
    if "cli_flags" in which:
        make_cli_flags()
    if "dataset" in which:
        make_dataset()
