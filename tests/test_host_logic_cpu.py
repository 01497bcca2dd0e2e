"""Host-side logic that needs no GPU: configs, noise sources, drop-in import paths, and the tensor-parallel sharding
algebra under a real 2-process `gloo` group (the N>1 path of bench.py / test/offloading_TP.py uses the same shard
function and the same all-reduce seams over NCCL)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from triforce_b200.config import LlamaShape, named_config
from triforce_b200.llama import shard_layer_weights
from triforce_b200.rng import CounterNoise
from triforce_b200.synth import numpy_prompt, numpy_state_dict
from triforce_b200.tp import shard_bounds

REPO = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def test_named_configs_match_reference_geometry():
    c = named_config("llama-7B-128K")
    assert (c.num_hidden_layers, c.num_attention_heads, c.head_dim, c.vocab_size) == (32, 32, 128, 32000)
    assert c.kv_bytes_per_token_layer() == 16384  # SURVEY §8d
    assert 6.5e9 < c.param_count() < 7.0e9
    assert named_config("llama-13B-128K").kv_bytes_per_token_layer() == 20480
    with pytest.raises(ValueError, match="MHA-only"):
        LlamaShape(num_attention_heads=32, num_key_value_heads=8)


def test_counter_noise_is_replayable_and_rewindable():
    a, b = CounterNoise(5), CounterNoise(5)
    ea, ua = a.exponential(1000), a.uniform()
    assert np.array_equal(ea, b.exponential(1000)) and ua == b.uniform()
    mark = a.mark()
    blk = [a.uniform() for _ in range(4)]
    a.rewind(mark, 2)  # only two of the four uniforms were really examined
    assert a.uniform() == blk[2]
    assert (ea > 0).all() and 0.0 <= ua < 1.0


def test_synthetic_inputs_are_stable():
    p = numpy_prompt(64, seed=3)
    assert p.shape == (1, 64) and p.dtype == torch.int64
    assert p[0, :4].tolist() == numpy_prompt(64, seed=3)[0, :4].tolist()
    sd = numpy_state_dict(named_config("llama-68M"), 2)
    assert sd["model.layers.0.self_attn.q_proj.weight"].shape == (768, 768)
    assert abs(float(sd["lm_head.weight"].float().std()) - 0.02) < 1e-3


def test_drop_in_import_paths():
    code = ("import models.cache as c, utils.decoding as d, utils.sampling as s, utils.graph_infer as g, models.TP_llama as t;"
            "assert all(hasattr(c, n) for n in ('FlashSimpleCache', 'RetrievalCache', 'StreamingLLMEvictionCache'));"
            "assert all(hasattr(d, n) for n in ('Autoregressive', 'TriForce', 'Middle_Spec', 'Baseline_Dist', 'TriForce_Dist', 'Middle_Spec_Dist'));"
            "assert all(hasattr(s, n) for n in ('norm_logits', 'sample', 'max_fn'));"
            "assert hasattr(g, 'GraphInferenceEngine') and hasattr(t, 'DistributedLlama') and hasattr(t, 'distributed_init');"
            "import inspect; sig = inspect.signature(d.TriForce);"
            "assert list(sig.parameters)[:8] == ['tokenizer', 'graph_engine', 'input_ids', 'gamma', 'max_len', 'top_k', 'top_p', 'temperature']")
    subprocess.check_call([sys.executable, "-c", code], cwd=REPO)


def test_product_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under triforce_b200/, models/, utils/, test/ may import it."""
    bad = []
    for root in ("triforce_b200", "models", "utils", "test"):
        for dp, _, files in os.walk(os.path.join(REPO, root)):
            for f in files:
                if f.endswith(".py"):
                    src = open(os.path.join(dp, f)).read()
                    if "import oracle" in src or "from oracle" in src:
                        bad.append(os.path.join(dp, f))
    assert not bad, bad


def test_shard_bounds():
    assert shard_bounds(32, 3, 8) == (12, 16)
    with pytest.raises(ValueError):
        shard_bounds(40, 0, 16)


def _tp_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        cfg = named_config("llama-68M")
        sd = {k: v.float() for k, v in numpy_state_dict(cfg, 7).items()}
        H, d, inter = cfg.num_attention_heads, cfg.head_dim, cfg.intermediate_size
        wqkv, wo, wgu, wd = shard_layer_weights(sd, cfg, 1, rank, world)
        Hl = H // world
        assert wqkv.shape == (3 * Hl * d, cfg.hidden_size) and wo.shape == (cfg.hidden_size, Hl * d)
        g = torch.Generator().manual_seed(0)
        x = torch.randn(5, cfg.hidden_size, generator=g)
        # attention seam: local heads → row-parallel o_proj → all-reduce (tensor_op.py:176-179)
        qkv = x @ wqkv.T
        attn_local = torch.tanh(qkv[:, :Hl * d])  # any per-head function of the local q/k/v
        o = attn_local @ wo.T
        dist.all_reduce(o)
        # MLP seam (tensor_op.py:353-359)
        gu = x @ wgu.T
        act = torch.nn.functional.silu(gu[:, :inter // world]) * gu[:, inter // world:]
        dn = act @ wd.T
        dist.all_reduce(dn)
        p = "model.layers.1."
        q_full = torch.tanh(x @ sd[p + "self_attn.q_proj.weight"].T)
        o_full = q_full @ sd[p + "self_attn.o_proj.weight"].T
        dn_full = (torch.nn.functional.silu(x @ sd[p + "mlp.gate_proj.weight"].T) * (x @ sd[p + "mlp.up_proj.weight"].T)) @ sd[p + "mlp.down_proj.weight"].T
        ok = torch.allclose(o, o_full, atol=1e-4) and torch.allclose(dn, dn_full, atol=1e-4)
        # replicated sampling: identical seeds → identical draws on every rank, no broadcast needed
        draws = torch.tensor([float(CounterNoise(11).uniform())])
        gathered = [torch.zeros(1) for _ in range(world)]
        dist.all_gather(gathered, draws)
        ok = ok and all(float(t) == float(draws) for t in gathered)
        out[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


def test_tensor_parallel_sharding_with_gloo_world_size_2():
    world = 2
    with mp.Manager() as m:
        out = m.dict()
        mp.spawn(_tp_worker, args=(world, 29517 + os.getpid() % 200, out), nprocs=world, join=True)
        assert dict(out) == {0: True, 1: True}


# ---------------------------------------------------------------------------------------------------------------------
# Sequoia tree host logic (SURVEY §8 row a18) — everything here runs without a GPU
# ---------------------------------------------------------------------------------------------------------------------
def test_grow_map_matches_the_reference_tree_file_and_the_oracle_mask_packing():
    from oracle import triforce_oracle as orc
    from triforce_b200.spectree import load_grow_map, pack_mask_bits

    gm = load_grow_map("512")
    assert gm["size"] == 512 and [len(r) for r in gm["roots"]] == [1, 7, 14, 22, 31, 30, 31, 29, 33, 37, 41, 45, 49, 53, 43, 46]
    mask = gm["mask"].numpy().astype(bool)
    # structural invariants SpecTree relies on: every node sees itself, only earlier nodes, and all ancestors of its parent
    assert mask.shape == (512, 512) and mask.diagonal().all() and not np.triu(mask, 1).any()
    parent = {}
    for n, children in enumerate(gm["Successors"]):
        for c in children:
            assert c > n and c not in parent
            parent[c] = n
    assert sorted(parent) == list(range(1, 512))
    for c, p in parent.items():
        want = mask[p].copy()
        want[c] = True
        assert np.array_equal(mask[c], want), f"node {c} must see exactly itself and what its parent {p} sees"
        assert int(gm["depth"][c]) == int(gm["depth"][p]) + 1
    bits = pack_mask_bits(gm["mask"]).numpy().view(np.uint32)
    np.testing.assert_array_equal(bits, orc.pack_tree_mask(mask))
    # the JSON is a re-encoding of the reference's tree/512.pt, whose contents tests/golden/reference_tree_512.json holds
    g = json.load(open(os.path.join(REPO, "tests", "golden", "reference_tree_512.json")))
    g["mask"] = torch.from_numpy(np.stack([np.unpackbits(np.frombuffer(bytes.fromhex(r), np.uint8))[:g["size"]] for r in g.pop("mask_rows")]).astype(np.int64))
    assert g["size"] == gm["size"] and g["roots"] == gm["roots"] and g["branches"] == gm["branches"]
    assert g["Successors"] == gm["Successors"]
    assert torch.equal((g["mask"] == 0) if g["mask"].dtype != torch.bool else g["mask"], gm["mask"].bool()) or \
        torch.equal(g["mask"].bool(), gm["mask"].bool())


def test_tree_sampling_tables_match_the_restated_script_helpers():
    """spectree.build_sampling (device-agnostic) == the helpers of test/offloading_seqouia.py:119-133 as restated in the
    reference harness; sampling without replacement picks the same positions on the same noise."""
    from oracle import ref_tree_harness as th
    from triforce_b200.spectree import build_sampling, load_grow_map

    gm = load_grow_map("512")
    mine_c, mine_g = build_sampling(gm, 0.6, "cpu")
    ref_c, ref_g = th.build_sampling(gm, 0.6)
    assert sorted(mine_g) == sorted(ref_g)
    g = torch.Generator().manual_seed(0)
    for i in mine_g:
        assert torch.equal(mine_g[i].cpu(), ref_g[i])
        rows = len(gm["branches"][i])
        logits = torch.randn((rows, 4096), generator=g)
        rand = torch.rand((rows, 4096), generator=g).clamp_(6.1e-5, 0.9994)
        assert torch.equal(mine_c[i](logits, rand), ref_c[i](logits, rand))


def test_tree_noise_is_replayable_and_never_one():
    a, b = CounterNoise(21), CounterNoise(21)
    ua = a.tree_uniform((64, 1000))
    assert ua.dtype == np.float16 and float(ua.max()) < 1.0 and float(ua.min()) > 0.0
    out = torch.empty((64, 1000), dtype=torch.float16)
    b.tree_uniform_into(out)
    assert np.array_equal(out.numpy(), ua)
    # the lazily consumed uniforms of the accept walk: draw a block, rewind to what was examined
    m = a.mark()
    blk = torch.empty(16)
    a.uniform_block_into(blk)
    a.rewind(m, 3)
    b.mark()
    firsts = [float(b.uniform()) for _ in range(4)]
    assert np.allclose(blk[:3].numpy(), firsts[:3]) and float(a.uniform()) == firsts[3]


def test_entry_points_keep_the_reference_command_line():
    """test/on_chip.py, test/offloading_TP.py, test/offloading_seqouia.py: every flag of the reference with the reference's
    default (checked against the flags of the reference's own argparse blocks, stored in tests/golden/reference_cli_flags.json)."""
    from triforce_b200 import cli

    ref_flags = json.load(open(os.path.join(REPO, "tests", "golden", "reference_cli_flags.json")))
    for entry in ("on_chip", "offloading_TP", "offloading_seqouia"):
        ns = vars(cli.build_parser(entry).parse_args([]))
        assert ns["prefill"] in (32768, 130048) and ns["temp"] == 0.6 and ns["top_p"] == 0.9
        script = os.path.join(REPO, "test", entry + ".py")
        out = subprocess.run([sys.executable, script, "--help"], capture_output=True, text=True, timeout=120)
        assert out.returncode == 0 and "--prefill" in out.stdout  # parses its flags without touching CUDA
        assert len(ref_flags[entry]) >= 12
        for flag, want, store_true in ref_flags[entry]:
            assert flag in ns, f"{entry}: flag --{flag} of the reference is missing"
            if want is not None:
                assert str(ns[flag]) == want, f"{entry}: --{flag} default {ns[flag]!r} != reference {want!r}"
            elif store_true:
                assert ns[flag] is False


def test_from_pretrained_reads_a_local_checkpoint_directory(tmp_path):
    """ADVICE r1: a local HF directory (what --target_path / --draft_path pass) resolves its shape from config.json and loads
    its safetensors; a name that is neither a directory nor explicitly synthetic raises instead of silently going random."""
    import json

    import pytest
    import torch
    from safetensors.torch import save_file

    from triforce_b200.config import LlamaShape
    from triforce_b200.hf_compat import DraftLlamaForCausalLM, TargetLlamaForCausalLM, shape_from_hf_config
    from triforce_b200.synth import numpy_state_dict

    shape = LlamaShape(hidden_size=64, intermediate_size=128, num_hidden_layers=2, num_attention_heads=4, vocab_size=96,
                       max_position_embeddings=512, rms_norm_eps=1e-6,
                       rope_scaling={"type": "yarn", "factor": 2.0, "original_max_position_embeddings": 256})
    sd = numpy_state_dict(shape, seed=5)
    d = tmp_path / "ckpt"
    d.mkdir()
    save_file({k: v.contiguous() for k, v in sd.items()}, str(d / "model.safetensors"))
    json.dump({"hidden_size": 64, "intermediate_size": 128, "num_hidden_layers": 2, "num_attention_heads": 4, "num_key_value_heads": 4,
               "vocab_size": 96, "max_position_embeddings": 512, "rms_norm_eps": 1e-6, "rope_theta": 10000.0,
               "rope_scaling": {"type": "yarn", "factor": 2.0, "original_max_position_embeddings": 256}}, open(d / "config.json", "w"))
    got = shape_from_hf_config(str(d))
    assert (got.hidden_size, got.num_hidden_layers, got.head_dim, got.vocab_size) == (64, 2, 16, 96)
    assert got.rope_scaling == shape.rope_scaling
    m = TargetLlamaForCausalLM.from_pretrained(str(d), torch_dtype=torch.float16, device_map="cpu")
    assert torch.equal(m.lm_head, sd["lm_head.weight"]) and torch.equal(m.layers[1].wo, sd["model.layers.1.self_attn.o_proj.weight"])
    assert m.layers[0].wqkv.shape == (3 * 64, 64) and not m.is_draft
    json.dump({"hidden_size": 64, "intermediate_size": 128, "num_hidden_layers": 2, "num_attention_heads": 4, "vocab_size": 96,
               "rope_scaling": {"rope_type": "default"}}, open(d / "config.json", "w"))
    assert DraftLlamaForCausalLM.from_pretrained(str(d), device_map="cpu").is_draft  # transformers-5 style "no scaling"
    with pytest.raises(FileNotFoundError):
        TargetLlamaForCausalLM.from_pretrained("NousResearch/Yarn-Llama-2-7b-128k", device_map="cpu")
    with pytest.raises(KeyError):
        TargetLlamaForCausalLM.from_pretrained("no/such-model", device_map="cpu", synthetic=True)


def test_ncu_summary_tool_reads_the_committed_capture(tmp_path):
    """tools/ncu_summary.py on the committed raw table of the round's `ncu --set full` capture: DRAM traffic of the full-KV
    attention = the algorithmic bytes to within half a percent, and the committed summary says the same."""
    import json
    import subprocess
    import sys
    repo = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
    raw = os.path.join(repo, "profiles", "r02_verify_attn_ncu_full_raw.csv.gz")
    out = tmp_path / "s.json"
    r = subprocess.run([sys.executable, os.path.join(repo, "tools", "ncu_summary.py"), raw, "--kernel", "verify_attn_mma_kernel", "--kv_len", "124936",
                        "--rows", "8", "--heads", "32", "--out", str(out)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr[-500:]
    got = json.load(open(out))
    committed = json.load(open(os.path.join(repo, "profiles", "r02_verify_attn_ncu_full.json")))
    assert got["algorithmic_bytes"] == committed["algorithmic_bytes"] == 124936 * 32 * 128 * 2 * 2
    assert len(got["launches"]) == len(committed["launches"]) == 2
    for a, b in zip(got["launches"], committed["launches"]):
        assert a["dram_bytes"] == b["dram_bytes"]
        assert 1.0 <= a["traffic_over_algorithmic"] < 1.005
        assert 250 < a["gpu__time_duration.sum"] < 400  # microseconds
