"""Attention kernels at the shapes and inputs where such kernels go wrong, against an fp64 reference under the fp16-rounding
bound of `attn_cases` (see there, and tests/test_attention_metric_cpu.py for why the bound catches lost tiles, causal
off-by-ones and unscaled partial merges that a fixed atol misses).  Every test prints its worst err / bound."""
import os

import numpy as np
import pytest
import torch

import attn_cases as ac
from oracle import triforce_oracle as orc
from triforce_b200 import _C, ops

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _sms() -> int:
    return torch.cuda.get_device_properties(0).multi_processor_count


def _kv_store(L, H, cap, d):
    Ks = torch.full((L, H, cap, d), ac.STALE_K, dtype=torch.float16, device=DEV)
    Vs = torch.full((L, H, cap, d), ac.STALE_V, dtype=torch.float16, device=DEV)
    return Ks, Vs


def _fill(family, layer_K, layer_V, q, R, H, d, S, scale, seed, **kw):
    return ac.make_inputs(family, R, H, d, S, layer_K.shape[1], scale, seed=seed, device=DEV,
                          out={"q": q, "K": layer_K, "V": layer_V}, **kw)


def _verify_modes(x, maps, layer, S, R, H, d, scale, ws, worst, tag, elementwise, vis=None):
    """Host length, device length (same plan: bit-identical), and kv_len_max = cache capacity (the grid a captured graph
    uses), each under the bound."""
    q = x["q"]
    ref, nz = ac.reference(q, x["K"], x["V"], scale, ac.causal_visibility(R, S, DEV) if vis is None else vis)
    out = torch.empty((R, H, d), dtype=torch.float16, device=DEV)
    ops.verify_attn(q, maps, layer, S, R, H, d, scale, out, ws)
    worst.add(ac.check(out, ref, nz, f"{tag} host", elementwise), f"{tag} host")
    out_dev = torch.zeros_like(out)
    dev_len = torch.tensor([S - R], dtype=torch.int32, device=DEV)
    ops.verify_attn(q, maps, layer, R, R, H, d, scale, out_dev, ws, kv_len_dev=dev_len, kv_len_max=S)
    assert torch.equal(out, out_dev), f"{tag}: device-side length changed the bits under the same split"
    out_cap = torch.zeros_like(out)
    ops.verify_attn(q, maps, layer, R, R, H, d, scale, out_cap, ws, kv_len_dev=dev_len)
    worst.add(ac.check(out_cap, ref, nz, f"{tag} cap", elementwise), f"{tag} cap")


# ---------------------------------------------------------------------------------------------------------------------
# verify_attn, causal
# ---------------------------------------------------------------------------------------------------------------------
# (d, R, H, S): every R in {1,2,8,16,17,31,32} (both MT instantiations) at both head dims, H in {1,2,3,4,8,12,32}, and lengths one
# tile either side of the 2 048 / 16 384 thresholds of the 8-tiles-per-CTA plan (cap = S + 70 crosses them for the graph grid)
CAUSAL_SHAPES = [(128, 1, 32, 4100), (128, 2, 2, 1984), (128, 8, 4, 2048), (128, 16, 8, 2112), (128, 17, 3, 4103),
                 (128, 31, 12, 3001), (128, 32, 1, 16320), (128, 8, 8, 16384), (128, 32, 2, 16448), (128, 8, 3, 1999),
                 (64, 1, 12, 2049), (64, 8, 3, 777), (64, 16, 4, 16383), (64, 17, 32, 1500), (64, 32, 2, 2047), (64, 31, 1, 5000),
                 (64, 2, 8, 16320), (128, 1, 1, 1)]


@pytest.mark.parametrize("d,R,H,S", CAUSAL_SHAPES, ids=[f"d{d}_R{R}_H{H}_S{S}" for d, R, H, S in CAUSAL_SHAPES])
def test_verify_attn_causal_families(d, R, H, S):
    R = min(R, S)
    cap = S + 70
    Ks, Vs = _kv_store(2, H, cap, d)  # layer 1 is attended; layer 0 keeps the stale sentinels
    maps = ops.KVTensorMaps(Ks, Vs)
    ws = ops.verify_attn_workspace(R, H, d, DEV)
    scale = orc.softmax_scale_fp16(d)
    G, _ = ac.attn_plan(R, H, d, S, _sms())
    q = torch.empty((R, H, d), dtype=torch.float16, device=DEV)
    worst = ac.Worst(f"verify_attn d={d} R={R} H={H} S={S}")
    for fi, fam in enumerate(ac.CAUSAL_FAMILIES):
        x = _fill(fam, Ks[1], Vs[1], q, R, H, d, S, scale, seed=fi * 7919 + S + R, G=G)
        _verify_modes(x, maps, 1, S, R, H, d, scale, ws, worst, fam, fam == "tile_indicator")
    worst.report()


@pytest.mark.parametrize("H", [1, 4, 32])
def test_verify_attn_every_short_length(H):
    """Every kv_len from R to 700 at every R: grids larger than the tile count (CTAs with no tile), heads split at every
    offset, and rows whose whole last tile is masked (e.g. R = 32, kv_len = 64k + 1)."""
    d, cap = 128, 768
    scale = orc.softmax_scale_fp16(d)
    Ks, Vs = _kv_store(1, H, cap, d)
    maps = ops.KVTensorMaps(Ks, Vs)
    worst = ac.Worst(f"verify_attn sweep H={H}")
    for R in (1, 2, 8, 16, 17, 31, 32):
        ws = ops.verify_attn_workspace(R, H, d, DEV)
        q = torch.empty((R, H, d), dtype=torch.float16, device=DEV)
        out = torch.empty((R, H, d), dtype=torch.float16, device=DEV)
        ratios, outs_ok = [], []
        for S in range(R, 701):
            for fam in ("tile_indicator", "diagonal"):
                x = _fill(fam, Ks[0], Vs[0], q, R, H, d, S, scale, seed=S * 31 + R)
                ref, nz = ac.reference(q, Ks[0], Vs[0], scale, ac.causal_visibility(R, S, DEV))
                ops.verify_attn(q, maps, 0, S, R, H, d, scale, out, ws)
                r = ac.bound_ratio(out, ref, nz).max()
                if fam == "tile_indicator":
                    r = torch.maximum(r, ac.bound_ratio(out, ref, nz, elementwise=True).max())
                ratios.append(r)
                outs_ok.append(torch.isfinite(out).all())
        rr = torch.stack(ratios).view(-1, 2).cpu()
        assert torch.stack(outs_ok).all(), f"R={R}: NaN/Inf output"
        k = int(rr.max(1).values.argmax())
        worst.add(float(rr.max()), f"R={R} kv_len={R + k}")
        assert float(rr.max()) <= 1.0, f"R={R} kv_len={R + k}: err/bound = {float(rr.max()):.3g} (indicator, diagonal) = {rr[k].tolist()}"
    worst.report()


def test_verify_attn_full_128k_families():
    """BASELINE cfg2 geometry (H = 32, 124 928-token prefix + 8 rows), one store allocation reused by every family."""
    R, H, d, S = 8, 32, 128, 124928 + 8
    cap = S + 56
    Ks, Vs = _kv_store(1, H, cap, d)
    maps = ops.KVTensorMaps(Ks, Vs)
    ws = ops.verify_attn_workspace(R, H, d, DEV)
    scale = orc.softmax_scale_fp16(d)
    G, _ = ac.attn_plan(R, H, d, S, _sms())
    q = torch.empty((R, H, d), dtype=torch.float16, device=DEV)
    worst = ac.Worst("verify_attn 128K")
    for fi, fam in enumerate(ac.CAUSAL_FAMILIES):
        x = _fill(fam, Ks[0], Vs[0], q, R, H, d, S, scale, seed=fi + 11, G=G)
        _verify_modes(x, maps, 0, S, R, H, d, scale, ws, worst, fam, fam == "tile_indicator")
    worst.report()


def test_verify_attn_head_sharded_families():
    """A tensor-parallel rank's share of the long store: dozens of partials per head, folded in two streams when R <= 8."""
    d = 128
    scale = orc.softmax_scale_fp16(d)
    worst = ac.Worst("verify_attn head-sharded")
    stores = {}
    for (R, H, S) in [(8, 4, 124928 + 8), (7, 2, 50000), (1, 4, 70001), (12, 4, 60000)]:
        if H not in stores:  # one store per head count, sized for the longest length
            Ks, Vs = _kv_store(1, H, 124928 + 8 + 56, d)
            stores[H] = (Ks, Vs, ops.KVTensorMaps(Ks, Vs))
        Ks, Vs, maps = stores[H]
        ws = ops.verify_attn_workspace(R, H, d, DEV)
        G, _ = ac.attn_plan(R, H, d, S, _sms())
        q = torch.empty((R, H, d), dtype=torch.float16, device=DEV)
        for fi, fam in enumerate(ac.CAUSAL_FAMILIES):
            x = _fill(fam, Ks[0], Vs[0], q, R, H, d, S, scale, seed=fi + S, G=G)
            _verify_modes(x, maps, 0, S, R, H, d, scale, ws, worst, f"R={R} H={H} S={S} {fam}", fam == "tile_indicator")
    worst.report()


@pytest.mark.parametrize("R", [7, 24, 32])
def test_verify_attn_calibrated_split_families(R):
    """Under a measured split table (table 0 for R <= 16, table 1 — one CTA per SM — for R > 16 at d = 128): every family under
    the bound, and two launches with the same table bit-identical."""
    H, d, S = 32, 128, 20000 + R
    cap = S + 64
    Ks, Vs = _kv_store(1, H, cap, d)
    maps = ops.KVTensorMaps(Ks, Vs)
    ws = ops.verify_attn_workspace(R, H, d, DEV)
    scale = orc.softmax_scale_fp16(d)
    G, tab = ac.attn_plan(R, H, d, S, _sms())
    assert tab == (1 if R > 16 else 0)
    q = torch.empty((R, H, d), dtype=torch.float16, device=DEV)
    x = _fill("random", Ks[0], Vs[0], q, R, H, d, S, scale, seed=5)
    scratch = torch.empty((R, H, d), dtype=torch.float16, device=DEV)
    ops.verify_attn_calibrate(q, maps, 0, S, R, H, d, scale, scratch, ws, rounds=2)
    assert int((ws.view(torch.int32) == G).sum()) >= 1  # a table for this grid is installed
    worst = ac.Worst(f"verify_attn calibrated R={R}")
    for fi, fam in enumerate(("tile_indicator", "diagonal", "sink_then_late_max", "needles")):
        x = _fill(fam, Ks[0], Vs[0], q, R, H, d, S, scale, seed=fi + 77, G=G)
        ref, nz = ac.reference(q, Ks[0], Vs[0], scale, ac.causal_visibility(R, S, DEV))
        out_a, out_b = torch.empty_like(scratch), torch.empty_like(scratch)
        ops.verify_attn(q, maps, 0, S, R, H, d, scale, out_a, ws)
        ops.verify_attn(q, maps, 0, S, R, H, d, scale, out_b, ws)
        assert torch.equal(out_a, out_b)
        worst.add(ac.check(out_a, ref, nz, fam, fam == "tile_indicator"), fam)
        dev_len = torch.tensor([S - R], dtype=torch.int32, device=DEV)
        out_c = torch.empty_like(scratch)
        ops.verify_attn(q, maps, 0, R, R, H, d, scale, out_c, ws, kv_len_dev=dev_len, kv_len_max=S)
        assert torch.equal(out_a, out_c)
    worst.report()


# ---------------------------------------------------------------------------------------------------------------------
# clean_keys (TMA loads before griddepcontrol.wait) and next_weights (L2 prefetch of o_proj)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("R,H,d,B", [(5, 32, 128, 4096), (17, 4, 64, 1024), (8, 8, 128, 4032)])
def test_verify_attn_clean_keys_and_prefetch_are_bit_identical(R, H, d, B):
    S = B + R
    Ks, Vs = _kv_store(1, H, S + 64, d)
    maps = ops.KVTensorMaps(Ks, Vs)
    ws = ops.verify_attn_workspace(R, H, d, DEV)
    scale = orc.softmax_scale_fp16(d)
    W = torch.randn((H * d, H * d), device=DEV).half()
    q = torch.empty((R, H, d), dtype=torch.float16, device=DEV)
    worst = ac.Worst(f"clean_keys/next_weights R={R} H={H} d={d} B={B}")
    for fi, fam in enumerate(("random", "diagonal", "sink_then_late_max")):
        x = _fill(fam, Ks[0], Vs[0], q, R, H, d, S, scale, seed=fi + B, G=ac.attn_plan(R, H, d, S, _sms())[0])
        ref, nz = ac.reference(q, Ks[0], Vs[0], scale, ac.causal_visibility(R, S, DEV))
        outs = []
        for kw in ({}, {"clean_keys": B}, {"next_weights": W}, {"clean_keys": B, "next_weights": W}):
            o = torch.empty((R, H, d), dtype=torch.float16, device=DEV)
            ops.verify_attn(q, maps, 0, S, R, H, d, scale, o, ws, **kw)
            outs.append(o)
        for o in outs[1:]:
            assert torch.equal(o, outs[0]), fam
        worst.add(ac.check(outs[0], ref, nz, fam), fam)
    worst.report()


def test_retrieval_verify_chain_under_programmatic_dependent_launch():
    """The retrieval-verify block as llama.py runs it: qkv projection -> rope_append(slot0 = budget) -> verify_attn(kv_len = budget + R,
    clean_keys = budget, next_weights = o_proj) -> o_proj, for several layers.  The predecessor of every attention launch
    writes q and the R fresh K/V rows, and the attention's producer loads the clean rows before griddepcontrol.wait: eager
    launches and a CUDA graph under the default PDL mask must give the bits of the same chain without PDL."""
    R, H, d, B, L = 5, 32, 128, 4096, 3
    hid = H * d
    S = B + R
    g = torch.Generator(device=DEV).manual_seed(21)
    Ks = torch.randn((L, H, S + 59, d), generator=g, device=DEV).half()
    Vs = torch.randn((L, H, S + 59, d), generator=g, device=DEV).half()
    maps = ops.KVTensorMaps(Ks, Vs)
    ws = ops.verify_attn_workspace(R, H, d, DEV)
    scale = orc.softmax_scale_fp16(d)
    cos, sin = (torch.from_numpy(t).to(DEV) for t in orc.rope_tables_plain(d, 8192))
    pos = torch.arange(B, B + R, dtype=torch.int32, device=DEV)
    Wqkv = [ops.WeightMap((torch.randn((3 * hid, hid), generator=g, device=DEV) * 0.02).half()) for _ in range(L)]
    Wo_t = [(torch.randn((hid, hid), generator=g, device=DEV) * 0.02).half() for _ in range(L)]
    Wo = [ops.WeightMap(w) for w in Wo_t]
    x0 = torch.randn((R, hid), generator=g, device=DEV).half()
    qs = [torch.empty((R, H, d), dtype=torch.float16, device=DEV) for _ in range(L)]
    att = [torch.empty((R, H, d), dtype=torch.float16, device=DEV) for _ in range(L)]

    def reset_fresh_rows():
        Ks[:, :, B:] = ac.STALE_K
        Vs[:, :, B:] = ac.STALE_V

    def chain():
        x = x0
        for l in range(L):
            qkv = ops.stream_linear(x, Wqkv[l])
            ops.rope_append(qkv, H, d, cos, sin, qs[l], Ks[l], Vs[l], pos_ids=pos, slot0=B)
            ops.verify_attn(qs[l], maps, l, S, R, H, d, scale, att[l], ws, clean_keys=B, next_weights=Wo_t[l])
            x = ops.stream_linear(att[l].view(R, hid), Wo[l])
        return x

    lib = _C.lib()
    try:
        lib.tf_set_pdl(0)
        reset_fresh_rows()
        want_x = chain().clone()
        want = [a.clone() for a in att]
        torch.cuda.synchronize()
        worst = ac.Worst("retrieval-verify chain")
        for l in range(L):  # the chain itself is right: every layer's attention against fp64
            ref, nz = ac.reference(qs[l], Ks[l], Vs[l], scale, ac.causal_visibility(R, S, DEV))
            worst.add(ac.check(att[l], ref, nz, f"layer {l}"), f"layer {l}")
        lib.tf_set_pdl(_C.DEFAULT_PDL_MASK)
        for rep in range(2):
            reset_fresh_rows()
            got_x = chain().clone()
            torch.cuda.synchronize()
            assert torch.equal(got_x, want_x) and all(torch.equal(a, w) for a, w in zip(att, want)), f"eager PDL run {rep}"
        reset_fresh_rows()
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            out = chain()
        for rep in range(3):
            reset_fresh_rows()
            gr.replay()
            torch.cuda.synchronize()
            assert torch.equal(out, want_x) and all(torch.equal(a, w) for a, w in zip(att, want)), f"graph replay {rep}"
        worst.report()
    finally:
        lib.tf_set_pdl(int(os.environ.get("TRIFORCE_PDL", str(_C.DEFAULT_PDL_MASK))))


# ---------------------------------------------------------------------------------------------------------------------
# tree verify: mma.sync kernel (verify_attn_tree) and the tcgen05 kernel (tree_attn_tc)
# ---------------------------------------------------------------------------------------------------------------------
TREE_SHAPES = [(1, 4, 128, 600, 32, 7), (7, 4, 128, 600, 64, 5), (32, 2, 128, 8704, 512, 200), (22, 3, 64, 390, 128, 40),
               (32, 2, 128, 1100, 512, 479), (16, 12, 64, 2100, 64, 30), (31, 32, 128, 4100, 64, 1)]


@pytest.mark.parametrize("R,H,d,S,T,row0", TREE_SHAPES, ids=[f"R{s[0]}_H{s[1]}_d{s[2]}_S{s[3]}_T{s[4]}_r{s[5]}" for s in TREE_SHAPES])
def test_verify_attn_tree_families(R, H, d, S, T, row0):
    tree = ac.random_tree(np.random.Generator(np.random.PCG64(S + R + T)), R, T, row0)
    vis = ac.tree_visibility(tree, S, DEV)
    Ks, Vs = _kv_store(1, H, S + 30, d)
    maps = ops.KVTensorMaps(Ks, Vs)
    ws = ops.verify_attn_workspace(R, H, d, DEV)
    scale = orc.softmax_scale_fp16(d)
    mask = torch.from_numpy(orc.pack_tree_mask(tree).view(np.int32)).to(DEV)
    q = torch.empty((R, H, d), dtype=torch.float16, device=DEV)
    worst = ac.Worst(f"verify_attn_tree R={R} H={H} d={d} S={S} T={T} row0={row0}")
    for fi, fam in enumerate(("tree_leak", "diagonal", "random")):
        x = _fill(fam, Ks[0], Vs[0], q, R, H, d, S, scale, seed=fi + S, own0=S - T + row0, tree=tree)
        ref, nz = ac.reference(q, Ks[0], Vs[0], scale, vis)
        out = torch.empty((R, H, d), dtype=torch.float16, device=DEV)
        ops.verify_attn_tree(q, maps, 0, S, R, H, d, scale, mask, T, out, ws)
        worst.add(ac.check(out, ref, nz, fam), fam)
        out_dev = torch.zeros_like(out)
        dev_len = torch.tensor([S - T], dtype=torch.int32, device=DEV)
        ops.verify_attn_tree(q, maps, 0, T, R, H, d, scale, mask, T, out_dev, ws, kv_len_dev=dev_len, kv_len_max=S)
        assert torch.equal(out, out_dev), fam
    worst.report()


@pytest.mark.parametrize("R,H,S,T", [(128, 2, 1024 + 128, 128), (256, 2, 3000, 256), (512, 2, 5000 + 512, 512), (128, 3, 777, 256)])
def test_tree_attn_tc_tree_leak(R, H, S, T):
    d = 128
    tree = ac.random_tree(np.random.Generator(np.random.PCG64(S + R)), R, T, 0)
    vis = ac.tree_visibility(tree, S, DEV)
    Ks, Vs = _kv_store(1, H, S + 30, d)
    maps = ops.KVTensorMaps(Ks, Vs)
    ws = ops.tree_attn_tc_workspace(R, H, S, DEV)
    scale = orc.softmax_scale_fp16(d)
    mask = torch.from_numpy(orc.pack_tree_mask(tree).view(np.int32)).to(DEV)
    q = torch.empty((R, H, d), dtype=torch.float16, device=DEV)
    worst = ac.Worst(f"tree_attn_tc R={R} H={H} S={S} T={T}")
    for fi, fam in enumerate(("tree_leak", "diagonal")):
        x = _fill(fam, Ks[0], Vs[0], q, R, H, d, S, scale, seed=fi + S, own0=S - T, tree=tree)
        ref, nz = ac.reference(q, Ks[0], Vs[0], scale, vis)
        out = torch.empty((R, H, d), dtype=torch.float16, device=DEV)
        ops.tree_attn_tc(q, maps, 0, S, R, H, d, scale, mask, T, out, ws)
        worst.add(ac.check(out, ref, nz, fam), fam)
    worst.report()


@pytest.mark.parametrize("R,H,S", [(40, 2, 333), (40, 2, 3000), (200, 3, 777), (200, 2, 3000), (1023, 1, 2500), (1023, 2, 3000), (128, 2, 129)])
def test_tree_attn_tc_causal_diagonal(R, H, S):
    """Causal mode with R < S: row i's own key dominates and the next key scores higher still (must stay invisible)."""
    d = 128
    Ks, Vs = _kv_store(1, H, S + 30, d)
    maps = ops.KVTensorMaps(Ks, Vs)
    ws = ops.tree_attn_tc_workspace(R, H, S, DEV)
    scale = orc.softmax_scale_fp16(d)
    q = torch.empty((R, H, d), dtype=torch.float16, device=DEV)
    worst = ac.Worst(f"tree_attn_tc causal R={R} H={H} S={S}")
    for fi, fam in enumerate(("diagonal", "sink_then_late_max")):
        x = _fill(fam, Ks[0], Vs[0], q, R, H, d, S, scale, seed=fi + S + R)
        ref, nz = ac.reference(q, Ks[0], Vs[0], scale, ac.causal_visibility(R, S, DEV))
        out = torch.empty((R, H, d), dtype=torch.float16, device=DEV)
        ops.tree_attn_tc(q, maps, 0, S, R, H, d, scale, None, 0, out, ws, causal=True)
        worst.add(ac.check(out, ref, nz, fam), fam)
    worst.report()


# ---------------------------------------------------------------------------------------------------------------------
# draft attention (RoPE on read)
# ---------------------------------------------------------------------------------------------------------------------
def _unrope(Kr: np.ndarray, cos: np.ndarray, sin: np.ndarray) -> np.ndarray:
    """Keys [S,H,d] whose RoPE at positions 0..S-1 is (up to fp16 rounding) Kr: the inverse rotation, in fp64."""
    S = Kr.shape[0]
    c = cos[:S].astype(np.float64)[:, None, :]
    s = sin[:S].astype(np.float64)[:, None, :]
    y = Kr.astype(np.float64)
    return (y * c - orc.rotate_half(y) * s).astype(np.float16)


@pytest.mark.parametrize("H,d,R,kv_len", [(12, 64, 1, 253), (12, 64, 7, 259), (12, 64, 48, 64), (12, 64, 40, 600), (12, 64, 64, 300),
                                          (4, 128, 5, 300), (2, 128, 33, 355), (3, 128, 16, 17)])
def test_draft_attn_families(H, d, R, kv_len):
    """The draft's StreamingLLM window (68M: H = 12, d = 64, and d = 128) with its 16 zero sink rows: the families are built in
    the rotated key space and stored un-rotated, so the kernel's RoPE-on-read must land on them."""
    cos, sin = orc.rope_tables_plain(d, 2048)
    scale = orc.softmax_scale_fp16(d)
    worst = ac.Worst(f"draft_attn H={H} d={d} R={R} kv_len={kv_len}")
    t = lambda a: torch.from_numpy(a).to(DEV)
    for fi, fam in enumerate(("diagonal", "sink_then_late_max")):
        x = ac.make_inputs(fam, R, H, d, kv_len, kv_len, scale, seed=fi + kv_len + R, sink=16)
        q = x["q"].numpy()
        K = _unrope(x["K"].permute(1, 0, 2).numpy(), cos, sin)
        V = x["V"].permute(1, 0, 2).numpy().copy()
        K[:16] = 0  # zero sinks (the reference's reset quirk)
        V[:16] = 0
        Kr = orc.apply_rope(K, cos, sin, np.arange(kv_len))  # what the kernel attends to
        Ks = torch.zeros((H, kv_len + 5, d), dtype=torch.float16, device=DEV)
        Vs = torch.zeros_like(Ks)
        Ks[:, :kv_len] = t(K).permute(1, 0, 2)
        Vs[:, :kv_len] = t(V).permute(1, 0, 2)
        Ks[:, kv_len:] = ac.STALE_K
        Vs[:, kv_len:] = ac.STALE_V
        ref, nz = ac.reference(t(q), t(Kr).permute(1, 0, 2), t(V).permute(1, 0, 2), scale, ac.causal_visibility(R, kv_len, DEV))
        out = torch.empty((R, H, d), dtype=torch.float16, device=DEV)
        ops.draft_attn(t(q), Ks, Vs, t(cos), t(sin), kv_len, scale, out)
        worst.add(ac.check(out, ref, nz, fam), fam)
    worst.report()
