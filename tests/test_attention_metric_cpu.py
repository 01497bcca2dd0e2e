"""Evidence for the attention metric of `attn_cases`, without a GPU.

A numpy model of tf_verify_attn's algorithm — 64-key tiles, an equal split of the tile axis over G CTAs, a per-CTA partial
(m, l, O) in fp32 with P rounded to fp16 before P.V, and the ordered merge of the partials — is run on every input family.
The correct model must stay 3x under the bound (this is what fixes C_BOUND); each bug that such a kernel typically has,
switched on in the model, must exceed the bound on at least one family at every shape, and the causal off-by-one must be
caught at the 128K shape of the 7B target."""
import numpy as np
import pytest
import torch

import attn_cases as ac
from oracle import triforce_oracle as orc

SMS = 148  # B200
CAUSAL_BUGS = ("drop_tile", "dup_tile", "causal_minus_1", "causal_plus_1", "no_rescale")
TREE_BUGS = ("drop_tile", "dup_tile", "no_rescale", "tree_leak")

# (name, R, d, S): one head; G from the kernel's plan for that shape (296, 8, 11, 3 CTAs)
CAUSAL_SHAPES = [("128k", 8, 128, 124936), ("4k", 8, 128, 4103), ("700", 8, 64, 700), ("130", 4, 64, 130)]
# (name, R, d, S, T, row0)
TREE_SHAPES = [("tree_128k", 32, 128, 124936, 512, 300), ("tree_8k", 32, 128, 8704, 512, 200), ("tree_390", 22, 64, 390, 128, 40)]


def model_verify_attn(q, K, V, scale, vis_kernel, G, bug=None):
    """q [R,d], K/V [S,d] fp16, vis_kernel bool [R,S] (the mask the kernel applies).  Returns fp16 [R,d]."""
    R, d = q.shape
    S = K.shape[0]
    ranges = ac.cta_tile_ranges(S, 1, G)
    if bug in ("drop_tile", "dup_tile"):
        b = len(ranges) // 2
        t = ranges[b][0]
        if bug == "drop_tile":
            ranges[b] = (t + 1, ranges[b][1])
        else:
            ranges[b - 1] = (ranges[b - 1][0], t + 1)
    l2e = np.float32(1.4426950408889634)
    sl2 = np.float32(scale) * l2e
    with np.errstate(invalid="ignore", over="ignore"):
        s = q.astype(np.float32) @ K.astype(np.float32).T
        s = np.where(vis_kernel, s * sl2, np.float32(-np.inf)).astype(np.float32)
        V32 = V.astype(np.float32)
        mr = np.full((R, 1), -np.inf, np.float32)
        acc = np.zeros((R, d), np.float32)
        den = np.zeros((R, 1), np.float32)
        for (t0, t1) in ranges:
            k0, k1 = t0 * ac.BN, min(t1 * ac.BN, S)
            if k1 <= k0:
                continue
            sc = s[:, k0:k1]
            m = sc.max(-1, keepdims=True)
            mu = np.where(m == -np.inf, np.float32(0), m)
            p = np.exp2(sc - mu).astype(np.float32)
            l = p.sum(-1, keepdims=True, dtype=np.float32)
            o = p.astype(np.float16).astype(np.float32) @ V32[k0:k1]
            mn = np.maximum(mr, m)
            mnu = np.where(mn == -np.inf, np.float32(0), mn)
            a = np.exp2(mr - mnu).astype(np.float32)
            if bug == "no_rescale":
                a = np.ones_like(a)
            w = np.exp2(m - mnu).astype(np.float32)
            acc = (w * o + acc * a).astype(np.float32)
            den = (w * l + den * a).astype(np.float32)
            mr = mn
        return (acc / den).astype(np.float16)


def _family_inputs(family, R, d, S, scale, own0, G, tree=None):
    x = ac.make_inputs(family, R, 1, d, S, S, scale, seed=1000 + S + R, own0=own0, G=G, tree=tree)
    return x["q"][:, 0].numpy(), x["K"][0].numpy(), x["V"][0].numpy()


def _ratio(out, ref, nz, elementwise):
    r = float(ac.bound_ratio(out, ref, nz).max())
    if elementwise:
        r = max(r, float(ac.bound_ratio(out, ref, nz, elementwise=True).max()))
    return r


def _run_shape(families, bugs, R, d, S, vis, own0, G, tree=None, bug_vis=None):
    scale = orc.softmax_scale_fp16(d)
    table = {}
    for fam in families:
        q, K, V = _family_inputs(fam, R, d, S, scale, own0, G, tree)
        assert np.isfinite(q.astype(np.float32)).all() and np.isfinite(K.astype(np.float32)).all()
        ref, nz = ac.reference_np(q[:, None], K[None], V[None], scale, vis)
        ref, nz = ref[:, 0], nz[:, 0]
        el = fam == "tile_indicator"
        table[(fam, None)] = _ratio(model_verify_attn(q, K, V, scale, vis, G), ref, nz, el)
        for bug in bugs:
            vk = bug_vis(bug, q, K) if bug_vis is not None else None
            out = model_verify_attn(q, K, V, scale, vis if vk is None else vk, G, bug=None if vk is not None else bug)
            table[(fam, bug)] = _ratio(out, ref, nz, el)
    for fam in families:
        print(f"  {fam:20s} correct {table[(fam, None)]:.3f}  " + "  ".join(f"{b} {table[(fam, b)]:.3g}" for b in bugs))
    return table


@pytest.mark.parametrize("name,R,d,S", CAUSAL_SHAPES, ids=[s[0] for s in CAUSAL_SHAPES])
def test_metric_separates_correct_from_buggy_causal_verify(name, R, d, S):
    G, _ = ac.attn_plan(R, 1, d, S, SMS)
    vis = ac.causal_visibility(R, S).numpy()

    def bug_vis(bug, q, K):
        delta = {"causal_minus_1": -1, "causal_plus_1": 1}.get(bug)
        if delta is None:
            return None
        return np.arange(S)[None, :] <= S - R + np.arange(R)[:, None] + delta

    print(f"\n{name}: R={R} d={d} S={S} G={G}")
    t = _run_shape(ac.CAUSAL_FAMILIES, CAUSAL_BUGS, R, d, S, vis, S - R, G, bug_vis=bug_vis)
    for fam in ac.CAUSAL_FAMILIES:
        assert t[(fam, None)] <= 1 / 3, f"correct model at {t[(fam, None)]:.3f} of the bound on {fam}: C_BOUND too small"
    for bug in CAUSAL_BUGS:
        caught = [fam for fam in ac.CAUSAL_FAMILIES if t[(fam, bug)] > 1.0]
        assert caught, f"{bug} passes every family at {name}"
    if name == "128k":
        assert t[("diagonal", "causal_minus_1")] > 1 and t[("diagonal", "causal_plus_1")] > 1


@pytest.mark.parametrize("name,R,d,S,T,row0", TREE_SHAPES, ids=[s[0] for s in TREE_SHAPES])
def test_metric_separates_correct_from_buggy_tree_verify(name, R, d, S, T, row0):
    G, _ = ac.attn_plan(R, 1, d, S, SMS)
    tree = ac.random_tree(np.random.Generator(np.random.PCG64(S + T)), R, T, row0)
    vis = ac.tree_visibility(tree, S).numpy()

    def bug_vis(bug, q, K):
        if bug != "tree_leak":
            return None
        # one column leaks to every row: the hidden tree column that row 0 scores highest
        s0 = q[0].astype(np.float32) @ K[S - T:].astype(np.float32).T
        s0[tree[0]] = -np.inf
        leak = vis.copy()
        leak[:, S - T + int(s0.argmax())] = True
        return leak

    families = ("random", "diagonal", "tree_leak")
    print(f"\n{name}: R={R} d={d} S={S} T={T} row0={row0} G={G}")
    t = _run_shape(families, TREE_BUGS, R, d, S, vis, S - T + row0, G, tree=tree, bug_vis=bug_vis)
    for fam in families:
        assert t[(fam, None)] <= 1 / 3, f"correct model at {t[(fam, None)]:.3f} of the bound on {fam}"
    for bug in TREE_BUGS:
        assert any(t[(fam, bug)] > 1.0 for fam in families), f"{bug} passes every family at {name}"
    assert t[("tree_leak", "tree_leak")] > 1.0


def test_split_model_covers_the_tile_axis():
    """The Python split model: CTA ranges tile the (head, tile) axis exactly, in order, with the min-tiles rule of attn_plan."""
    assert ac.attn_plan(8, 32, 128, 124936, SMS) == (296, 0)
    assert ac.attn_plan(24, 32, 128, 124936, SMS) == (148, 1)
    assert ac.attn_plan(7, 3, 128, 4103, SMS) == (3 * 65 // 8, 0)       # 8 tiles per CTA: H <= 8, 2048 <= kv_len_max < 16384
    assert ac.attn_plan(7, 3, 128, 16384, SMS) == (296, 0)
    assert ac.attn_plan(7, 3, 128, 2047, SMS) == (3 * 32, 0)
    for S, H, G in [(124936, 32, 296), (700, 4, 296), (4103, 3, 24), (65, 1, 296), (1, 1, 296)]:
        rngs = ac.cta_tile_ranges(S, H, G)
        tph = (S + 63) // 64
        assert rngs[0][0] == 0 and rngs[-1][1] == H * tph
        assert all(a[1] == b[0] and a[0] < a[1] for a, b in zip(rngs, rngs[1:]))
        per_head = ac.head_key_ranges(S, H, G)
        for h in range(H):
            keys = [k for lo, hi in per_head[h] for k in range(lo, hi)]
            assert keys == list(range(S))
