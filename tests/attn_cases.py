"""Shared pieces of the attention tests: an fp64 reference, an error bound tied to fp16 rounding, input families that each
aim at one way an attention kernel goes wrong, and a Python model of how `tf_verify_attn` splits its work over CTAs.

Why not a fixed atol: with standard-normal q, K, V the softmax is nearly uniform, so at long context the output is the mean
of ~10^5 random rows (RMS ~4e-3) and every key carries ~1/S of it.  A lost 64-key tile or a causal limit that is off by one
then moves the output by less than any fixed tolerance that the correct kernel also passes.  The families below make single
keys (or single tiles) carry O(1) of the output, and the bound scales with what fp16 rounding can actually do:

    ||got - ref||_2  <=  c * u16 * (||ref||_2 + n_r) + tiny,     n_r = sqrt(sum_j p_rj^2 * ||v_j||^2),   u16 = 2^-11

per (row, head).  ||ref|| covers the final rounding of the output to fp16; n_r covers rounding each probability to fp16
before the P.V product (independent relative errors of size ~u16 on every term p_rj v_j).  `tests/test_attention_metric_cpu.py`
fixes c on a numpy model of the kernel's algorithm and shows that every modelled bug exceeds the bound.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch

U16 = 2.0 ** -11
C_BOUND = 4.0
TINY = 1e-6
BN = 64                  # keys per tile of tf_verify_attn (TF_VERIFY_BOX_KEYS)
STALE_K, STALE_V = 77.0, -55.0  # rows past kv_len: a kernel that reads them moves the output far outside the bound

CAUSAL_FAMILIES = ("random", "tile_indicator", "diagonal", "sink_then_late_max", "large_magnitude", "needles")

# score gaps (nats, after the softmax scale) of the needle-style families
GAP_OWN, GAP_NEXT = 16.0, 20.8      # diagonal: own key, and the next key that the row must not see
GAP_SINK, GAP_LATE = 30.0, 40.0     # sink_then_late_max
GAP_NEEDLE = 16.0                   # needles, tree_leak


# ---------------------------------------------------------------------------------------------------------------------
# visibility
# ---------------------------------------------------------------------------------------------------------------------
def causal_visibility(R: int, S: int, device="cpu") -> torch.Tensor:
    """bool [R, S]: bottom-right causal, row i sees key j iff j <= S - R + i."""
    i = torch.arange(R, device=device)[:, None]
    j = torch.arange(S, device=device)[None, :]
    return j <= S - R + i


def tree_visibility(vis_tree: np.ndarray, S: int, device="cpu") -> torch.Tensor:
    """bool [R, S]: the first S - T keys are visible to every row, the last T follow the ancestor mask [R, T]."""
    R, T = vis_tree.shape
    out = torch.ones((R, S), dtype=torch.bool, device=device)
    out[:, S - T:] = torch.from_numpy(np.ascontiguousarray(vis_tree)).to(device)
    return out


def random_tree(rng: np.random.Generator, R: int, T: int, row0: int) -> np.ndarray:
    """Ancestor-closed visibility like grow_map["mask"]: node n sees itself and a random chain of earlier nodes."""
    vis = np.zeros((R, T), dtype=bool)
    for i in range(R):
        n = row0 + i
        vis[i, n] = True
        p = n
        while p > 0:
            p = int(rng.integers(0, p))
            vis[i, p] = True
    return vis


# ---------------------------------------------------------------------------------------------------------------------
# reference + metric
# ---------------------------------------------------------------------------------------------------------------------
def reference(q: torch.Tensor, K: torch.Tensor, V: torch.Tensor, scale: float, vis: torch.Tensor):
    """fp64 attention from the same fp16 inputs.  q [R,H,d]; K, V head-major [H, >=S, d] (S = vis.shape[1]); vis bool [R,S].
    Returns (out [R,H,d], noise_elem [R,H,d]) in float64; noise_elem[r,h,c] = sqrt(sum_j p_rj^2 V_jc^2)."""
    R, H, d = q.shape
    S = vis.shape[1]
    neg = ~vis.to(q.device)
    if H * S * (d + R) <= (1 << 24):  # small: all heads in one batch
        Vd = V[:, :S].double()
        s = torch.einsum("rhd,hsd->hrs", q.double(), K[:, :S].double()) * scale
        s.masked_fill_(neg[None], -math.inf)
        p = torch.softmax(s, dim=-1)
        out = torch.einsum("hrs,hsd->rhd", p, Vd)
        nz = torch.einsum("hrs,hsd->rhd", p * p, Vd * Vd).sqrt()
        return out, nz
    out = torch.empty((R, H, d), dtype=torch.float64, device=q.device)
    nz = torch.empty_like(out)
    for h in range(H):
        Vh = V[h, :S].double()
        s = (q[:, h].double() @ K[h, :S].double().T) * scale
        s.masked_fill_(neg, -math.inf)
        p = torch.softmax(s, dim=-1)
        out[:, h] = p @ Vh
        nz[:, h] = ((p * p) @ (Vh * Vh)).sqrt()
    return out, nz


def reference_np(q: np.ndarray, K: np.ndarray, V: np.ndarray, scale: float, vis: np.ndarray):
    """numpy float64 version of `reference` for the CPU model: q [R,H,d], K/V [H,S,d], vis [R,S]."""
    R, H, d = q.shape
    out = np.empty((R, H, d))
    nz = np.empty((R, H, d))
    for h in range(H):
        Vh = V[h].astype(np.float64)
        s = (q[:, h].astype(np.float64) @ K[h].astype(np.float64).T) * scale
        s = np.where(vis, s, -np.inf)
        s -= s.max(-1, keepdims=True)
        p = np.exp(s)
        p /= p.sum(-1, keepdims=True)
        out[:, h] = p @ Vh
        nz[:, h] = np.sqrt((p * p) @ (Vh * Vh))
    return out, nz


def bound_ratio(got, ref, noise_elem, c: float = C_BOUND, elementwise: bool = False):
    """err / bound per (row, head) — or per element with `elementwise` — as float64 (torch or numpy, like the inputs)."""
    if isinstance(got, torch.Tensor):
        diff = got.double() - ref
        if elementwise:
            return diff.abs() / (c * U16 * (ref.abs() + noise_elem) + TINY)
        err = diff.norm(dim=-1)
        return err / (c * U16 * (ref.norm(dim=-1) + noise_elem.norm(dim=-1)) + TINY)
    diff = got.astype(np.float64) - ref
    if elementwise:
        return np.abs(diff) / (c * U16 * (np.abs(ref) + noise_elem) + TINY)
    return np.linalg.norm(diff, axis=-1) / (c * U16 * (np.linalg.norm(ref, axis=-1) + np.linalg.norm(noise_elem, axis=-1)) + TINY)


def check(got: torch.Tensor, ref: torch.Tensor, noise_elem: torch.Tensor, what: str, elementwise: bool = False) -> float:
    """Asserts finite output within the bound; returns the worst err / bound (the per-row ratio, and for `elementwise`
    families also the per-element one)."""
    assert torch.isfinite(got).all(), f"{what}: NaN/Inf in the output"
    r = bound_ratio(got, ref, noise_elem)
    worst = float(r.max())
    if elementwise:
        worst = max(worst, float(bound_ratio(got, ref, noise_elem, elementwise=True).max()))
    if worst > 1.0:
        idx = np.unravel_index(int(r.argmax()), tuple(r.shape))
        raise AssertionError(f"{what}: err/bound = {worst:.3g} (worst row, head = {tuple(int(x) for x in idx)}); "
                             f"|ref| there = {float(ref[idx].norm()):.4g}")
    return worst


class Worst:
    """Collects the worst ratio of a test and prints it (shown with pytest -s)."""

    def __init__(self, name: str):
        self.name, self.value, self.where = name, 0.0, ""

    def add(self, ratio: float, where: str):
        if ratio >= self.value:
            self.value, self.where = ratio, where

    def report(self):
        print(f"[attn-metric] {self.name}: worst err/bound = {self.value:.4f} at {self.where}")


# ---------------------------------------------------------------------------------------------------------------------
# split model of tf_verify_attn (attn_plan + split_start, equal split)
# ---------------------------------------------------------------------------------------------------------------------
def attn_plan(R: int, H: int, d: int, kv_len_max: int, sm_count: int) -> Tuple[int, int]:
    """(grid G, split-table index) of verify_attn.cu:attn_plan."""
    slots_max = 2 * sm_count
    min_tiles = 8 if (H <= 8 and 2048 <= kv_len_max < 16384) else 1
    max_tiles = H * ((kv_len_max + BN - 1) // BN)
    G, tab = slots_max, 0
    if d == 128 and R > 16:
        G, tab = max(slots_max // 2, 1), 1
    if G > max_tiles // min_tiles:
        G = max_tiles // min_tiles
    return max(G, 1), tab


def cta_tile_ranges(kv_len: int, H: int, G: int) -> List[Tuple[int, int]]:
    """[begin, end) on the (head, tile) axis for every CTA that owns tiles (equal split, G_eff = min(G, total))."""
    tph = (kv_len + BN - 1) // BN
    total = tph * H
    g = min(G, total)
    return [(b * total // g, (b + 1) * total // g) for b in range(g)]


def head_key_ranges(kv_len: int, H: int, G: int) -> List[List[Tuple[int, int]]]:
    """Per head: the [lo, hi) key ranges of the CTAs that deliver a partial of it, in merge order."""
    tph = (kv_len + BN - 1) // BN
    out: List[List[Tuple[int, int]]] = [[] for _ in range(H)]
    for (b, e) in cta_tile_ranges(kv_len, H, G):
        for h in range(b // tph, (e - 1) // tph + 1):
            t0, t1 = max(b, h * tph) - h * tph, min(e, (h + 1) * tph) - h * tph
            out[h].append((t0 * BN, min(t1 * BN, kv_len)))
    return out


def boundary_keys(kv_len: int, H: int, G: int, last_visible: int) -> List[List[int]]:
    """Per head: the first and last key of every CTA range of the head (these include the head's first and last key, i.e.
    the tiles where a head boundary meets a CTA boundary), limited to keys <= last_visible."""
    out = []
    for rngs in head_key_ranges(kv_len, H, G):
        ks = sorted({k for lo, hi in rngs for k in (lo, hi - 1) if k <= last_visible})
        out.append(ks)
    return out


def late_keys(kv_len: int, H: int, G: int, last_visible: int, first: int = 0) -> List[Optional[int]]:
    """Per head: a key in the last CTA range of the head that every row sees (the first key of that range, or the last
    visible key when the range holds only diagonal keys); None when only key `first` is visible to every row."""
    out: List[Optional[int]] = []
    for rngs in head_key_ranges(kv_len, H, G):
        lo = rngs[-1][0]
        if first < lo <= last_visible:
            out.append(lo)
        else:  # one range per head, or the last range holds only diagonal keys
            out.append(last_visible if last_visible > first else None)
    return out


# ---------------------------------------------------------------------------------------------------------------------
# input families
# ---------------------------------------------------------------------------------------------------------------------
def _directions(n: int, d: int, g: torch.Generator, device) -> torch.Tensor:
    """n unit vectors in R^d (float32): one-hot when n <= d (exactly orthogonal), else random."""
    if n <= d:
        return torch.eye(d, device=device)[:n]
    u = torch.randn((n, d), generator=g, device=device)
    return u / u.norm(dim=-1, keepdim=True)


def make_inputs(family: str, R: int, H: int, d: int, S: int, cap: int, scale: float, *, seed: int, device="cpu",
                own0: Optional[int] = None, G: Optional[int] = None, tree: Optional[np.ndarray] = None,
                sink: int = 0, out: Optional[Dict[str, torch.Tensor]] = None) -> Dict[str, torch.Tensor]:
    """q [R,H,d]; K, V head-major [H, cap, d] fp16 (rows >= S hold the stale sentinels).

    own0: key of row 0's own position (causal: S - R; tree: S - T + row0).  G: the grid, for the families that place keys
    on CTA boundaries.  tree: ancestor mask [R, T] for tree_leak.  sink: first key that is not a zero row (draft cache).
    `out`: tensors to fill in place (the 128K tests keep one store allocation)."""
    g = torch.Generator(device=device).manual_seed(seed)
    if out is None:
        q = torch.empty((R, H, d), dtype=torch.float16, device=device)
        K = torch.empty((H, cap, d), dtype=torch.float16, device=device)
        V = torch.empty_like(K)
    else:
        q, K, V = out["q"], out["K"], out["V"]
    own0 = S - R if own0 is None else own0
    last_vis = S - R  # the last key every row sees under the causal mask (needles, sink_then_late_max)
    qs = 1.0 / scale  # q = gap * qs * u gives a scaled score of `gap` against a key equal to u

    def small_bg():  # background keys score ~N(0, (0.02 gap)^2) against the needle directions
        K[:, :S] = (torch.randn((H, S, d), generator=g, device=device) * 0.02).half()
        V[:, :S] = torch.randn((H, S, d), generator=g, device=device).half()

    if family == "random":
        q.copy_(torch.randn((R, H, d), generator=g, device=device).half())
        K[:, :S] = torch.randn((H, S, d), generator=g, device=device).half()
        V[:, :S] = torch.randn((H, S, d), generator=g, device=device).half()
    elif family == "tile_indicator":
        # q = 0: exactly uniform softmax; V[j, c] = 1 iff c == (j // 64) % d, so output c counts the visible keys of one tile class
        q.zero_()
        K[:, :S] = torch.randn((H, S, d), generator=g, device=device).half()
        cls = (torch.arange(S, device=device) // BN) % d
        V[:, :S] = torch.nn.functional.one_hot(cls, d).half()[None]
    elif family == "diagonal":
        # row i: own key own0+i scores GAP_OWN, the next key own0+i+1 scores GAP_NEXT (> own: a limit one too far takes it)
        small_bg()
        u = _directions(R + 1, d, g, device)
        rows = u.clone()
        rows[1:] += (GAP_NEXT / GAP_OWN) * u[:R]  # key own0+i: u_i (row i, GAP_OWN) + 1.3 u_{i-1} (row i-1, GAP_NEXT)
        n = max(0, min(R + 1, S - own0))
        K[:, own0:own0 + n] = rows[:n].half()[None]
        q.copy_((GAP_OWN * qs * u[:R]).half()[:, None, :].expand(R, H, d))
    elif family == "sink_then_late_max":
        # key `sink` scores GAP_SINK, a key in the last CTA range of the head GAP_LATE: the running max moves between partials
        small_bg()
        q.copy_((qs * torch.eye(d, device=device)[0]).half()[None, None, :].expand(R, H, d))
        K[:, sink] = 0
        K[:, sink, 0] = GAP_SINK
        late = late_keys(S, H, G, last_vis, first=sink) if G is not None else [last_vis if last_vis > sink else None] * H
        for h, k in enumerate(late):
            if k is not None:
                K[h, k] = 0
                K[h, k, 0] = GAP_LATE
    elif family == "needles":
        # equal high scores on the first and last key of every CTA range of the head (all rows see them): a lost or doubled
        # boundary tile changes the needle count by one
        small_bg()
        q.copy_((GAP_NEEDLE * qs * torch.eye(d, device=device)[0]).half()[None, None, :].expand(R, H, d))
        for h, ks in enumerate(boundary_keys(S, H, G, last_vis)):
            idx = torch.tensor(ks, dtype=torch.long, device=device)
            K[h, idx] = 0
            K[h, idx, 0] = 1.0
    elif family == "large_magnitude":
        # integer q, K (exact fp32 dot products) with scaled scores ~280 nats; V ~ +-3e4: an unnormalised fp16 accumulator or a
        # softmax without the max subtraction overflows
        b = torch.randint(0, 2, (H, 1, d), generator=g, device=device).float() * 2 - 1
        K[:, :S] = (25 * b + torch.randint(-5, 6, (H, S, d), generator=g, device=device).float()).half()
        qq = b.permute(1, 0, 2) + torch.randint(-1, 2, (R, H, d), generator=g, device=device).float() * (
            torch.rand((R, H, d), generator=g, device=device) < 0.1).float()
        q.copy_(qq.half())
        sgn = torch.randint(0, 2, (H, S, d), generator=g, device=device).float() * 2 - 1
        V[:, :S] = (sgn * 3e4 * (1 + 0.1 * torch.rand((H, S, d), generator=g, device=device))).half()
    elif family == "tree_leak":
        # every row's highest score is on a tree column outside its ancestor set (distinct V per column)
        assert tree is not None
        Rt, T = tree.shape
        small_bg()
        rng = np.random.Generator(np.random.PCG64(seed))
        u = _directions(R, d, g, device)
        for i in range(R):
            hidden = np.nonzero(~tree[i])[0]
            if hidden.size:
                c = int(rng.choice(hidden))
                K[:, S - T + c] = (K[:, S - T + c].float() + u[i][None]).half()
        q.copy_((GAP_NEEDLE * qs * u).half()[:, None, :].expand(R, H, d))
    else:
        raise ValueError(family)
    K[:, S:] = STALE_K
    V[:, S:] = STALE_V
    return {"q": q, "K": K, "V": V}
