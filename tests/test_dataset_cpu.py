"""Input pipeline (SURVEY §8 row f-4): `data.dataset.get_dataset` against hand-made jsonl books and against what the reference's
own `get_dataset` returned on a sample of its PG-19 files."""
import json
import os
import sys

import numpy as np
import pytest
import torch

REPO = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, REPO)
from data.dataset import build_chat_input_lwm, get_dataset, read_books  # noqa: E402


class ByteTokenizer:
    """Stand-in with the two calls the pipeline makes: utf-8 bytes (+1, 0 = BOS) as ids."""

    def encode(self, text, return_tensors=None):
        ids = [0] + [b + 1 for b in text.encode("utf-8")]
        return torch.tensor([ids], dtype=torch.long) if return_tensors == "pt" else ids

    def decode(self, ids, skip_special_tokens=True):
        return bytes(i - 1 for i in ids if i > 0).decode("utf-8", errors="ignore")


def _write_books(tmp_path, n):
    texts = []
    for i in range(n):
        t = f"Book {i}. " + "chapter " * (5 + i) + "the end — né."
        texts.append(t)
        (tmp_path / f"{i:03d}.json").write_text(json.dumps({"text": t}) + "\n", encoding="utf-8")
    return texts


def test_get_dataset_reads_books_in_listdir_order(tmp_path):
    texts = _write_books(tmp_path, 23)
    by_name = {f"{i:03d}.json": t for i, t in enumerate(texts)}
    want = [by_name[n] for n in os.listdir(tmp_path)]
    tok = ByteTokenizer()
    assert read_books(str(tmp_path)) == want
    for name, count in (("128k", 23), ("gs", 20), ("one-shot", 1)):
        got = get_dataset(name, tok, root=str(tmp_path))
        assert len(got) == count
        for ids, text in zip(got, want):
            assert ids.dtype == torch.long and ids.dim() == 2 and ids.shape[0] == 1
            assert tok.decode(ids[0].tolist()) == text
    with pytest.raises(Exception, match="Dataset not found"):
        get_dataset("nope", tok, root=str(tmp_path))
    with pytest.raises(RuntimeError):
        get_dataset("lwm", tok, root=str(tmp_path))
    with pytest.raises(FileNotFoundError):
        get_dataset("gs", tok, root=str(tmp_path / "missing"))


def test_lwm_chat_wrapper_truncates_and_wraps():
    tok = ByteTokenizer()
    ids = build_chat_input_lwm(tok, "x" * 500, prefill=184)
    text = tok.decode(ids[0].tolist())
    assert text.startswith("You are a helpful assistant. USER: Please read a part of the book below")
    assert "[start of the book]\n" + "x" * 99 + "\n[end of the book]" in text  # 100 ids = BOS + 99 bytes
    assert text.endswith("ASSISTANT: ")


def test_against_the_reference_get_dataset(golden_dir):
    """The reference's own get_dataset('gs') on a sample of its PG-19 files (tests/golden/pg19_sample), as stored by
    tests/golden/make_golden.py in dataset_gs.npz: the 20 id tensors concatenated, and their lengths."""
    g = np.load(os.path.join(golden_dir, "dataset_gs.npz"))
    want = np.split(g["ids"].astype(np.int64), np.cumsum(g["lengths"])[:-1])
    got = get_dataset("gs", ByteTokenizer(), root=os.path.join(golden_dir, "pg19_sample"))
    assert len(got) == len(want) == 20
    for a, b in zip(got, want):
        assert torch.equal(a, torch.from_numpy(b)[None])
