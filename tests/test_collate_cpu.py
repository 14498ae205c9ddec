"""SFT collate fast path (bioreason_b200/collate.py) against the reference's own loop: the labels the label-search body of
bioreason/dataset/kegg.py:258-323 produced when executed from the reference source (recorded by tests/golden/make_source_golden.py),
and a plain restatement of it."""
import json
import os

import pytest
import torch

from bioreason_b200 import collate

REFERENCE = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_source.json")))
START, END, PAD = [5, 6, 7], [9], 0


def _loop_labels(ids, start_m, end_m, pad):
    """Restatement of kegg.py:279-323 (TEST side): per-position window compares, first end after each start, pad mask last."""
    B, L = ids.shape
    labels = torch.full_like(ids, -100)
    for i in range(B):
        row = ids[i].tolist()
        starts = [p + len(start_m) for p in range(L - len(start_m) + 1) if row[p:p + len(start_m)] == start_m]
        ends = [p for p in range(L - len(end_m) + 1) if row[p:p + len(end_m)] == end_m]
        for s in starts:
            ve = [e for e in ends if e > s]
            e = min(ve) if ve else L
            if s < e and s < L:
                labels[i, s:min(e, L)] = ids[i, s:min(e, L)]
    labels[ids == pad] = -100
    return labels


def _random_rows(seed, B=6, L=90):
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(10, 40, (B, L), generator=g)
    for b in range(B):
        n_pad = int(torch.randint(0, 12, (1,), generator=g))
        ids[b, :n_pad] = PAD
        for _ in range(int(torch.randint(0, 4, (1,), generator=g))):
            p = int(torch.randint(n_pad, L - 4, (1,), generator=g))
            ids[b, p:p + 3] = torch.tensor(START)
        for _ in range(int(torch.randint(0, 5, (1,), generator=g))):
            ids[b, int(torch.randint(n_pad, L, (1,), generator=g))] = END[0]
    ids[0, -3:] = torch.tensor(START)          # a start marker that ends exactly at the row end
    ids[1, 20:23] = torch.tensor(START); ids[1, 23] = END[0]        # end marker right at the start position (does not close it)
    return ids


@pytest.mark.parametrize("seed", range(6))
def test_labels_match_the_loop(seed):
    ids = _random_rows(seed)
    got = collate.assistant_span_labels(ids, START, END, PAD)
    assert torch.equal(got, _loop_labels(ids, START, END, PAD))


@pytest.mark.parametrize("seed", [0, 3])
def test_labels_match_the_reference_source(seed):
    """The labels the body of the reference's qwen_dna_collate_fn, from `labels = torch.full_like(...)` to the pad mask, produced
    unmodified on `_random_rows(seed)`."""
    rec = REFERENCE["collate_labels"][str(seed)]
    ids = torch.tensor(rec["input_ids"])
    assert torch.equal(collate.assistant_span_labels(ids, START, END, PAD), torch.tensor(rec["labels"]))


def test_placeholder_expansion_and_counts():
    dna = torch.tensor([[3, 8, 9, 1, 1], [3, 8, 1, 1, 1], [3, 4, 5, 6, 7]])
    counts = collate.dna_token_counts(dna)
    assert counts == [3, 2, 5]
    texts = ["a <D> b <D> c", "no dna here", "<D>"]
    out = collate.expand_dna_placeholders(texts, counts, "<D>")
    assert out == ["a <D><D><D> b <D><D> c", "no dna here", "<D><D><D><D><D>"]
    # the reference's loop (processing_dl.py:185-193) on the same inputs
    ref, index = list(texts), 0
    for i in range(len(ref)):
        while "<D>" in ref[i]:
            ref[i] = ref[i].replace("<D>", "<|placeholder|>" * counts[index], 1); index += 1
        ref[i] = ref[i].replace("<|placeholder|>", "<D>")
    assert out == ref


def test_collate_fn_shape_of_work():
    class Tok:
        pad_token_id = PAD
        def encode(self, s, add_special_tokens=False):
            return START if "assistant" in s else END
    class Proc:
        tokenizer = Tok()
        def __call__(self, text, batch_dna_sequences, **kw):
            assert kw["padding_side"] == "left" and kw["max_length_dna"] == 64
            return {"input_ids": _random_rows(1, B=len(text)), "attention_mask": torch.ones(len(text), 90, dtype=torch.long)}
    ex = [dict(prompt="p", dna_sequences=["AC"], answer=" yes "), dict(prompt="q", dna_sequences=["GT"], answer="no")]
    b = collate.qwen_dna_collate_fn(ex, Proc(), 32, 64, return_answer_in_batch=True, apply_chat_template=lambda e, p: {"prompt": e["prompt"]})
    assert b["answer"] == ["yes", "no"] and b["labels"].shape == b["input_ids"].shape
    assert torch.equal(b["labels"], _loop_labels(b["input_ids"], START, END, PAD))
