"""End-to-end DNA-LLM forward parity: CUDA path vs the CPU oracle / the golden reference outputs."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _to_cuda_batch(b):
    return b   # DNALLMModel moves tensors itself (as HF/accelerate would)


def _err_budget(test_logits, ref32, ref16, valid):
    """Regime: bf16 storage / fp32 accumulate.  Accept if we sit as close to the reference's fp32 result as the
    reference's OWN --bf16 path does (x2 slack), measured over attended positions."""
    e_mine = (test_logits - ref32)[valid].abs()
    e_ref = (ref16 - ref32)[valid].abs()
    return e_mine.max().item(), e_ref.max().item(), e_mine.mean().item(), e_ref.mean().item()


def test_forward_tiny_golden(golden, tiny_oracle, reference_logits):
    from bioreason_b200.models import DNALLMModel
    m = DNALLMModel.from_oracle(tiny_oracle)
    A, ref = golden["A"], reference_logits
    out = m(**A["batch"], labels=A["labels"])
    logits = out.logits.float().cpu()
    valid = A["batch"]["attention_mask"].bool()
    mx, rmx, mean, rmean = _err_budget(logits, ref["A"], ref["A_bf16"], valid)
    print(f"tiny: max|err| {mx:.4g} (reference bf16 path: {rmx:.4g}); mean {mean:.4g} (ref {rmean:.4g}); logit std {ref['A'][valid].std():.3g}")
    assert mx <= 2.0 * rmx + 1e-3 and mean <= 2.0 * rmean + 1e-4
    assert abs(out.loss.item() - A["loss"].item()) <= 2 * abs(A["loss_bf16"].item() - A["loss"].item()) + 2e-3
    # text-only path
    Bc = golden["B"]
    lb = m(**Bc["batch"]).logits.float().cpu()
    vb = Bc["batch"]["attention_mask"].bool()
    assert (lb - ref["B"])[vb].abs().max().item() <= 2.0 * rmx + 1e-3
    # count mismatch raises exactly like dna_llm.py:222-225
    with pytest.raises(ValueError, match="do not match"):
        m(**golden["C"]["batch"])
    with pytest.raises(ValueError, match="must be provided"):
        m(input_ids=None, attention_mask=None)


def test_process_dna_embeddings_tiny(golden, tiny_oracle):
    """The list-returning public method (dna_llm.py:103-179): per batch item, the valid rows of its sequences, projected."""
    from bioreason_b200.models import DNALLMModel
    m = DNALLMModel.from_oracle(tiny_oracle)
    b = golden["A"]["batch"]
    B = b["input_ids"].shape[0]
    with torch.no_grad():
        want = tiny_oracle.process_dna_embeddings(b["dna_tokenized"], b["batch_idx_map"], B)
    got = m.process_dna_embeddings(b["dna_tokenized"], b["batch_idx_map"], B)
    assert len(got) == len(want) == B
    for g, w in zip(got, want):
        assert g.shape == w.shape
        torch.testing.assert_close(g.float().cpu(), w, rtol=3e-2, atol=3e-2)
    empty = m.process_dna_embeddings({k: v[:2] for k, v in b["dna_tokenized"].items()}, [1, 1], 3)
    assert empty[0].shape[0] == 0 and empty[2].shape[0] == 0 and empty[1].shape[0] > 0


def test_per_token_logps_tiny_golden(golden, tiny_oracle):
    from bioreason_b200.models import DNALLMModel
    m = DNALLMModel.from_oracle(tiny_oracle)
    E, D = golden["E"], golden["D"]
    lp = m.per_token_logps(E["input_ids"], E["attention_mask"], D["batch"]["dna_tokenized"], D["batch"]["batch_idx_map"]).cpu()
    att = E["attention_mask"][:, 1:].bool()
    err = (lp - E["logps"])[att].abs().max().item()
    print("logps max err", err)
    assert err < 0.02
    C = E["completion_ids"].shape[1]
    lp_c = m.per_token_logps(E["input_ids"], E["attention_mask"], D["batch"]["dna_tokenized"], D["batch"]["batch_idx_map"], keep_last=C).cpu()
    assert torch.equal(lp_c, lp[:, -C:])


@pytest.mark.parametrize("B,n_seq,dna_len,text_len", [(2, 2, [40, 33], [70, 51]), (3, 1, 168, 128)])
def test_forward_small_vs_oracle(B, n_seq, dna_len, text_len):
    """Bigger-than-tiny shapes (multi-tile GEMMs, several attention blocks) against the fp32 CPU oracle."""
    from bioreason_b200.configs import text_config, dna_config
    from bioreason_b200.models import DNALLMModel
    from oracle.models import build_oracle, synth_batch
    tc, dc = text_config("small"), dna_config("small")
    oracle = build_oracle(tc, dc, seed=7)
    batch = synth_batch(tc, dc, batch=B, n_seq=n_seq, dna_len=dna_len, text_len=text_len, seed=3)
    with torch.no_grad():
        ref32 = oracle(**batch).logits
        ref16 = oracle.to(torch.bfloat16)(**batch).logits.float()
    oracle.float()
    m = DNALLMModel.from_oracle(oracle)
    logits = m(**batch).logits.float().cpu()
    valid = batch["attention_mask"].bool()
    mx, rmx, mean, rmean = _err_budget(logits, ref32, ref16, valid)
    print(f"small: max|err| {mx:.4g} (HF bf16: {rmx:.4g}); mean {mean:.4g} (HF bf16 {rmean:.4g}); logit std {ref32[valid].std():.3g}")
    assert mx <= 2.0 * rmx + 1e-3 and mean <= 2.0 * rmean + 1e-4


@pytest.mark.skipif(__import__("os").environ.get("BR_SKIP_LARGE") == "1", reason="BR_SKIP_LARGE=1")
def test_forward_config_a_real_shapes():
    """BASELINE.json configs[0] / SURVEY.md §8d (a): NT-v2-500M + Qwen3-1.7B at the REAL widths and depths, one forward on
    2 x 168-token DNA (1 002 bp) + 128-token prompt (L = 464), CUDA path vs the CPU oracle (HF fp32 and HF bf16)."""
    import time
    from bioreason_b200.configs import text_config, dna_config
    from bioreason_b200.models import DNALLMModel
    from oracle.models import build_oracle, synth_batch
    torch.set_num_threads(min(32, __import__("os").cpu_count() or 8))
    tc, dc = text_config("qwen3-1.7b"), dna_config("nt-v2-500m")
    t0 = time.time()
    oracle = build_oracle(tc, dc, seed=1234)
    batch = synth_batch(tc, dc, batch=1, n_seq=2, dna_len=168, text_len=128, seed=1234)
    assert batch["input_ids"].shape == (1, 128 + 2 * 168 + 4) or batch["input_ids"].shape[1] >= 464
    with torch.no_grad():
        ref32 = oracle(**batch).logits
    t_cpu = time.time() - t0
    m = DNALLMModel.from_oracle(oracle)
    torch.cuda.synchronize(); t1 = time.time()
    logits = m(**batch).logits.float().cpu()
    t_gpu = time.time() - t1
    with torch.no_grad():
        ref16 = oracle.to(torch.bfloat16)(**batch).logits.float()
    e_mine = (logits - ref32).abs(); e_ref = (ref16 - ref32).abs()
    std = ref32.std().item()
    print(f"config (a): L={batch['input_ids'].shape[1]} V={tc.vocab_size}; max|err| ours {e_mine.max():.4g} vs HF-bf16 {e_ref.max():.4g}; "
          f"mean {e_mine.mean():.4g} vs {e_ref.mean():.4g}; logit std {std:.3g}; argmax agreement with fp32: ours "
          f"{(logits.argmax(-1) == ref32.argmax(-1)).float().mean():.3f}, HF-bf16 {(ref16.argmax(-1) == ref32.argmax(-1)).float().mean():.3f}; "
          f"oracle build+fwd {t_cpu:.0f}s, CUDA fwd (incl. lazy logits) {t_gpu * 1e3:.0f} ms")
    assert e_mine.max().item() <= 2.0 * e_ref.max().item() + 1e-3
    assert e_mine.mean().item() <= 2.0 * e_ref.mean().item() + 1e-4
