"""Pin the CPU oracle against outputs of the unmodified reference (tests/golden/make_golden.py)."""
import ctypes, os, subprocess
import numpy as np
import pytest
import torch

from oracle import grpo as og
from oracle.golden import tensor_sha256

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_forward_logits_and_loss_match_reference(golden, tiny_oracle):
    A = golden["A"]
    with torch.no_grad():
        o = tiny_oracle(**A["batch"], labels=A["labels"])
    assert tensor_sha256(o.logits) == A["logits_sha256"]          # same HF code, same weights -> bit-exact
    assert torch.equal(o.loss, A["loss"])


def test_bf16_regime_error_budget(golden, reference_logits):
    """How far the reference's own --bf16 path sits from its fp32 path: the budget GPU parity uses."""
    A, ref = golden["A"], reference_logits
    valid = A["batch"]["attention_mask"].bool()
    err = (ref["A_bf16"] - ref["A"])[valid].abs().max().item()
    assert 0 < err < 0.1 * ref["A"][valid].std().item() * 10


def test_text_only_path(golden, tiny_oracle):
    B = golden["B"]
    with torch.no_grad():
        o = tiny_oracle(**B["batch"])
    assert tensor_sha256(o.logits) == B["logits_sha256"]


def test_count_mismatch_raises(golden, tiny_oracle):
    assert golden["C"]["raised"]
    with pytest.raises(ValueError, match="do not match"):
        tiny_oracle(**golden["C"]["batch"])


def test_generate_matches_reference(golden, tiny_oracle):
    from transformers import GenerationConfig
    D = golden["D"]
    cfg = tiny_oracle.text_config
    ids = tiny_oracle.generate(**D["batch"], max_new_tokens=12, do_sample=False,
                               pad_token_id=cfg.pad_token_id, eos_token_id=cfg.eos_token_id)
    assert torch.equal(ids, D["greedy"])
    gc = GenerationConfig(max_new_tokens=12, do_sample=True, temperature=0.6, top_p=0.95, top_k=20,
                          pad_token_id=cfg.pad_token_id, eos_token_id=cfg.eos_token_id)
    torch.manual_seed(D["sample_seed"])
    assert torch.equal(tiny_oracle.generate(**D["batch"], generation_config=gc), D["sampled"])
    ids = tiny_oracle.generate(**D["ragged_batch"], max_new_tokens=8, do_sample=False,
                               pad_token_id=cfg.pad_token_id, eos_token_id=cfg.eos_token_id)
    assert torch.equal(ids, D["ragged_greedy"])


def test_per_token_logps_and_eos_mask(golden, tiny_oracle):
    E, D = golden["E"], golden["D"]
    m = og.completion_mask_from_eos(E["completion_ids"], tiny_oracle.text_config.eos_token_id)
    assert torch.equal(m, E["completion_mask"])
    with torch.no_grad():
        lps = og.per_token_logps(tiny_oracle, E["input_ids"], E["attention_mask"],
                                 dna_tokenized=D["batch"]["dna_tokenized"], batch_idx_map=D["batch"]["batch_idx_map"])
    assert torch.equal(lps, E["logps"])


def test_advantages(golden):
    F = golden["F"]
    adv = og.group_advantages(F["rewards_per_func"], F["G"])
    assert torch.equal(adv, F["advantages"])
    assert torch.all(adv[8:12] == 0)                    # zero-variance group -> 0/(0+1e-4)


@pytest.mark.parametrize("case,beta,lo,hi,use_old", [("mu1", 0.04, 0.2, 0.2, False), ("mu2", 0.04, 0.2, 0.2, True),
                                                     ("mu2_nokl", 0.0, 0.2, 0.2, True), ("mu2_asym", 0.1, 0.1, 0.3, True)])
def test_grpo_loss_torch_and_c(golden, case, beta, lo, hi, use_old):
    G = golden["G"]; ref = G[case]
    lp = G["lp"].clone().requires_grad_(True)
    loss, kl, clip = og.grpo_loss(lp, G["old"] if use_old else None, G["ref"] if beta > 0 else None, G["adv"],
                                  G["mask"], beta, lo, hi)
    loss.backward()
    assert torch.equal(loss.detach(), ref["loss"]) and torch.equal(lp.grad, ref["dlp"])
    assert abs(clip.item() - ref["clip_ratio"].item()) < 1e-7
    if beta > 0:
        assert abs(kl.item() - ref["kl"].item()) < 1e-7
    if use_old:
        assert ref["clip_ratio"].item() > 0            # the fixture really exercises clipping
    # plain-C restatement (what smoke() and the GPU parity tests check against)
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle")])
    lib = ctypes.CDLL(os.path.join(ROOT, "oracle", "_build", "libgrpo_ref.so"))
    f32 = lambda t: np.ascontiguousarray(t.detach().numpy(), dtype=np.float32)
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p) if a is not None else None
    a_lp, a_old, a_ref, a_adv = f32(G["lp"]), f32(G["old"]) if use_old else None, f32(G["ref"]) if beta > 0 else None, f32(G["adv"])
    a_mask = np.ascontiguousarray(G["mask"].numpy(), dtype=np.int32)
    out3 = np.zeros(3, np.float32); dlp = np.zeros_like(a_lp)
    B, C = a_lp.shape
    lib.oracle_grpo_loss(P(a_lp), P(a_old), P(a_ref), P(a_adv), P(a_mask), B, C, ctypes.c_float(beta),
                         ctypes.c_float(lo), ctypes.c_float(hi), P(out3), P(dlp))
    np.testing.assert_allclose(out3[0], ref["loss"].item(), rtol=2e-6)
    np.testing.assert_allclose(out3[2], ref["clip_ratio"].item(), rtol=1e-6)
    np.testing.assert_allclose(dlp, ref["dlp"].numpy(), rtol=2e-5, atol=1e-8)
    if beta > 0:
        np.testing.assert_allclose(out3[1], ref["kl"].item(), rtol=2e-6)
    Fg = golden["F"]
    r = f32(Fg["rewards_per_func"]); adv = np.zeros(r.shape[0], np.float32)
    lib.oracle_group_advantages(P(r), r.shape[0], r.shape[1], Fg["G"], P(adv))
    np.testing.assert_allclose(adv, Fg["advantages"].numpy(), rtol=2e-5, atol=1e-6)


def test_repeat_sampler(golden):
    for (n, mini, bs, rep, seed), want in golden["H"].items():
        assert og.repeat_random_sampler(n, mini, bs, rep, seed) == want


def test_manual_generate_matches_hf_greedy(golden, tiny_oracle):
    """Pins oracle/generate.py (the replayable-sampling loop) against HF generate() and the reference's golden ids."""
    from oracle.generate import manual_generate
    D = golden["D"]; cfg = tiny_oracle.text_config
    ids = manual_generate(tiny_oracle, D["batch"], max_new_tokens=12, eos_token_id=cfg.eos_token_id, pad_token_id=cfg.pad_token_id)
    assert torch.equal(ids, D["greedy"])
    ids = manual_generate(tiny_oracle, D["ragged_batch"], max_new_tokens=8, eos_token_id=cfg.eos_token_id, pad_token_id=cfg.pad_token_id)
    assert torch.equal(ids, D["ragged_greedy"])
    # sampled: every drawn token must be inside HF's own top-k/top-p support and be reproducible from the uniforms
    u = torch.rand(6, 4, generator=torch.Generator().manual_seed(3))
    a = manual_generate(tiny_oracle, D["batch"], max_new_tokens=6, do_sample=True, temperature=0.6, top_k=20, top_p=0.95, uniforms=u)
    b = manual_generate(tiny_oracle, D["batch"], max_new_tokens=6, do_sample=True, temperature=0.6, top_k=20, top_p=0.95, uniforms=u)
    assert torch.equal(a, b) and a.shape == (4, 6)
    assert len({tuple(r.tolist()) for r in a}) > 1          # different uniforms per row -> the G samples differ
