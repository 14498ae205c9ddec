"""Generate golden fixtures by running the UNMODIFIED reference code (/root/reference) here.

Run in the build container only:  python tests/golden/make_golden.py
Writes tests/golden/*.pt (committed).  /root/reference does not exist on the GPU box; tests only
read the fixtures.  What executes from the reference: DNALLMModel.forward / .generate /
.process_dna_embeddings (bioreason/models/dna_llm.py:103-305), DNALLMGRPOTrainer._get_per_token_logps
and .compute_loss (grpo_trainer.py:510-520, 751-814), the EOS-mask and advantage blocks
(grpo_trainer.py:605-609, 682-692; executed from the file's own source lines) and
RepeatRandomSampler (:72-119).  Model weights are seeded random (no checkpoints offline).  The oracle
regenerates the weights and the logits of cases A and B exactly, so the fixture keeps the weight seed and
SHA-256 digests of those tensors (oracle/golden.py) rather than megabytes of them; the tests recompute and
compare the digests.
"""
import os, sys, textwrap, types, collections
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT); sys.path.insert(0, HERE)

import _ref_import
from bioreason_b200.configs import text_config, dna_config
from oracle.golden import state_sha256, tensor_sha256
from oracle.models import build_text_model, build_dna_model, round_to_bf16_, synth_batch

torch.manual_seed(0)
ref_dna_llm, ref_trainer = _ref_import.load_reference()
RefModel = ref_dna_llm.DNALLMModel
RefTrainer = ref_trainer.DNALLMGRPOTrainer


def make_ref_model(tc, dc, seed):
    """Build the reference DNALLMModel around seeded HF modules, bypassing only the
    from_pretrained/tokenizer loading in __init__ (dna_llm.py:64-100 needs the network)."""
    m = RefModel.__new__(RefModel)
    torch.nn.Module.__init__(m)
    m.text_model = build_text_model(tc, seed)
    m.dna_model = build_dna_model(dc, seed)
    m.text_config, m.dna_config = m.text_model.config, m.dna_model.config
    m.text_hidden_size, m.dna_hidden_size = tc.hidden_size, dc.hidden_size
    torch.manual_seed(seed + 7)
    m.dna_projection = torch.nn.Linear(dc.hidden_size, tc.hidden_size)
    m.dna_token_id = tc.dna_token_ids[1]
    m.dna_is_evo2, m.dna_embedding_layer = False, None
    m.max_length_dna, m.max_length_text = 2048, 512
    round_to_bf16_(m)
    return m.eval()


def ref_source_block(first, last):
    lines = open("/root/reference/bioreason/trainer/grpo_trainer.py").read().split("\n")[first - 1:last]
    return textwrap.dedent("\n".join(lines))


def main():
    out = {}
    tc, dc = text_config("tiny"), dna_config("tiny")
    model = make_ref_model(tc, dc, seed=1234)
    out["weights_seed"], out["weights_sha256"] = 1234, state_sha256(model)     # oracle.models.build_oracle(..., seed=1234)

    # ---- case A: ragged batch, forward + CE loss (fp32 compute, bf16-representable weights)
    batch = synth_batch(tc, dc, batch=3, n_seq=2, dna_len=[12, 9, 12], text_len=[24, 17, 30], seed=11)
    labels = batch["input_ids"].clone()
    labels[batch["attention_mask"] == 0] = -100
    labels[:, :20] = -100
    with torch.no_grad():
        o = model(**batch, labels=labels)
    out["A"] = dict(batch=batch, labels=labels, logits_sha256=tensor_sha256(o.logits), loss=o.loss.clone())
    # the reference's own --bf16 regime
    m16 = make_ref_model(tc, dc, seed=1234).to(torch.bfloat16)
    with torch.no_grad():
        o16 = m16(**batch, labels=labels)
    out["A"]["logits_bf16_sha256"] = tensor_sha256(o16.logits)
    out["A"]["loss_bf16"] = o16.loss.float().clone()

    # ---- case B: no DNA at all (dna_tokenized=None, batch_idx_map=[]) -- text-only path
    batch_b = synth_batch(tc, dc, batch=2, n_seq=0, dna_len=0, text_len=[16, 11], seed=12)
    with torch.no_grad():
        ob = model(**batch_b)
    out["B"] = dict(batch=batch_b, logits_sha256=tensor_sha256(ob.logits))

    # ---- case C: count mismatch must raise ValueError (dna_llm.py:222-225)
    bad = synth_batch(tc, dc, batch=1, n_seq=1, dna_len=8, text_len=10, seed=13)
    bad["input_ids"][0, -1] = tc.dna_token_ids[1]
    try:
        model(**bad); raised = False
    except ValueError as e:
        raised = "do not match" in str(e)
    out["C"] = dict(batch=bad, raised=raised)

    # ---- case D: generate (greedy, and sampled under a torch seed) on a G-replicated prompt
    gen_batch = synth_batch(tc, dc, batch=4, n_seq=2, dna_len=10, text_len=18, seed=14, same_prompt=True)
    from transformers import GenerationConfig
    ids_greedy = model.generate(**gen_batch, max_new_tokens=12, do_sample=False,
                                pad_token_id=tc.pad_token_id, eos_token_id=tc.eos_token_id)
    gc = GenerationConfig(max_new_tokens=12, do_sample=True, temperature=0.6, top_p=0.95, top_k=20,
                          pad_token_id=tc.pad_token_id, eos_token_id=tc.eos_token_id)   # grpo_trainer.py:384-391
    torch.manual_seed(77)
    ids_sampled = model.generate(**gen_batch, generation_config=gc)
    # ragged prompts (left-padded), greedy
    rag = synth_batch(tc, dc, batch=3, n_seq=1, dna_len=[10, 6, 8], text_len=[12, 20, 9], seed=15)
    ids_rag = model.generate(**rag, max_new_tokens=8, do_sample=False,
                             pad_token_id=tc.pad_token_id, eos_token_id=tc.eos_token_id)
    out["D"] = dict(batch=gen_batch, greedy=ids_greedy, sampled=ids_sampled, sample_seed=77,
                    ragged_batch=rag, ragged_greedy=ids_rag)

    # ---- case E: _get_per_token_logps through the reference model
    comp = torch.randint(0, tc.eos_token_id, (4, 6))
    comp[1, 3] = tc.eos_token_id; comp[1, 4:] = tc.pad_token_id
    full_ids = torch.cat([gen_batch["input_ids"], comp], dim=1)
    # EOS mask block, executed from the reference's own source (grpo_trainer.py:605-609)
    ns = dict(torch=torch, completion_ids=comp, device="cpu",
              self=types.SimpleNamespace(processing_class=types.SimpleNamespace(eos_token_id=tc.eos_token_id)))
    exec(ref_source_block(605, 609), ns)
    completion_mask = ns["completion_mask"]
    full_mask = torch.cat([gen_batch["attention_mask"], completion_mask], dim=1)
    mm = dict(dna_tokenized=gen_batch["dna_tokenized"], batch_idx_map=gen_batch["batch_idx_map"])
    with torch.no_grad():
        lps = RefTrainer._get_per_token_logps(None, model, full_ids, full_mask, **mm)
    out["E"] = dict(completion_ids=comp, completion_mask=completion_mask, input_ids=full_ids,
                    attention_mask=full_mask, logps=lps.clone())

    # ---- case F: advantage block from the reference's own source (grpo_trainer.py:682-692)
    rewards_per_func = torch.randn(16, 3)
    rewards_per_func[8:12] = rewards_per_func[8:9]            # a zero-variance group
    ns = dict(torch=torch, rewards_per_func=rewards_per_func, self=types.SimpleNamespace(num_generations=4))
    exec(ref_source_block(682, 692), ns)
    out["F"] = dict(rewards_per_func=rewards_per_func, G=4, advantages=ns["advantages"].clone())

    # ---- case G: compute_loss (grpo_trainer.py:751-814) on a stub trainer
    class Stub:
        pass
    def run_compute_loss(lp_in, old, ref, adv, cmask, beta, mu, eps_lo=0.2, eps_hi=0.2):
        st = Stub()
        st.state = types.SimpleNamespace(global_step=0)
        st.num_iterations = mu
        st.args = types.SimpleNamespace(gradient_accumulation_steps=1)
        st._buffered_inputs = [None]; st._step = 0
        st.beta, st.epsilon_low, st.epsilon_high = beta, eps_lo, eps_hi
        st._metrics = collections.defaultdict(list)
        st.accelerator = types.SimpleNamespace(gather_for_metrics=lambda x: x)
        P = 5
        lp = lp_in.clone().requires_grad_(True)
        prepared = dict(prompt_ids=torch.zeros(lp.shape[0], P, dtype=torch.long),
                        prompt_mask=torch.ones(lp.shape[0], P, dtype=torch.long),
                        completion_ids=torch.zeros(lp.shape, dtype=torch.long), completion_mask=cmask,
                        old_per_token_logps=old, ref_per_token_logps=ref, advantages=adv, multimodal_inputs={})
        st._generate_and_score_completions = lambda inputs, model: prepared
        # compute_loss slices [:, P-1:] off what _get_per_token_logps returns
        st._get_per_token_logps = lambda model, ids, mask, **kw: torch.cat(
            [torch.zeros(lp.shape[0], P - 1), lp], dim=1)
        import io, contextlib
        with contextlib.redirect_stdout(io.StringIO()):
            loss = RefTrainer.compute_loss(st, None, {})
        loss.backward()
        return dict(loss=loss.detach().clone(), dlp=lp.grad.clone(),
                    kl=torch.tensor(st._metrics["kl"][0]) if beta > 0 else None,
                    clip_ratio=torch.tensor(st._metrics["clip_ratio"][0]))
    B, C = 8, 16
    g = torch.Generator().manual_seed(5)
    lp = -torch.rand(B, C, generator=g) * 3
    old = lp + torch.randn(B, C, generator=g) * 0.3         # wide enough that clipping triggers
    ref = lp + torch.randn(B, C, generator=g) * 0.2
    adv = torch.randn(B, generator=g)
    cmask = (torch.arange(C)[None, :] < torch.randint(3, C + 1, (B, 1), generator=g)).int()
    out["G"] = dict(lp=lp, old=old, ref=ref, adv=adv, mask=cmask,
                    mu1=run_compute_loss(lp, None, ref, adv, cmask, beta=0.04, mu=1),
                    mu2=run_compute_loss(lp, old, ref, adv, cmask, beta=0.04, mu=2),
                    mu2_nokl=run_compute_loss(lp, old, None, adv, cmask, beta=0.0, mu=2),
                    mu2_asym=run_compute_loss(lp, old, ref, adv, cmask, beta=0.1, mu=2, eps_lo=0.1, eps_hi=0.3))

    # ---- case H: RepeatRandomSampler (grpo_trainer.py:72-119)
    samp = {}
    for (n, mini, bs, rep, seed) in [(10, 4, 2, 1, 42), (7, 2, 3, 2, 7), (16, 8, 1, 1, 0)]:
        s = ref_trainer.RepeatRandomSampler(range(n), mini, bs, rep, seed)
        samp[(n, mini, bs, rep, seed)] = list(iter(s))
    out["H"] = samp

    torch.save(out, os.path.join(HERE, "reference_tiny.pt"))
    print("wrote", os.path.join(HERE, "reference_tiny.pt"),
          os.path.getsize(os.path.join(HERE, "reference_tiny.pt")) // 1024, "KiB")
    print("greedy", ids_greedy.tolist()); print("sampled", ids_sampled.tolist()); print("C raised", raised)


if __name__ == "__main__":
    main()
