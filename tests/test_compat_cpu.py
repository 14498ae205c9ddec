"""The `peft` / `trl` stand-ins under compat/ against the reference's OWN source: the calls `_get_target_modules` and
`_prep_for_training` (reason.py:362-394) make on a CPU stand-in that records what the kernels' LoRA entry point would be asked to do,
recorded from the reference source by tests/golden/make_source_golden.py and replayed here."""
import json
import os
import sys
import weakref

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFERENCE = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_source.json")))


@pytest.fixture()
def compat_path():
    p = os.path.join(ROOT, "compat")
    sys.path.insert(0, p)
    for m in [k for k in sys.modules if k.split(".")[0] in ("peft", "trl")]:
        del sys.modules[m]
    yield p
    sys.path.remove(p)
    for m in [k for k in sys.modules if k.split(".")[0] in ("peft", "trl")]:
        del sys.modules[m]


class _StandIn(torch.nn.Module):
    """CPU stand-in with the attributes reason.py touches; records the enable_lora() call the shim makes."""
    def __init__(self):
        super().__init__()
        from transformers import Qwen3ForCausalLM
        from bioreason_b200.configs import text_config
        tc = text_config("tiny"); tc.num_hidden_layers = 1
        self.text_model = Qwen3ForCausalLM(tc)
        self.dna_model = torch.nn.Linear(4, 4)
        self.dna_projection = torch.nn.Linear(4, 4)
        self.calls = []
        object.__setattr__(self.text_model, "_b200_owner", weakref.ref(self))

    @property
    def text(self):
        return self.text_model

    def enable_lora(self, r, alpha, seed=0):
        self.calls.append((r, alpha))


def test_reference_prep_for_training_runs_against_the_shims(compat_path):
    import peft
    rec = REFERENCE["prep_for_training"]
    assert rec["training_args"] == dict(lora_r=32, lora_alpha=64, lora_dropout=0.05) and not rec["dna_model_finetune"]
    m, objs = _StandIn(), {}
    for op, *args in rec["calls"]:                                  # reason.py:362-394 on this stand-in, in the reference's order
        if op == "requires_grad":
            name, flag = args
            for p in getattr(m, name).parameters():
                p.requires_grad = flag
        elif op == "LoraConfig":
            objs[op] = peft.LoraConfig(**args[0])
        else:                                                       # model.<module> = <peft entry point>(model.<module>, ...)
            names = args[0]
            setattr(m, names[0], getattr(peft, op)(*[objs[n] if n in objs else getattr(m, n) for n in names]))
    cfg = objs[rec["returns"]]
    assert m.calls == [(32, 64.0)] and m.lora_dropout == 0.05
    assert cfg.r == 32 and {"q_proj", "k_proj", "v_proj", "o_proj", "gate_proj", "up_proj", "down_proj"} <= set(cfg.target_modules)
    assert not any(p.requires_grad for p in m.dna_model.parameters()) and all(p.requires_grad for p in m.dna_projection.parameters())
    assert not any(p.requires_grad for p in m.text_model.parameters())                             # prepare_model_for_kbit_training froze the base


def test_shims_refuse_foreign_models_and_partial_targets(compat_path):
    import peft
    with pytest.raises(TypeError, match="DNALLMModel"):
        peft.get_peft_model(torch.nn.Linear(2, 2), peft.LoraConfig(r=4))
    m = _StandIn()
    with pytest.raises(NotImplementedError, match="subset"):
        peft.get_peft_model(m.text_model, peft.LoraConfig(r=4, target_modules=["q_proj", "v_proj"]))


def test_trl_parser_builds_the_dataclass_tuple(compat_path):
    import trl
    from bioreason_b200.trainer import DNALLMGRPOConfig
    s, t, mo = trl.TrlParser((trl.ScriptArguments, DNALLMGRPOConfig, trl.ModelConfig)).parse_args_and_config(
        ["--num_generations", "4", "--learning_rate", "2e-6", "--use_peft", "true", "--lora_r", "8", "--dataset_name", "kegg"])
    assert t.num_generations == 4 and t.learning_rate == 2e-6 and mo.lora_r == 8 and s.dataset_name == "kegg"
    cfg = trl.get_peft_config(mo)
    assert cfg.r == 8 and cfg.bias == "none"
    assert trl.get_peft_config(trl.ModelConfig(use_peft=False)) is None
