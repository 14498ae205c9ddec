"""Record what two pieces of the UNMODIFIED reference source do, for the tests that compare against them.

    python tests/golden/make_source_golden.py <checkout of the original BioReason project>

Writes tests/golden/reference_source.json (committed):
  * collate_labels: the label-search body of `qwen_dna_collate_fn` (bioreason/dataset/kegg.py:258-323, from
    `labels = torch.full_like(...)` to the pad mask), executed unmodified on the inputs of tests/test_collate_cpu.py;
    its input ids and the labels it produced (tests/test_collate_cpu.py::test_labels_match_the_reference_source).
  * prep_for_training: the calls `_get_target_modules` + `_prep_for_training` (reason.py:362-394), executed unmodified on
    the CPU stand-in of tests/test_compat_cpu.py, make against the `peft` stand-in under compat/: the requires_grad changes
    they make and each peft entry point with its arguments, in order (replayed by
    tests/test_compat_cpu.py::test_reference_prep_for_training_runs_against_the_shims).
Both functions are extracted with ast and executed; no reference source is stored.
"""
import ast
import json
import os
import sys
import types

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

MODULES = ("text_model", "dna_model", "dna_projection")


def collate_labels(ref):
    import test_collate_cpu as tcc
    path = os.path.join(ref, "bioreason", "dataset", "kegg.py")
    tree = ast.parse(open(path).read())
    fn = next(n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "qwen_dna_collate_fn")
    first = next(i for i, st in enumerate(fn.body) if isinstance(st, ast.Assign) and getattr(st.targets[0], "id", "") == "labels")
    last = next(i for i, st in enumerate(fn.body) if isinstance(st, ast.Assign) and isinstance(st.targets[0], ast.Subscript)
                and getattr(st.targets[0].value, "id", "") == "batch" and getattr(st.targets[0].slice, "value", "") == "labels")
    code = compile(ast.Module(body=fn.body[first:last], type_ignores=[]), path, "exec")
    out = {}
    for seed in (0, 3):
        ids = tcc._random_rows(seed)
        tok = types.SimpleNamespace(pad_token_id=tcc.PAD,
                                    encode=lambda s, add_special_tokens=False: tcc.START if "assistant" in s else tcc.END)
        ns = {"torch": torch, "batch": {"input_ids": ids}, "processor": types.SimpleNamespace(tokenizer=tok)}
        exec(code, ns)
        out[str(seed)] = {"input_ids": ids.tolist(), "labels": ns["labels"].tolist()}
    return out


def prep_for_training(ref):
    sys.path.insert(0, os.path.join(ROOT, "compat"))
    import peft
    import test_compat_cpu as tcp
    path = os.path.join(ref, "reason.py")
    tree = ast.parse(open(path).read())
    fns = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in {"_get_target_modules", "_prep_for_training"}]
    m = tcp._StandIn()
    training_args = dict(lora_r=32, lora_alpha=64, lora_dropout=0.05)
    calls = []

    def flags():
        return {name: [p.requires_grad for p in getattr(m, name).parameters()] for name in MODULES}
    state = {"last": flags()}

    def record_requires_grad():
        """requires_grad changes the reference made since the last peft call (whole modules: the stand-in has no partial ones)."""
        now = flags()
        for name in MODULES:
            if now[name] != state["last"][name]:
                assert len(set(now[name])) == 1, name
                calls.append(["requires_grad", name, now[name][0]])

    def describe(a):
        if isinstance(a, peft.LoraConfig):
            return "LoraConfig"
        return next(name for name in MODULES if getattr(m, name) is a)

    def wrap(name, fn):
        def call(*args, **kwargs):
            record_requires_grad()
            if name == "LoraConfig":
                assert not args
                calls.append([name, kwargs])
            else:
                assert not kwargs
                calls.append([name, [describe(a) for a in args]])
            out = fn(*args, **kwargs)
            state["last"] = flags()
            return out
        return call

    ns = {"torch": torch, "DNALLMModel": tcp._StandIn}
    ns.update({k: wrap(k, getattr(peft, k)) for k in ("LoraConfig", "get_peft_model", "prepare_model_for_kbit_training")})
    exec(compile(ast.Module(body=fns, type_ignores=[]), path, "exec"), ns)
    cfg = ns["_prep_for_training"](m, types.SimpleNamespace(**training_args), dna_model_finetune=False)
    record_requires_grad()
    assert isinstance(cfg, peft.LoraConfig)
    return {"training_args": training_args, "dna_model_finetune": False, "calls": calls, "returns": "LoraConfig"}


def main():
    ref = sys.argv[1]
    out = {"collate_labels": collate_labels(ref), "prep_for_training": prep_for_training(ref)}
    path = os.path.join(HERE, "reference_source.json")
    with open(path, "w") as f:
        json.dump(out, f, separators=(",", ":"))
        f.write("\n")
    print("wrote", path, os.path.getsize(path), "bytes")
    print(json.dumps(out["prep_for_training"], indent=1))


if __name__ == "__main__":
    main()
