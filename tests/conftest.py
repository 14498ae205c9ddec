import os, sys
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu under gpurun)")
    config.addinivalue_line("markers", "needs_lib: CPU test that loads libbioreason_b200.so (symbols only, no compute)")


_BUILT = []


@pytest.fixture(autouse=True)
def _built_library(request):
    """GPU tests (and the ABI test, which asks for it explicitly) need libbioreason_b200.so to match the sources (hash-checked,
    a no-op when up to date).  CPU tests that mock the ops must run on a box without nvcc: nothing is built for them."""
    if request.node.get_closest_marker("gpu") is None and request.node.get_closest_marker("needs_lib") is None:
        return
    if not _BUILT:
        import shutil
        from bioreason_b200 import build
        if not (shutil.which("nvcc") or os.path.exists(build.NVCC)):
            if os.path.exists(build.LIB):
                _BUILT.append(build.LIB)
                return
            pytest.skip("nvcc not available and libbioreason_b200.so not built")
        _BUILT.append(build.build())


@pytest.fixture(scope="session")
def golden():
    import torch
    return torch.load(os.path.join(ROOT, "tests", "golden", "reference_tiny.pt"), weights_only=True)


@pytest.fixture(scope="session")
def tiny_oracle(golden):
    """Oracle DNA-LLM carrying exactly the weights the reference run used: regenerated from their seed, checked by digest."""
    from bioreason_b200.configs import text_config, dna_config
    from oracle.golden import state_sha256
    from oracle.models import build_oracle
    m = build_oracle(text_config("tiny"), dna_config("tiny"), seed=golden["weights_seed"])
    assert state_sha256(m) == golden["weights_sha256"], "the seeded init no longer reproduces the reference run's weights"
    return m.eval()


@pytest.fixture(scope="session")
def reference_logits(golden, tiny_oracle):
    """Logits of the reference run (cases A and B, and A through the reference's bf16 path), recomputed by the oracle and checked
    bit for bit against the fixture's digests."""
    import torch
    from bioreason_b200.configs import text_config, dna_config
    from oracle.golden import tensor_sha256
    from oracle.models import build_oracle
    A, B = golden["A"], golden["B"]
    # a fresh model, as the reference run built one: a used one carries its fp32 rotary cos/sin caches into bf16
    m16 = build_oracle(text_config("tiny"), dna_config("tiny"), seed=golden["weights_seed"]).to(torch.bfloat16).eval()
    with torch.no_grad():
        out = {"A": tiny_oracle(**A["batch"]).logits, "B": tiny_oracle(**B["batch"]).logits, "A_bf16": m16(**A["batch"]).logits}
    for key, want in (("A", A["logits_sha256"]), ("B", B["logits_sha256"]), ("A_bf16", A["logits_bf16_sha256"])):
        assert tensor_sha256(out[key]) == want, f"oracle logits of case {key} differ from the reference run"
    out["A_bf16"] = out["A_bf16"].float()
    return out
