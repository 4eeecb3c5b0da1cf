import os
import sys
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")
# PyTorch splits the CPU oracle's convolution / matmul sums over its intra-op threads, so their rounding depends on the
# thread count; the vectors under tests/golden/ were recorded with 8 threads and several tests compare bit for bit
GOLDEN_THREADS = 8


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA (B200, sm_100a) device; run with -m gpu on the GPU box")


def pytest_collection_modifyitems(config, items):
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(autouse=True)
def golden_threads():
    import torch
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


@pytest.fixture(scope="session")
def golden():
    import torch

    def load(name):
        return torch.load(os.path.join(GOLDEN, name), map_location="cpu", weights_only=False)
    return load


@pytest.fixture(scope="session")
def parity_log():
    """record(stage, got, ref): appends the measured error of one comparison to gpurun_out/r02_parity_errors.jsonl
    (tools/parity_table.py turns the file into profiles/r02_parity_errors.md); returns (max_abs, max_rel)."""
    import json
    import torch
    out_dir = os.path.join(ROOT, "gpurun_out")
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, "r02_parity_errors.jsonl")

    def record(stage, got, ref, tol=None):
        a, b = got.detach().float().cpu(), ref.detach().float().cpu()
        err = (a - b).abs()
        rms = b.pow(2).mean().sqrt().item()
        # worst violation of |err| <= atol + rtol |ref| expressed as the rtol needed at atol = 1e-4
        need_rtol = ((err - 1e-4).clamp(min=0) / b.abs().clamp(min=1e-12)).max().item()
        rec = dict(stage=stage, max_abs=err.max().item(), mean_abs=err.mean().item(), ref_rms=rms, ref_max=b.abs().max().item(),
                   rtol_needed_at_atol1e4=need_rtol, n=a.numel(), tol=tol)
        with open(path, "a") as f:
            f.write(json.dumps(rec) + "\n")
        return rec["max_abs"], need_rtol
    return record
