import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")
# The CPU oracle is compared bit for bit with fixtures the reference produced on 8 intra-op threads.  The last bits of
# its fp32 GEMMs depend on the number of threads the work is split over (1, 2 or 4 threads give other encoder outputs
# than 8), so every test starts from this count instead of whatever the machine or an earlier test left.
ORACLE_THREADS = 8


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu on the GPU box")


@pytest.fixture(autouse=True)
def oracle_threads():
    import torch
    torch.set_num_threads(ORACLE_THREADS)


def load_golden(name):
    with open(os.path.join(GOLDEN, name + ".json")) as f:
        meta = json.load(f)
    arrays = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    return meta, arrays


def weights_checksum(sd):
    import torch
    return float(sum(v.double().abs().sum().item() for k, v in sorted(sd.items()) if v.is_floating_point()))


@pytest.fixture(scope="session")
def golden_cases():
    return {n: load_golden(n) for n in ("causal_ln", "sym_bn")}


@pytest.fixture(scope="session")
def model_dirs(tmp_path_factory, golden_cases):
    """Synthetic model directories + wavs regenerated from the seeds stored with the golden fixtures."""
    import torch
    from reverb_b200 import synth
    out = {}
    for name, (meta, _) in golden_cases.items():
        d = str(tmp_path_factory.mktemp(name))
        synth.write_model_dir(d, causal=meta["causal"], cnn_module_norm=meta["cnn_module_norm"],
                              seed=meta["model_seed"], blank_rate=meta["blank_rate"])
        sd = torch.load(os.path.join(d, "synth.pt"))
        cs = weights_checksum(sd)
        assert abs(cs - meta["weights_checksum"]) <= 1e-6 * abs(meta["weights_checksum"]), \
            "synthetic weight generator drifted from the one that produced tests/golden"
        wav = synth.write_wav(os.path.join(d, "golden.wav"), synth.synth_audio(meta["audio_seconds"], seed=meta["audio_seed"]))
        out[name] = (d, wav)
    return out


@pytest.fixture(scope="session")
def bench_model_dir(tmp_path_factory):
    """Synthetic model directory at the BENCHMARKED shape (reverb_asr_v1-like: d=1024, L=18, V=10001), the same
    weights bench.py times (seed 0, causal conv, LayerNorm conv-module norm, right decoder present)."""
    from reverb_b200 import synth
    d = str(tmp_path_factory.mktemp("bench_shape"))
    synth.write_model_dir(d, shape=synth.BENCH_SHAPE, seed=0, causal=True, cnn_module_norm="layer_norm",
                          reverse_weight=0.3)
    return d
