import ast
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")
WEIGHTS = os.path.join(ROOT, "oracle", "_ref", "weights")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu on the GPU box")
    config.addinivalue_line("markers", "slow: ~1 min of CPU oracle (full-depth student on a 10 s utterance)")
    # the CPU oracles are torch fp32 convs: more than a few dozen threads makes them slower, and on a box whose cgroup
    # quota is below os.cpu_count() a thread per core gets throttled to a crawl
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    torch.set_num_threads(max(1, min(16, n)))


def pytest_collection_modifyitems(config, items):
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device here")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def golden_weights(d):
    return {k[2:]: torch.from_numpy(d[k]) for k in d.files if k.startswith("w:")}


def golden_cfg(d):
    return ast.literal_eval(str(d["cfg"]))


def staged(name):
    p = os.path.join(WEIGHTS, name)
    return p if os.path.exists(p) else None


def load_staged(name):
    p = staged(name)
    if p is None:
        return None
    sd = torch.load(p, map_location="cpu", weights_only=False)
    return sd["generator"] if isinstance(sd, dict) and "generator" in sd else sd


@pytest.fixture(scope="session")
def neb():
    from oracle import hifigan_ref as H
    sd = load_staged("g_00600000")
    if sd is None:
        pytest.skip("trained HiFi-GAN checkpoint not staged (oracle/stage_weights.py)")
    return sd, dict(H.CONFIG_NEB)


def neb_weights():
    """(state_dict, config, trained?) with the shipped generator's architecture: its checkpoint when staged, else seeded
    random weights scaled so that the tests' synthetic mel gives loud (peak 0.6 - 1.0) but unsaturated audio."""
    from oracle import hifigan_ref as H
    cfg = dict(H.CONFIG_NEB)
    sd = load_staged("g_00600000")
    if sd is not None:
        return sd, cfg, True
    return H.random_state_dict(cfg, seed=21, std=0.3, g_scale=0.125), cfg, False


@pytest.fixture(scope="session")
def neb_arch():
    return neb_weights()


@pytest.fixture(scope="session")
def clarinet_weights():
    """(student_sd, teacher_sd, trained?) - shipped checkpoints when staged, else seeded random."""
    from oracle import clarinet_ref as C
    s, t = load_staged("pnn_vocoder.network"), load_staged("nn_vocoder.network")
    if s is not None and t is not None:
        return s, t, True
    return C.random_state_dict("student", 1), C.random_state_dict("teacher", 2), False
