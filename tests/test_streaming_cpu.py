"""Streaming HiFi-GAN without a GPU: the layer geometry (cube_voc_hifigan_support) against perturbation of the CPU oracle,
the stream schedule driven through the oracle, and the C ABI of the two streaming entry points."""
import ctypes as C
import os
import random
import re

import pytest
import torch

from oracle import hifigan_ref as H
from tts_cube_b200 import CubeGenerator, _lib
from tts_cube_b200.streaming import HifiganStream, step_streams

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SMALL = dict(upsample_initial_channel=32)
CONFIG_V3_SHAPE = {   # hifigan/config_v3.json's shape: ResBlock2, three stages
    "resblock": "2", "upsample_rates": [8, 8, 4], "upsample_kernel_sizes": [16, 16, 8], "upsample_initial_channel": 32,
    "resblock_kernel_sizes": [3, 5, 7], "resblock_dilation_sizes": [[1, 2], [2, 6], [3, 12]], "num_mels": 80,
}
CONFIGS = {
    "neb": dict(H.CONFIG_NEB, **SMALL),      # shipped generator's geometry, [3, 5, 4, 4]
    "v1": dict(H.CONFIG_V1, **SMALL),        # [5, 3, 4, 4]
    "v3": CONFIG_V3_SHAPE,
}


def _gen(cfg):
    return CubeGenerator(cfg, math=_lib.MATH_FP32_SIMT)


def _oracle(cfg, seed):
    sd = H.random_state_dict(cfg, seed=seed, std=0.3, g_scale=0.5)
    return lambda mel: H.generator_forward(sd, cfg, mel, dtype=torch.float64)


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_sample_support_matches_oracle_perturbation(name):
    cfg = CONFIGS[name]
    g = _gen(cfg)
    fwd = _oracle(cfg, seed=3)
    F_ = 72
    mel = H.synthetic_mel(1, F_, seed=5).to(torch.float64)
    base = fwd(mel)[0, 0]
    T = base.shape[0]
    changed = torch.zeros(F_, T, dtype=torch.bool)
    for f in range(F_):
        m = mel.clone()
        m[0, :, f] += 1.0
        changed[f] = fwd(m)[0, 0] != base
    hop = g.hop
    rng = random.Random(11)
    ranges = [(0, 1), (T - 1, T), (0, T), (hop * 36, hop * 36 + 1), (hop * 36 - 1, hop * 37 + 1)]
    ranges += [(s, s + rng.randint(1, 3 * hop)) for s in (rng.randrange(T - 1) for _ in range(12))]
    for s0, s1 in ranges:
        s1 = min(s1, T)
        f0, f1 = g.sample_support(s0, s1)
        frames = changed[:, s0:s1].any(dim=1).nonzero().flatten().tolist()
        assert frames, (s0, s1)
        assert f0 <= frames[0] and frames[-1] < f1, (name, s0, s1, f0, f1, frames[0], frames[-1])   # sound
        assert frames[0] - f0 <= 1, (name, s0, s1, f0, frames[0])                                    # tight
        if f1 <= F_:
            assert f1 - 1 - frames[-1] <= 1, (name, s0, s1, f1, frames[-1])


def test_sample_support_rejects_bad_arguments():
    g = _gen(CONFIGS["neb"])
    for s0, s1 in ((5, 5), (6, 5), (-1, 3)):
        with pytest.raises(_lib.CubeVocError):
            g.sample_support(s0, s1)
    cfg = _lib.VocConfig()
    cfg.arch = _lib.ARCH_PWN_STUDENT
    f0, f1 = C.c_int64(), C.c_int64()
    assert _lib.lib().cube_voc_hifigan_support(C.byref(cfg), 0, 10, C.byref(f0), C.byref(f1)) != 0


def _oracle_range(fwd):
    def vocode_range(mb, n_frames, begin, end):
        out = []
        for b in range(mb.shape[0]):
            y = fwd(mb[b:b + 1, :, :n_frames[b]])[0, 0]
            assert end[b] <= y.shape[0]
            out.append(y[begin[b]:end[b]])
        return out
    return vocode_range


def _stream(g, cfg):
    return HifiganStream(g.sample_support, lambda n: H.out_len(cfg, n), g.hop, 80)


def _run(streams, chunks_of, mels, vr):
    """Feed every stream its chunks in lock step (one step per round, all streams batched); returns the pieces."""
    got = [[] for _ in streams]
    pos = [0] * len(streams)
    rounds = max(len(c) for c in chunks_of) + 1
    for r in range(rounds):
        for i, s in enumerate(streams):
            if r < len(chunks_of[i]):
                n = chunks_of[i][r]
                s.feed(mels[i][:, pos[i]:pos[i] + n])
                pos[i] += n
            elif not s.closed:
                s.close_input()
        for i, piece in enumerate(step_streams(streams, vr)):
            got[i].append(piece)
    return [torch.cat(p) if p else torch.zeros(0) for p in got]


def _chunking(F_, rng, kind):
    if kind == "ones":
        return [1] * F_
    out, left = [], F_
    while left > 0:
        n = min(left, rng.choice([0, 1, 2, 5, 17, 31, 46, 64]))
        out.append(n)
        left -= n
    return out


@pytest.mark.parametrize("name", ["neb", "v3"])
def test_stream_schedule_concatenates_to_whole_utterance(name):
    cfg = CONFIGS[name]
    g = _gen(cfg)
    fwd = _oracle(cfg, seed=4)
    vr = _oracle_range(fwd)
    rng = random.Random(7)
    lengths = [90, 5, 1, 40, 3]        # 5, 1 and 3 frames are shorter than the ~31-frame halo
    kinds = ["rand", "ones", "rand", "ones", "rand"]
    mels = [H.synthetic_mel(1, n, seed=10 + i)[0].to(torch.float64) for i, n in enumerate(lengths)]
    chunks = [_chunking(n, rng, k) for n, k in zip(lengths, kinds)]
    chunks[2] = [0, 0, 1]              # empty pushes, then the only frame
    streams = [_stream(g, cfg) for _ in lengths]
    got = _run(streams, chunks, mels, vr)
    for i, n in enumerate(lengths):
        want = fwd(mels[i][None])[0, 0]
        assert want.shape[0] == H.out_len(cfg, n)
        assert got[i].shape == want.shape, (i, got[i].shape, want.shape)
        assert torch.allclose(got[i], want, rtol=0, atol=1e-12), (i, (got[i] - want).abs().max())
        assert streams[i].done


def test_stream_keeps_only_frames_it_can_still_need():
    cfg = CONFIGS["neb"]
    g = _gen(cfg)
    fwd = _oracle(cfg, seed=4)
    s = _stream(g, cfg)
    mel = H.synthetic_mel(1, 400, seed=2)[0].to(torch.float64)
    for k in range(0, 400, 40):
        s.feed(mel[:, k:k + 40])
        step_streams([s], _oracle_range(fwd))
        assert s.kept_frames() <= 40 + 2 * 33, s.kept_frames()
    assert s.emitted > 0


def test_streaming_abi_declared_and_bound():
    hdr = open(os.path.join(ROOT, "include", "cube_vocoder.h")).read()
    for name in ("cube_voc_hifigan_support", "cube_voc_forward_range"):
        assert re.search(r"\bint\s+%s\s*\(" % name, hdr), name
        assert name in _lib.SYMBOLS
        assert getattr(_lib.lib(), name).argtypes is not None
    assert C.sizeof(_lib.VocConfig) == 524     # cube_voc_config keeps its size
