"""Streaming HiFi-GAN on the GPU: cube_voc_forward_range and stream sessions are bit-identical to the whole-utterance
call, write nothing outside the requested samples, and reject what they do not cover."""
import os
import random

import pytest
import torch

from conftest import neb_weights
from oracle import hifigan_ref as H

pytestmark = pytest.mark.gpu
MATHS = [pytest.param(0, id="fp32_simt"), pytest.param(1, id="tcgen05_split16")]
CONFIG_V3_SHAPE = {
    "resblock": "2", "upsample_rates": [8, 8, 4], "upsample_kernel_sizes": [16, 16, 8], "upsample_initial_channel": 128,
    "resblock_kernel_sizes": [3, 5, 7], "resblock_dilation_sizes": [[1, 2], [2, 6], [3, 12]], "num_mels": 80,
}


def _gen(cfg, sd, math):
    import tts_cube_b200 as cube
    g = cube.CubeGenerator(cfg, math=math).to("cuda:0")
    g.load_state_dict(sd)
    return g.eval()


_GENS = {}


def _neb(math):
    if math not in _GENS:
        sd, cfg, _ = neb_weights()
        _GENS[math] = _gen(cfg, sd, math)
    return _GENS[math]


def _ranges(T, hop, u0, rng, n):
    """random sub-ranges plus single samples, ends on phase boundaries of the first ConvT and the length-law tail"""
    out = [(0, 1), (T - 1, T), (0, T), (T - 96, T), (hop * 3, hop * 3 + u0), (u0 * 7, u0 * 11), (T // 2, T // 2 + 1)]
    for _ in range(n):
        a = rng.randrange(T)
        out.append((a, min(T, a + rng.randint(1, 4 * hop))))
    return [(a, b) for a, b in out if 0 <= a < b <= T]


def _check_range_equals_forward(g, mel, nf, int16, rng):
    B = mel.shape[0]
    whole = g.forward_int16(mel, nf)[1] if int16 else g(mel, nf)
    whole = whole.reshape(B, -1)
    lens = [g.out_len(f) for f in nf]
    per_item = [_ranges(L, g.hop, int(g._cfg.upsample_rates[0]), rng, 6) for L in lens]
    for k in range(max(len(r) for r in per_item)):
        begin = [per_item[b][k % len(per_item[b])][0] for b in range(B)]
        end = [per_item[b][k % len(per_item[b])][1] for b in range(B)]
        pieces = g.forward_range(mel, nf, begin, end, int16=int16)
        for b in range(B):
            want = whole[b, begin[b]:end[b]]
            assert pieces[b].shape == want.shape
            assert torch.equal(pieces[b], want), (b, begin[b], end[b], (pieces[b].float() - want.float()).abs().max())


@pytest.mark.parametrize("math", MATHS)
@pytest.mark.parametrize("int16", [False, True], ids=["f32", "i16"])
def test_forward_range_bit_identical_to_forward(math, int16):
    g = _neb(math)
    rng = random.Random(3 + math)
    with torch.no_grad():
        mel1 = H.synthetic_mel(1, 157, seed=1).to("cuda:0")
        _check_range_equals_forward(g, mel1, [157], int16, rng)
        mel3 = H.synthetic_mel(3, 203, seed=2).to("cuda:0")
        _check_range_equals_forward(g, mel3, [203, 61, 148], int16, rng)


def test_forward_range_resblock2_fp32():
    cfg = CONFIG_V3_SHAPE
    sd = H.random_state_dict(cfg, seed=9, std=0.3, g_scale=0.25)
    g = _gen(cfg, sd, 0)
    with torch.no_grad():
        mel = H.synthetic_mel(2, 90, seed=4).to("cuda:0")
        _check_range_equals_forward(g, mel, [90, 37], False, random.Random(5))


@pytest.mark.parametrize("math", MATHS)
def test_forward_range_leaves_other_samples_untouched(math):
    g = _neb(math)
    with torch.no_grad():
        mel = H.synthetic_mel(2, 120, seed=3).to("cuda:0")
        nf = [120, 77]
        whole = g(mel, nf)
        T = whole.shape[-1]
        out = torch.full((2, 1, T), float("nan"), device="cuda:0")
        begin, end = [1000, 5], [4321, 18000]
        g.forward_range(mel, nf, begin, end, out=out)
        for b in range(2):
            assert torch.equal(out[b, 0, begin[b]:end[b]], whole[b, 0, begin[b]:end[b]])
            assert torch.isnan(out[b, 0, :begin[b]]).all() and torch.isnan(out[b, 0, end[b]:]).all()
        o16 = torch.full((2, T), -7, dtype=torch.int16, device="cuda:0")
        g.forward_range(mel, nf, begin, end, int16=True, out=o16)
        w16 = g.forward_int16(mel, nf)[1]
        for b in range(2):
            assert torch.equal(o16[b, begin[b]:end[b]], w16[b, begin[b]:end[b]])
            assert (o16[b, :begin[b]] == -7).all() and (o16[b, end[b]:] == -7).all()


def test_forward_range_errors():
    import ctypes as C
    import tts_cube_b200 as cube
    from tts_cube_b200 import _lib
    g = _neb(1)
    mel = H.synthetic_mel(2, 40, seed=3).to("cuda:0")
    nf = [40, 20]
    T0, T1 = g.out_len(40), g.out_len(20)
    for begin, end in (([0, 0], [T0 + 1, 10]), ([0, 0], [10, T1 + 1]), ([5, 0], [5, 10]), ([-1, 0], [3, 3]), ([9, 0], [3, 3])):
        with pytest.raises(cube.CubeVocError):
            g.forward_range(mel, nf, begin, end)
    for arch in (_lib.ARCH_PWN_STUDENT, _lib.ARCH_UPSAMPLENET):   # the IAF student and UpsampleNet have no range call
        cfg = _lib.VocConfig()
        cfg.arch, cfg.num_mels, cfg.n_flows, cfg.n_upsample = arch, 80, 1, 1
        cfg.res_channels, cfg.skip_channels, cfg.gate_channels, cfg.kernel_size = 128, 128, 256, 3
        cfg.upsample_scales[0] = 4
        h = C.c_void_p()
        _lib.check(_lib.lib().cube_voc_create(C.byref(h), C.byref(cfg), 0))
        try:
            b0, b1 = (C.c_int64 * 1)(0), (C.c_int64 * 1)(1)
            out = torch.zeros(1, 1, 400, device="cuda:0")
            rc = _lib.lib().cube_voc_forward_range(h, C.c_void_p(mel.data_ptr()), None, b0, b1, C.c_void_p(out.data_ptr()),
                                                   None, 1, 40, None)
            assert rc != 0 and b"HiFi-GAN" in _lib.lib().cube_voc_last_error()
        finally:
            _lib.lib().cube_voc_destroy(h)


def _stream_all(g, mels, chunkings, int16=False, start=None):
    """Sessions fed in lock step (session i starts at round start[i]) and stepped together; returns the concatenations."""
    n = len(mels)
    start = start or [0] * n
    streams = [None] * n
    got = [[] for _ in range(n)]
    pos = [0] * n
    r = 0
    while True:
        live = []
        for i in range(n):
            if r < start[i]:
                continue
            if streams[i] is None:
                streams[i] = g.open_stream(int16=int16)
            s, k = streams[i], r - start[i]
            if s.done:
                continue
            if k < len(chunkings[i]):
                c = chunkings[i][k]
                s.feed(mels[i][:, pos[i]:pos[i] + c])
                pos[i] += c
            else:
                s.close_input()
            live.append(i)
        if not live and r >= max(start):
            break
        for i, piece in zip(live, g.step_streams([streams[i] for i in live])):
            got[i].append(piece)
        r += 1
    return [torch.cat(p) for p in got]


def _chunks(F_, size, rng=None):
    out, left = [], F_
    while left > 0:
        c = rng.choice([0, 1, 3, 7, 19, 31, 46, 80]) if rng else size
        c = min(c, left)
        out.append(c)
        left -= c
    return out


@pytest.mark.parametrize("math", MATHS)
def test_stream_equals_whole(math):
    g = _neb(math)
    with torch.no_grad():
        F_ = 211
        mel = H.synthetic_mel(1, F_, seed=6).to("cuda:0")
        want = g(mel)[0, 0, :g.out_len(F_)]
        want16 = g.forward_int16(mel)[1][0, :g.out_len(F_)]
        rng = random.Random(8)
        for size in (1, 7, 31, 32, 46, 200, None):
            got = _stream_all(g, [mel[0]], [_chunks(F_, size, rng if size is None else None)])[0]
            assert torch.equal(got, want), (size, (got - want).abs().max() if got.shape == want.shape else got.shape)
        got16 = _stream_all(g, [mel[0]], [_chunks(F_, 46)], int16=True)[0]
        assert torch.equal(got16, want16)
        short = H.synthetic_mel(1, 5, seed=7).to("cuda:0")
        got = _stream_all(g, [short[0]], [[2, 0, 3]])[0]
        assert torch.equal(got, g(short)[0, 0])
        s = g.open_stream()                        # push / finish
        parts = [s.push(mel[0, :, k:k + 50]) for k in range(0, F_, 50)] + [s.finish()]
        assert torch.equal(torch.cat(parts), want)


@pytest.mark.parametrize("math", MATHS)
def test_sixteen_staggered_sessions(math):
    g = _neb(math)
    rng = random.Random(12)
    with torch.no_grad():
        lens = [rng.randint(3, 260) for _ in range(16)]
        mels = [H.synthetic_mel(1, n, seed=30 + i).to("cuda:0")[0] for i, n in enumerate(lens)]
        chunkings = [_chunks(n, None, rng) for n in lens]
        start = [rng.randint(0, 12) for _ in lens]
        got = _stream_all(g, mels, chunkings, start=start)
        for i, n in enumerate(lens):
            want = g(mels[i][None])[0, 0]
            assert torch.equal(got[i], want), (i, n)


@pytest.mark.parametrize("env", [{"CUBE_TC_WIDE": "0"}, {"CUBE_TC_WIDE": "2"}, {"CUBE_TC_RBFUSE": "0"}, {"CUBE_TC_WIN": "0"},
                                 {"CUBE_TC_CG2": "1"}, {"CUBE_TC_LEAN": "0"}, {"CUBE_RB_PK": "1"}],
                         ids=lambda e: "_".join(f"{k}={v}" for k, v in e.items()))
def test_stream_variants_in_subprocess(env):
    """The kernel switches are read once per process: rerun the range and stream tests of the tensor-core path in a child."""
    import subprocess
    import sys
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-k",
                        "tcgen05 and (stream_equals_whole or bit_identical or sixteen) and not subprocess"],
                       env=dict(os.environ, **env), capture_output=True, text=True, timeout=900)
    tail = (r.stdout or "")[-1500:] + (r.stderr or "")[-500:]
    assert r.returncode == 0, tail
    assert " passed" in r.stdout, tail
