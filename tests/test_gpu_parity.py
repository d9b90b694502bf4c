"""Parity of the CUDA path (through the C ABI) with the CPU oracle and the reference-generated golden
fixtures.  Tolerance for waveforms: 1e-3 max-abs on fp32 samples (BASELINE.json north_star); integer
work (mu-law codes, int16 audio away from rounding ties) is bit-exact."""
import numpy as np
import pytest
import torch

from conftest import golden_cfg, golden_weights, load_golden
from oracle import clarinet_ref as C, heads_ref as W, hifigan_ref as H

pytestmark = pytest.mark.gpu
TOL = 1e-3
MATHS = [pytest.param(0, id="fp32_simt"), pytest.param(1, id="tcgen05_split16")]
# The student's default tensor-core path runs GEMM1's two correction passes on 8-bit operands (CUBE_TC_FP8, default on):
# inside the 1e-3 budget with a 20-40x margin, but no longer at fp32 round-off - the CPU emulation
# (profiles/r1_split_precision_study.md) predicts 3e-5 .. 5e-5.  CUBE_TC_FP8=0 (three fp16 passes) is held to the tight bounds.
FP8 = __import__("os").environ.get("CUBE_TC_FP8", "1") != "0"


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def _gen(cfg, sd, dev, math=0):
    import tts_cube_b200 as cube
    g = cube.CubeGenerator(cfg, math=math).to(dev)
    g.load_state_dict(sd)
    return g.eval()



def _cached_oracle(tag, fn):
    """CPU oracle results of the long cases are cached in the temporary directory, one cache per user: the kernel-variant
    tests re-run this file in child processes (one per env switch) and would otherwise repeat a 45 s CPU run each time."""
    import hashlib
    import os
    import tempfile
    d = os.path.join(tempfile.gettempdir(), f"cube_oracle_cache_{os.getuid()}")
    p = os.path.join(d, hashlib.sha1(tag.encode()).hexdigest()[:16] + ".pt")
    if os.path.exists(p):
        try:
            return torch.load(p)
        except Exception:
            pass
    y = fn()
    try:
        os.makedirs(d, exist_ok=True)
        torch.save(y, p + f".{os.getpid()}.tmp")
        os.replace(p + f".{os.getpid()}.tmp", p)
    except OSError:     # a cache that cannot be written only costs time
        pass
    return y


def _report(name, y, ref):
    """max-abs error and where it occurs"""
    e = (y - ref).abs()
    k = int(e.argmax())
    idx = np.unravel_index(k, tuple(e.shape))
    err = float(e.reshape(-1)[k])
    print(f"{name}: max-abs {err:.3e} at {tuple(int(i) for i in idx)} of {tuple(e.shape)} (peak {float(ref.abs().max()):.2f}, rms err {float(e.pow(2).mean().sqrt()):.2e})")
    return err


# ------------------------------------------------ Path H ------------------------------------------------
@pytest.mark.parametrize("name", ["hifigan_mini.npz", "hifigan_mini_rb2.npz"])
def test_hifigan_golden_mini(dev, name):
    d = load_golden(name)
    g = _gen(golden_cfg(d), golden_weights(d), dev)
    with torch.no_grad():
        y = g(torch.from_numpy(d["mel"]).to(dev)).cpu().numpy()
    assert y.shape == d["wav"].shape
    err = float(np.abs(y - d["wav"]).max())
    assert err <= TOL, err
    assert err <= 2e-5, f"fp32 SIMT path should sit near fp32 round-off, got {err}"


@pytest.mark.parametrize("math", MATHS)
def test_hifigan_golden_trained(dev, neb, math):
    sd, cfg = neb
    d = load_golden("hifigan_neb.npz")
    g = _gen(cfg, sd, dev, math)
    with torch.no_grad():
        wav, w16 = g.forward_int16(torch.from_numpy(d["mel"]).to(dev))
    err = float(np.abs(wav.cpu().numpy() - d["wav"]).max())
    print(f"hifigan trained golden math={math}: max-abs {err:.3e} (peak {float(np.abs(d['wav']).max()):.2f})")
    assert err <= TOL, err
    # int16 epilogue: identical wherever the float product is not within fp32 noise of an integer
    ref16 = d["wav_int16"].astype(np.int32)
    got16 = w16.cpu().numpy().astype(np.int32)
    assert np.abs(got16 - ref16).max() <= int(32767 * err) + 1
    v = d["wav"].squeeze(1).astype(np.float64) * 32767
    mism = got16 != ref16                                     # only where truncation sits on an integer edge
    assert mism.mean() <= 4 * 32767 * err + 1e-3              # a flip needs v within 32767*err of an integer
    assert np.all(np.abs(v - np.round(v))[mism] <= 32767 * err + 1e-3)
    # and exactly int16(wav*32767) of the wav it returned (cube/api.py:65)
    assert torch.equal(w16.cpu(), H.wav_to_int16(wav.cpu()).squeeze(1))


@pytest.mark.parametrize("math", MATHS)
@pytest.mark.parametrize("level", [-5.0, 0.0, 1.0])
def test_hifigan_trained_loudness_sweep(dev, neb_arch, level, math):
    sd, cfg, _ = neb_arch
    mel = H.synthetic_mel(2, 40, seed=1237 + int(level), level=level)
    ref = H.generator_forward(sd, cfg, mel)
    g = _gen(cfg, sd, dev, math)
    with torch.no_grad():
        y = g(mel.to(dev)).cpu()
    print(f"hifigan level={level} math={math}: max-abs {float((y - ref).abs().max()):.3e} (peak {float(ref.abs().max()):.2f})")
    assert float((y - ref).abs().max()) <= TOL
    if level >= 0:
        assert float(ref.abs().max()) > 0.5  # loud: the tolerance check means something


@pytest.mark.parametrize("math,c0,gs", [pytest.param(0, 64, 0.36, id="fp32_simt"), pytest.param(1, 512, 0.125, id="tcgen05_split16")])
def test_hifigan_config_v1_random_weights_ragged(dev, math, c0, gs):
    cfg = dict(H.CONFIG_V1, upsample_initial_channel=c0)
    sd = H.random_state_dict(cfg, seed=21, std=0.3, g_scale=gs)
    mel = H.synthetic_mel(3, 21, seed=8)
    frames = [21, 1, 12]
    ref = H.generator_forward_ragged(sd, cfg, mel, frames)
    assert float(ref.abs().max()) > 0.05
    mel_pad = mel.clone()
    mel_pad[1, :, 1:] = -5.0   # VocoderCollate pads with -5 (cube/io_utils/io_vocoder.py:86): must be ignored
    mel_pad[2, :, 12:] = 7.0
    g = _gen(cfg, sd, dev, math)
    with torch.no_grad():
        y = g(mel_pad.to(dev), n_frames=frames).cpu()
    assert y.shape == ref.shape
    print(f"hifigan v1 ragged math={math}: max-abs {float((y - ref).abs().max()):.3e} (peak {float(ref.abs().max()):.2f})")
    assert float((y - ref).abs().max()) <= TOL
    for b, f in enumerate(frames):
        tail = y[b, 0, H.out_len(cfg, f):]
        assert tail.numel() == 0 or float(tail.abs().max()) == 0.0


def test_hifigan_edge_cases(dev):
    import tts_cube_b200 as cube
    cfg = dict(H.CONFIG_V1, upsample_initial_channel=32)
    sd = H.random_state_dict(cfg, seed=11, std=0.3, g_scale=0.42)
    g = _gen(cfg, sd, dev)
    with torch.no_grad():
        one = g(H.synthetic_mel(1, 1, seed=1).to(dev))        # a single frame
        assert one.shape == (1, 1, H.out_len(cfg, 1))
        ref = H.generator_forward(sd, cfg, H.synthetic_mel(1, 1, seed=1))
        assert float((one.cpu() - ref).abs().max()) <= TOL
        z = g(H.synthetic_mel(2, 5, seed=2).to(dev), n_frames=[0, 5]).cpu()  # an empty utterance in a batch
        assert float(z[0].abs().max()) == 0.0
        with pytest.raises(cube.CubeVocError):
            g(torch.zeros(1, 80, 4))                             # CPU tensor: no fallback
        with pytest.raises(cube.CubeVocError):
            g(torch.zeros(1, 80, 4, device=dev), n_frames=[9])   # n_frames > Fmax
    bad = cube.CubeGenerator(cfg).to(dev)
    sd2 = dict(sd)
    del sd2["ups.1.bias"]
    bad.load_state_dict(sd2)
    with pytest.raises(cube.CubeVocError, match="ups.1.bias"):
        bad(torch.zeros(1, 80, 4, device=dev))                  # strict load like the reference
    x = torch.zeros(1, 80, 4, device=dev, requires_grad=True)
    with pytest.raises(cube.CubeVocError):
        g(x)                                                    # inference only


def test_hifigan_host_call_matches_device_call(dev):
    cfg = dict(H.CONFIG_V1, upsample_initial_channel=32)
    sd = H.random_state_dict(cfg, seed=11, std=0.3, g_scale=0.42)
    g = _gen(cfg, sd, dev)
    mel = H.synthetic_mel(2, 17, seed=3)
    with torch.no_grad():
        a = g(mel.to(dev)).cpu().squeeze(1)
    b = g.forward_host(mel.pin_memory())
    assert torch.equal(a, b)
    c = g.forward_host(mel, int16=True)
    assert torch.equal(c, H.wav_to_int16(a))


def test_forward_host_graph_replay(dev):
    """cube_voc_forward_host replays a CUDA graph from the second call with a geometry on: results must stay identical to
    the stream-launched device call for changing inputs and changing n_frames masks (the graph bakes in neither), after
    a geometry change (workspace growth invalidates older graphs) and when coming back to the first geometry."""
    cfg = dict(H.CONFIG_V1)
    sd = H.random_state_dict(cfg, seed=21, std=0.3, g_scale=0.125)
    g = _gen(cfg, sd, dev, 1)
    ssd, tsd = C.random_state_dict("student", 3, blocks=[6, 1, 1, 2]), C.random_state_dict("teacher", 4, blocks=[1])
    v = _student(ssd, tsd, dev, 1)
    for rnd, (B, F_) in enumerate([(2, 9), (2, 9), (2, 9), (3, 14), (2, 9), (2, 9)]):
        mel = H.synthetic_mel(B, F_, seed=300 + rnd)
        frames = [F_] + [max(1, F_ - 2 - rnd - b) for b in range(1, B)]
        with torch.no_grad():
            a = g(mel.to(dev), n_frames=frames).cpu().squeeze(1)
        assert torch.equal(g.forward_host(mel.pin_memory(), n_frames=frames), a), (rnd, "hifigan")
        i16 = g.forward_host(mel, n_frames=frames, int16=True)
        assert torch.equal(i16, H.wav_to_int16(a)), (rnd, "hifigan int16")
        melc = C.synthetic_mel01(B, F_, seed=400 + rnd)
        z = torch.randn(B, 1, F_ * 256, generator=torch.Generator().manual_seed(500 + rnd))
        with torch.no_grad():
            d_ = v(melc.to(dev), z.to(dev), n_frames=frames).cpu().squeeze(1)
        assert torch.equal(v.forward_host(melc.pin_memory(), z.pin_memory(), n_frames=frames), d_), (rnd, "student")
    import tts_cube_b200 as cube
    with pytest.raises(cube.CubeVocError):
        g.forward_host(H.synthetic_mel(2, 9, seed=1), n_frames=[9, 10])        # n_frames > Fmax is still rejected on the replay path


@pytest.mark.parametrize("math", MATHS)
def test_hifigan_full_size_properties(dev, neb_arch, math):
    """BASELINE config 3 shape (10 s utterances) through size-independent properties: batch items are
    independent and a long utterance equals the same utterance inside a padded batch."""
    sd, cfg, _ = neb_arch
    g = _gen(cfg, sd, dev, math)
    F = 919
    mel = H.synthetic_mel(2, F, seed=77)
    with torch.no_grad():
        y2 = g(mel.to(dev))
        y1 = g(mel[1:2].to(dev))
        short = g(torch.cat([mel[:1], mel[:1]], 0).to(dev), n_frames=[F, 300])
    assert y2.shape == (2, 1, H.out_len(cfg, F))
    assert torch.equal(y2[1], y1[0])                       # no cross-utterance leakage, deterministic
    assert torch.equal(short[0], y2[0])
    alone = g(mel[:1, :, :300].contiguous().to(dev))
    assert torch.equal(short[1, :, : alone.shape[2]], alone[0])
    assert float(y2.abs().max()) > 0.5 and bool(torch.isfinite(y2).all())
    # oracle spot-check on the first second only would need the full receptive field; instead check the
    # head of the utterance against the oracle run on a prefix long enough to cover it
    pre = H.generator_forward(sd, cfg, mel[:1, :, :64])
    n = H.out_len(cfg, 40)
    assert float((y2[0, 0, :n].cpu() - pre[0, 0, :n]).abs().max()) <= TOL
    if math == 1:   # tensor-core path against the fp32 path over the whole 10 s
        with torch.no_grad():
            ys = _gen(cfg, sd, dev, 0)(mel.to(dev))
        print(f"hifigan 10 s tc-vs-fp32: max-abs {float((y2 - ys).abs().max()):.3e}")
        assert float((y2 - ys).abs().max()) <= 5e-4


@pytest.mark.parametrize("math", MATHS)
@pytest.mark.parametrize("level", [0.0, 1.0])
def test_hifigan_full_length_oracle(dev, neb_arch, level, math):
    """BASELINE configs[2] geometry, compared with the oracle over the WHOLE 10-s utterance (F = 919, T = 220 656), the
    shipped generator (seeded weights of its architecture when the checkpoint is not staged), speech level (0) and the
    saturating corner (+1), both math modes.  hifigan/models.py:100-116."""
    sd, cfg, trained = neb_arch
    F = 919
    mel = H.synthetic_mel(2, F, seed=177 + int(level), level=level)
    ref = _cached_oracle(f"hifigan_neb_full_F{F}_lvl{level}_seed{177 + int(level)}_trained{trained}", lambda: H.generator_forward(sd, cfg, mel))
    g = _gen(cfg, sd, dev, math)
    with torch.no_grad():
        y = g(mel.to(dev)).cpu()
    assert y.shape == ref.shape == (2, 1, H.out_len(cfg, F))
    err = _report(f"hifigan 10 s full oracle level={level} math={math}", y, ref)
    assert float(ref.abs().max()) > 0.5
    assert err <= TOL


# ------------------------------------------------ Path C ------------------------------------------------
def _student(ssd, tsd, dev, math=0):
    import tts_cube_b200 as cube
    return cube.ParallelWaveNetVocoder(ssd, tsd, math=math).to(dev).eval()



def test_upsample2_golden(dev):
    d = load_golden("upsample2.npz")
    tsd = golden_weights(d)
    ssd = C.random_state_dict("student", 5, blocks=[1, 1])
    v = _student(ssd, tsd, dev)
    mel = torch.from_numpy(d["mel"])
    T = mel.shape[2] * 256
    with torch.no_grad():
        v(mel.to(dev), torch.zeros(1, 1, T, device=dev))
    c = v.conditioning(1, T).cpu().numpy()
    assert float(np.abs(c - d["c_up"]).max()) <= 1e-5


@pytest.mark.parametrize("math", MATHS)
def test_student_small_random_weights(dev, math):
    ssd, tsd = C.random_state_dict("student", 3, blocks=[7, 2, 1, 3]), C.random_state_dict("teacher", 4, blocks=[1])
    mel = C.synthetic_mel01(2, 5, seed=2)
    z = torch.randn(2, 1, 5 * 256, generator=torch.Generator().manual_seed(1))
    ref = C.vocode_student(ssd, tsd, mel, z)
    v = _student(ssd, tsd, dev, math)
    with torch.no_grad():
        x = v(mel.to(dev), z.to(dev)).cpu()
    err = float((x - ref).abs().max())
    print(f"student small math={math}: max-abs {err:.3e} (peak {float(ref.abs().max()):.2f})")
    assert float(ref.abs().max()) > 0.05
    assert err <= TOL
    assert err <= (3e-4 if FP8 and math == 1 else 5e-5)   # both default math modes sit near fp32 round-off


@pytest.mark.parametrize("math", MATHS)
def test_student_shipped_weights(dev, clarinet_weights, math):
    ssd, tsd, trained = clarinet_weights
    mel = C.synthetic_mel01(2, 8, seed=8)
    z = torch.randn(2, 1, 8 * 256, generator=torch.Generator().manual_seed(9))
    ref = C.vocode_student(ssd, tsd, mel, z)
    v = _student(ssd, tsd, dev, math)
    with torch.no_grad():
        x = v(mel.to(dev), z.to(dev)).cpu()
    err = float((x - ref).abs().max())
    print(f"student shipped={trained} math={math}: max-abs {err:.3e} (peak {float(ref.abs().max()):.2f})")
    assert float(ref.abs().max()) > 0.1
    assert err <= TOL
    if trained:
        d = load_golden("clarinet_regress.npz")
        with torch.no_grad():
            xr = v(torch.from_numpy(d["mel"]).to(dev), torch.from_numpy(d["z"]).to(dev)).cpu().numpy()
        assert float(np.abs(xr - d["wav"]).max()) <= TOL


@pytest.mark.parametrize("math", MATHS)
def test_student_ragged_and_causal(dev, math):
    ssd, tsd = C.random_state_dict("student", 3, blocks=[6, 1, 1, 2]), C.random_state_dict("teacher", 4, blocks=[1])
    mel = C.synthetic_mel01(2, 6, seed=12)
    z = torch.randn(2, 1, 6 * 256, generator=torch.Generator().manual_seed(3))
    v = _student(ssd, tsd, dev, math)
    mel_pad = mel.clone()
    mel_pad[1, :, 4:] = 9.0
    with torch.no_grad():
        x = v(mel_pad.to(dev), z.to(dev), n_frames=[6, 4]).cpu()
    alone = C.vocode_student(ssd, tsd, mel[1:2, :, :4], z[1:2, :, : 4 * 256])
    assert float((x[1, :, : 4 * 256] - alone[0]).abs().max()) <= TOL
    assert float(x[1, :, 4 * 256:].abs().max()) == 0.0
    full = C.vocode_student(ssd, tsd, mel[:1], z[:1])
    assert float((x[0] - full[0]).abs().max()) <= TOL
    # host-buffer call == device call
    with torch.no_grad():
        d_ = v(mel.to(dev), z.to(dev)).cpu().squeeze(1)
    assert torch.equal(v.forward_host(mel.pin_memory(), z.pin_memory()), d_)


@pytest.mark.parametrize("math", MATHS)
def test_student_full_length_properties(dev, math):
    """Config-2 length (10 s, T=220672) with a shallow student: finite, deterministic, causal (a change
    of z at sample s never alters samples < s) and batch items independent."""
    ssd, tsd = C.random_state_dict("student", 3, blocks=[6, 1]), C.random_state_dict("teacher", 4, blocks=[1])
    F = 862
    mel = C.synthetic_mel01(2, F, seed=5)
    g = torch.Generator().manual_seed(11)
    z = torch.randn(2, 1, F * 256, generator=g)
    v = _student(ssd, tsd, dev, math)
    with torch.no_grad():
        a = v(mel.to(dev), z.to(dev))
        z2 = z.clone()
        s = 150000
        z2[0, 0, s:] += 1.0
        b = v(mel.to(dev), z2.to(dev))
    assert bool(torch.isfinite(a).all())
    assert torch.equal(a[0, 0, :s], b[0, 0, :s]) and not torch.equal(a[0, 0, s:], b[0, 0, s:])
    assert torch.equal(a[1], b[1])
    # head of the utterance against the oracle (causal: a prefix is self-contained)
    n = 3 * 256
    ref = C.vocode_student(ssd, tsd, mel[:1, :, :8], z[:1, :, : 8 * 256])
    assert float((a[0, 0, :n].cpu() - ref[0, 0, :n]).abs().max()) <= TOL
    # and the tensor-core path against the fp32 SIMT path over the WHOLE 10 s utterance
    if math == 1:
        with torch.no_grad():
            s_ = _student(ssd, tsd, dev, 0)(mel.to(dev), z.to(dev))
        assert float((a - s_).abs().max()) <= (5e-4 if FP8 else 1e-4)


def _student_case(case, F):
    """inputs of the full-depth parity cases: (mel, z)"""
    mel = C.synthetic_mel01(1, F, seed=31)
    z = torch.randn(1, 1, F * 256, generator=torch.Generator().manual_seed(32))
    if case == "temp0.7":          # the legacy CLI's sampling temperature (examples/tts-colab-demo.ipynb:247)
        z = z * 0.7
    elif case == "loud":           # mel pushed towards 1 (ClariNet-era [0,1] normalisation): a loud, dense spectrum
        mel = mel.sqrt()
    return mel, z


@pytest.mark.parametrize("math", MATHS)
@pytest.mark.parametrize("case,F", [("plain", 173), ("temp0.7", 173), ("loud", 173),
                                    pytest.param("plain", 862, marks=pytest.mark.slow)])
def test_student_shipped_full_depth_oracle(dev, clarinet_weights, case, F, math):
    """The shipped 42-block student ([6,6,6,24] blocks, 4 IAF flows; receptive field 5 220 samples) against the oracle over
    WHOLE utterances: F = 173 (BASELINE configs[0] length, 2 s) and F = 862 (configs[1] length, 10 s: ~45 s of CPU oracle,
    cached on disk for the kernel-variant child processes).  Run for the default kernel (CTA pair + 8-bit correction
    passes), and through test_variants_in_subprocess for CUBE_TC_FP8=0, the single-CTA kernels and the unfused pair."""
    ssd, tsd, trained = clarinet_weights
    mel, z = _student_case(case, F)
    ref = _cached_oracle(f"student_full_{case}_F{F}_trained{trained}", lambda: C.vocode_student(ssd, tsd, mel, z))
    v = _student(ssd, tsd, dev, math)
    with torch.no_grad():
        x = v(mel.to(dev), z.to(dev)).cpu()
    assert x.shape == ref.shape == (1, 1, F * 256)
    err = _report(f"student full depth shipped={trained} case={case} F={F} math={math} fp8={FP8}", x, ref)
    assert bool(torch.isfinite(x).all()) and float(ref.abs().max()) > 0.1
    assert err <= TOL


# ------------------------------------------------ heads ------------------------------------------------
def test_mulaw_bit_exact(dev):
    import tts_cube_b200 as cube
    d = load_golden("heads.npz")
    m = cube.MULAWOutput()
    for xs, qs in ((d["mulaw_x"], d["mulaw_q"]), (d["mulaw_nb_x"], d["mulaw_nb_q"])):
        q = m.encode(torch.from_numpy(xs).to(dev))
        assert q.dtype == torch.int64
        assert np.array_equal(q.cpu().numpy(), qs)
    assert np.array_equal(m.decode(torch.arange(256, device=dev)).cpu().numpy(), d["mulaw_table"])
    assert m.encode(m.decode(torch.arange(256, device=dev))).cpu().tolist() == list(range(256))
    # a large seeded sweep against the oracle restatement, plus shapes / empties
    g = torch.Generator().manual_seed(123)
    x = torch.rand(1 << 20, generator=g) * 2.2 - 1.1
    assert torch.equal(m.encode(x.to(dev)).cpu(), W.mulaw_encode_by_edges(x, d["mulaw_edges"]))
    assert m.encode(torch.zeros(3, 0, device=dev)).shape == (3, 0)
    x3 = torch.rand(2, 5, 7, generator=g) * 2 - 1
    assert torch.equal(m.encode(x3.to(dev)).cpu(), W.mulaw_encode(x3))


def test_raw_mol_gaussian_categorical(dev):
    import tts_cube_b200 as cube
    d = load_golden("heads.npz")
    r = cube.RAWOutput()
    assert np.array_equal(r.encode(torch.from_numpy(d["raw_x"]).to(dev)).cpu().numpy(), d["raw_q"])
    assert np.array_equal(r.decode(torch.arange(256, device=dev)).cpu().numpy(), d["raw_table"])
    y, um, ux = (torch.from_numpy(d[k]) for k in ("mol_y", "mol_u_mix", "mol_u_x"))
    xm = cube.MOLOutput().sample(y.to(dev), u_mix=um.to(dev), u_x=ux.to(dev)).cpu()
    ok = W.mol_argmax_margin(y, um) > 1e-5          # float32 near-ties may legitimately flip the pick
    assert float(ok.float().mean()) > 0.99
    assert float((xm - torch.from_numpy(d["mol_x"]))[ok].abs().max()) <= 1e-5
    xg = cube.GaussianOutput().sample(torch.from_numpy(d["gau_y"]).to(dev), eps=torch.from_numpy(d["gau_eps"]).to(dev)).cpu()
    assert float((xg - torch.from_numpy(d["gau_x"])).abs().max()) <= 1e-6
    g = torch.Generator().manual_seed(5)
    logits = torch.randn(4, 33, 256, generator=g) * 3
    u = torch.empty(4, 33, 256).uniform_(1e-5, 1 - 1e-5, generator=g)
    from tts_cube_b200.heads import _categorical
    idx = _categorical(logits.to(dev), u.to(dev)).cpu()
    ref = W.categorical_sample_gumbel(logits, u)
    ok = W.categorical_margin(logits, u) > 1e-4
    assert torch.equal(idx[ok], ref[ok]) and float(ok.float().mean()) > 0.99
    # sample() = decode(categorical): values come from the 256-entry table
    s = cube.MULAWOutput().sample(logits.to(dev), u.to(dev)).cpu()
    assert torch.equal(s[ok], W.mulaw_decode(ref)[ok])


def test_categorical_distribution(dev):
    """W2: the Gumbel-max sampler is DISTRIBUTION-equivalent to the reference's `Categorical(logits=y).sample()`
    (cube/networks/loss.py:227-229, 288-290) - not replayable draw for draw (torch's sampler consumes its generator
    differently): a chi-square goodness-of-fit of 400 000 draws against softmax(logits), for a peaked and a flat
    256-way distribution, plus a two-sample check against torch's own Categorical on the CPU."""
    from scipy import stats
    from tts_cube_b200.heads import _categorical
    g = torch.Generator().manual_seed(77)
    N, Cn = 400_000, 256
    for scale in (3.0, 0.5):
        logits = torch.randn(Cn, generator=g) * scale
        p = torch.softmax(logits.double(), 0).numpy()
        u = torch.rand(N, Cn, generator=g)            # full-range uniforms (a truncated range biases the rare classes)
        idx = _categorical(logits.expand(N, Cn).contiguous().to(dev), u.to(dev)).cpu().numpy()
        cnt = np.bincount(idx, minlength=Cn).astype(np.float64)
        keep = N * p >= 5                                  # chi-square needs expected counts >= 5: pool the rest
        obs = np.append(cnt[keep], cnt[~keep].sum())
        exp = np.append(N * p[keep], N * p[~keep].sum())
        if exp[-1] < 5:
            obs, exp = obs[:-1], exp[:-1] * (obs[:-1].sum() / exp[:-1].sum())
        chi2 = float(((obs - exp) ** 2 / exp).sum())
        crit = float(stats.chi2.ppf(1 - 1e-6, len(obs) - 1))
        print(f"categorical chi2 scale={scale}: {chi2:.1f} (df {len(obs) - 1}, critical at p=1e-6: {crit:.1f})")
        assert chi2 < crit
        ref = torch.distributions.Categorical(logits=logits).sample((N,)).numpy()    # the reference's sampler, CPU
        rc = np.bincount(ref, minlength=Cn).astype(np.float64)
        both = (cnt + rc) >= 10
        chi2_2 = float((((cnt - rc) ** 2) / (cnt + rc))[both].sum())                   # two-sample chi-square, equal N
        assert chi2_2 < float(stats.chi2.ppf(1 - 1e-6, int(both.sum()) - 1))
    # the default draws of the Python layer (no `u` given) are distribution-correct too
    logits = torch.randn(Cn, generator=g) * 3.0
    p = torch.softmax(logits.double(), 0).numpy()
    idx = _categorical(logits.expand(N, Cn).contiguous().to(dev)).cpu().numpy()
    cnt = np.bincount(idx, minlength=Cn).astype(np.float64)
    keep = N * p >= 5
    chi2 = float(((cnt[keep] - N * p[keep]) ** 2 / (N * p[keep])).sum())
    assert chi2 < float(stats.chi2.ppf(1 - 1e-6, int(keep.sum())))


# ------------------------------------------------ Path W4 / W5 ------------------------------------------------
@pytest.mark.parametrize("head", ["mol", "gm"])
def test_wavernn_golden(dev, head):
    """The persistent WaveRNN kernel replays the reference WaveRNN sample for sample (seeded weights and draws)."""
    import tts_cube_b200 as cube
    d = load_golden(f"wavernn_{head}.npz")
    sd = golden_weights(d)
    v = cube.WaveRNNVocoder(num_layers=2, layer_size=32, upsample=int(d["upsample"]), upsample_low=int(d["upsample_low"]),
                            use_lowres=True, output=head).to(dev)
    v.load_state_dict(sd)
    if head == "mol":
        draws = torch.cat([torch.from_numpy(d["d:u_mix"]), torch.from_numpy(d["d:u_x"]).unsqueeze(2)], dim=2)
    else:
        draws = torch.from_numpy(d["d:eps"]).unsqueeze(2)
    x = v.inference(torch.from_numpy(d["mel"]).to(dev), torch.from_numpy(d["x_low"]).to(dev), draws.to(dev)).cpu().numpy()
    err = float(np.abs(x - d["x"]).max())
    print(f"wavernn {head}: max-abs {err:.3e}")
    assert x.shape == d["x"].shape and err <= 1e-4
    y = v({"mel": torch.from_numpy(d["mel"]), "x_low": torch.from_numpy(d["x_low"])}, draws=draws)
    assert y.shape == d["x"].shape + (1,) and y.dtype == np.float32


@pytest.mark.parametrize("head,H,L,lowres", [("mol", 512, 2, True), ("mulaw", 128, 1, False), ("raw", 64, 2, True), ("gm", 512, 2, False)])
def test_wavernn_vs_oracle(dev, head, H, L, lowres):
    """Full-size geometry (2 x 512 GRU, 20 folded chunks) and the categorical heads against the CPU oracle."""
    import tts_cube_b200 as cube
    from oracle import wavernn_ref as R
    S = {"mol": 30, "gm": 2, "mulaw": 256, "raw": 256}[head]
    sd = R.random_state_dict(H, L, lowres, S, seed=5)
    up, upl, B, Fr = 10, 5, 20, 3
    g = torch.Generator().manual_seed(3)
    mel = torch.rand(B, Fr, 80, generator=g)
    x_low = (torch.rand(B, Fr * up // upl, generator=g) * 1.6 - 0.8) if lowres else None
    T = Fr * up
    v = cube.WaveRNNVocoder(num_layers=L, layer_size=H, upsample=up, upsample_low=upl, use_lowres=lowres, output=head).to(dev)
    v.load_state_dict(sd)
    K = v.draws_shape(B, T)[2]
    draws = torch.randn(T, B, K, generator=g) if head == "gm" else torch.empty(T, B, K).uniform_(1e-5, 1 - 1e-5, generator=g)
    if head == "mol":
        od = {"u_mix": draws[:, :, :10], "u_x": draws[:, :, 10]}
    elif head == "gm":
        od = {"eps": draws[:, :, 0]}
    else:
        od = {"u": draws}
    ref = R.wavernn_inference(sd, mel, x_low, up, upl, head, od)
    x = v.inference(mel.to(dev), x_low.to(dev) if lowres else None, draws.to(dev)).cpu()
    # an autoregressive sampler amplifies a flipped arg-max; rows whose trajectories agree must agree closely,
    # and (seeded) at least 90 % of them do
    rowerr = (x - ref).abs().amax(dim=1)
    good = rowerr <= 2e-3
    print(f"wavernn {head} H={H}: rows ok {int(good.sum())}/{B}, max-abs over ok rows {float(rowerr[good].max()):.3e}")
    assert float(good.float().mean()) >= 0.9


def test_cubenet_vocoder_fold(dev):
    """W5: fold/unfold equals the reference's numpy version; CubenetVocoder runs lr -> fold -> hr -> unfold."""
    import tts_cube_b200 as cube
    from tts_cube_b200.wavernn import fold_batch, unfold_batch
    from oracle import wavernn_ref as R
    mel = torch.rand(1, 43, 80)
    xl = torch.rand(1, 430)
    m, x = fold_batch(mel, xl, 10, 20)
    mr, xr = R.fold_batch(mel, xl, 10, 20)
    assert torch.equal(m, mr) and torch.equal(x, xr)
    y = torch.rand(20, 300)
    assert torch.equal(unfold_batch(y, 100), R.unfold_batch(y, 100))
    voc = cube.CubenetVocoder(2, 64, 2, 64, upsample=20, upsample_low=4, output="mol").to(dev)
    sd = {}
    sd.update({"_wavernn_hr." + k: v for k, v in R.random_state_dict(64, 2, True, 30, seed=1).items()})
    sd.update({"_wavernn_lr." + k: v for k, v in R.random_state_dict(64, 2, False, 30, seed=2).items()})
    voc.load_state_dict(sd)
    x_lr, x_hr = voc({"mel": torch.rand(1, 40, 80)})
    # hr chunk: 3 frames x 20 = 60 vs (10 + 4) low samples x 4 = 56 -> T = 56 (the reference's min()), minus the 20-sample context
    assert x_lr.shape == (1, 40 * 5, 1) and x_hr.shape == (1, 20 * (56 - 20))
    assert np.isfinite(x_lr).all() and bool(torch.isfinite(x_hr).all())


def test_hifigan_tcgen05_edge_cases(dev):
    """Tensor-core path: a single frame (every TMA box mostly out of bounds), an empty utterance in a batch, batch of
    one, odd lengths - against the oracle."""
    cfg = dict(H.CONFIG_V1)
    sd = H.random_state_dict(cfg, seed=21, std=0.3, g_scale=0.125)
    g = _gen(cfg, sd, dev, 1)
    with torch.no_grad():
        for F_, frames in ((1, None), (2, None), (7, [0, 7, 3])):
            B = len(frames) if frames else 1
            mel = H.synthetic_mel(B, F_, seed=40 + F_)
            y = g(mel.to(dev), n_frames=frames).cpu()
            ref = H.generator_forward_ragged(sd, cfg, mel, frames) if frames else H.generator_forward(sd, cfg, mel)
            assert y.shape == ref.shape
            assert float((y - ref).abs().max()) <= TOL, (F_, frames)
            if frames:
                assert float(y[0].abs().max()) == 0.0


def test_integration_stub_runs_verbatim(dev):
    """INTEGRATION.md's raw ctypes stub, executed as written, drives the .so to the reference-made golden."""
    import types
    from test_host_logic import integration_stub_namespace
    ns = integration_stub_namespace()
    d = load_golden("hifigan_mini.npz")
    cfg = golden_cfg(d)
    h = types.SimpleNamespace(**cfg)
    hnd = ns["make_generator"](h, golden_weights(d), device=0)
    with torch.cuda.device(dev):
        wav = ns["generate"](hnd, torch.from_numpy(d["mel"]).to(dev))
        torch.cuda.synchronize()
    assert float(np.abs(wav.cpu().numpy() - d["wav"]).max()) <= 2e-5
    ns["lib"].cube_voc_destroy(hnd)


# ------------------------------------------------ configs[4]: behind the reference Cubegan ------------------------------------------------
def test_cubegan_inference_through_the_drop_in(dev):
    """tests/golden/cubegan_e2e.npz = the unmodified reference `Cubegan.inference` run end to end in the build container
    (oracle/make_cubegan_golden.py): seeded Languasito2 -> conditioning -> reference Generator.  Here the same
    conditioning goes through `install_into_cubegan` + the same 8 lines of `inference` and must give the same wav, and
    the int16 audio of `TTSCube.__call__` (cube/api.py:64-65)."""
    import types
    import tts_cube_b200 as cube
    from test_host_logic import CubeganStandIn, generator_shell
    d = load_golden("cubegan_e2e.npz")
    sd = H.random_state_dict(H.CONFIG_V1, seed=int(d["gen_seed"]), std=float(d["gen_std"]), g_scale=float(d["gen_gscale"]))
    cond = torch.from_numpy(d["conditioning"]).to(dev)                     # [1, F, 80] as Languasito2.inference returns it
    for math in (None, 0):
        model = CubeganStandIn(generator_shell(sd, types.SimpleNamespace(**H.CONFIG_V1)).to(dev), [cond])
        cube.install_into_cubegan(model, math=math)
        assert isinstance(model._generator, cube.CubeGenerator) and model._generator.device == dev
        audio = model.inference({"utt": 0})                                # cube/networks/cubegan.py:74-83
        assert audio.shape == d["wav"].shape
        err = _report(f"cubegan e2e math={math}", audio.cpu(), torch.from_numpy(d["wav"]))
        assert err <= TOL
        a16 = np.asarray(audio.detach().cpu().numpy().squeeze() * 32767, dtype=np.int16)      # cube/api.py:64-65
        assert np.abs(a16.astype(np.int32) - d["wav_int16"].astype(np.int32)).max() <= int(32767 * err) + 1
    # batch > 1 glue: several utterances (different lengths) through the per-utterance frontend and ONE batched vocoder call
    conds = [cond, cond[:, :17].contiguous(), cond[:, :1].contiguous(), cond[:, :0]]
    model = CubeganStandIn(generator_shell(sd, types.SimpleNamespace(**H.CONFIG_V1)).to(dev), conds)
    cube.install_into_cubegan(model)
    wavs = cube.cubegan_inference_batch(model, [{"utt": i} for i in range(4)])
    w16 = cube.cubegan_inference_batch(model, [{"utt": i} for i in range(4)], int16=True)
    for i, c in enumerate(conds):
        if c.shape[1] == 0:                                                # the reference's empty-utterance guard: one zero frame
            c = torch.zeros(1, 1, 80, device=dev)
        ref = H.generator_forward(sd, H.CONFIG_V1, c.permute(0, 2, 1).cpu())[0, 0]
        assert wavs[i].shape == ref.shape and float((wavs[i].cpu() - ref).abs().max()) <= TOL, i
        assert w16[i].dtype == torch.int16 and torch.equal(w16[i].cpu(), H.wav_to_int16(wavs[i].cpu()))
    assert float((wavs[0].cpu() - torch.from_numpy(d["wav"])[0, 0]).abs().max()) <= TOL


def test_upsamplenet_golden_and_oracle(dev):
    """Reference UpsampleNet (cube/networks/modules.py:317-343): reference-run golden, then a wider / longer / ragged case
    (kernel 5, scales [4, 2], livelier weights) against the oracle."""
    import tts_cube_b200 as cube
    from oracle import wavernn_ref as R
    d = load_golden("upsamplenet.npz")
    sd = golden_weights(d)
    scales = [int(s) for s in d["scales"]]
    m = cube.UpsampleNet(scales, int(d["in_channels"]), int(d["out_channels"]), int(d["kernel_size"])).to(dev)
    m.load_state_dict(sd)
    y = m(torch.from_numpy(d["c"]).to(dev)).cpu().numpy()
    assert y.shape == d["y"].shape
    assert float(np.abs(y - d["y"]).max()) <= 1e-6
    g = torch.Generator().manual_seed(3)
    Cin, Co, K, sc = 40, 96, 5, [4, 2]
    sd2 = {}
    ic = Cin
    for i in range(3):
        sd2[f"_conv.{2 * i}.weight"] = torch.randn(Co, ic, K, generator=g) * (1.5 / (ic * K) ** 0.5)
        sd2[f"_conv.{2 * i}.bias"] = torch.randn(Co, generator=g) * 0.1
        ic = Co
    for n, s_ in enumerate(sc):
        sd2[f"_upsample_conv.{2 * n}.weight_v"] = torch.randn(Co, Co, 2 * s_, generator=g) * 0.1
        sd2[f"_upsample_conv.{2 * n}.weight_g"] = 0.5 + torch.rand(Co, 1, 1, generator=g)
        sd2[f"_upsample_conv.{2 * n}.bias"] = torch.randn(Co, generator=g) * 0.1
    m2 = cube.UpsampleNet(sc, Cin, Co, K).to(dev)
    m2.load_state_dict(sd2)
    c = torch.rand(3, Cin, 37, generator=g) * 2 - 1
    frames = [37, 5, 20]
    y2 = m2(c.to(dev), n_frames=frames).cpu()
    assert y2.shape == (3, Co, 37 * 8)
    for b, f in enumerate(frames):
        ref = R.upsamplenet_forward(sd2, c[b:b + 1, :, :f], sc, K)[0]
        assert float(ref.abs().max()) > 0.3
        assert float((y2[b, :, : f * 8] - ref).abs().max()) <= 2e-5, b
        assert f == 37 or float(y2[b, :, f * 8:].abs().max()) == 0.0
    with pytest.raises(cube.CubeVocError):
        cube.UpsampleNet([3], 8, 8, 3).to(dev).forward(torch.zeros(1, 8, 4, device=dev))      # odd scale: rejected


# ------------------------------------------------ mel front-end ------------------------------------------------
MEL_TOL = 2e-4      # log-mel units (fp32 DFT by direct summation vs torch's FFT; measured ~1e-5)


def test_mel_hifigan_golden_and_oracle(dev):
    import tts_cube_b200 as cube
    from oracle import mel_ref as M
    d = load_golden("mel_hifigan.npz")
    for tag in "ab":
        a = [int(v) for v in d[f"args_{tag}"]]
        y = torch.from_numpy(d[f"y_{tag}"])
        mel = cube.mel_spectrogram(y.to(dev), *a).cpu().numpy()
        err = float(np.abs(mel - d[f"mel_{tag}"]).max())
        print(f"mel golden {tag}: max-abs {err:.2e}")
        assert mel.shape == d[f"mel_{tag}"].shape and err <= MEL_TOL
    # longer, ragged batch with a silent stretch (hits the 1e-5 clamp) against the oracle
    n_fft, M_, sr, hop, win, fmin, fmax = 1024, 80, 22050, 256, 1024, 0, 8000
    y = M.test_signal(3, 40000, seed=9)
    y[1, 12000:20000] = 0.0
    lens = [40000, 30000 - 37, 2049]
    fe = cube.MelSpectrogram(n_fft, M_, sr, hop, win, fmin, fmax)
    out = fe(y.to(dev), n_samples=lens).cpu()
    assert out.shape == (3, 80, fe.n_frames(40000))
    for b, L in enumerate(lens):
        ref = M.hifigan_mel_spectrogram(y[b:b + 1, :L], n_fft, M_, sr, hop, win, fmin, fmax)[0]
        F = ref.shape[1]
        assert F == fe.n_frames(L)
        assert float((out[b, :, :F] - ref).abs().max()) <= MEL_TOL
        assert bool((out[b, :, F:] == float(np.log(1e-5))).all())
    assert float(out[1].min()) == pytest.approx(float(np.log(1e-5)), abs=1e-6)      # the silent stretch sits on the floor


def test_mel_cube_flavour(dev):
    import tts_cube_b200 as cube
    from oracle import mel_ref as M
    y = M.test_signal(1, 30000, seed=4)[0]
    for pre in (False, True):
        ref = M.cube_melspectrogram(y, 22050, 80, 256, use_preemphasis=pre).numpy()
        got = cube.MelVocoder().melspectrogram(y.numpy(), 22050, 80, 256, use_preemphasis=pre, device=dev)
        assert got.shape == ref.shape and got.dtype == np.float32
        assert float(np.abs(got - ref).max()) <= MEL_TOL
    # librosa >= 0.10 pads stft frames with zeros instead of reflecting (the reference does not pin librosa)
    ref0 = M.cube_melspectrogram(y, 22050, 80, 256, pad_mode="constant").numpy()
    got0 = cube.MelVocoder().melspectrogram(y.numpy(), 22050, 80, 256, device=dev, pad_mode="constant")
    assert got0.shape == ref0.shape and float(np.abs(got0 - ref0).max()) <= MEL_TOL
    assert float(np.abs(ref0[:2] - ref[:2]).max()) > 1e-2        # the two conventions really differ at the edges
    # 24 kHz / hop 240 (the Cubegan call), too-short input -> error from the library, not garbage
    fe = cube.MelSpectrogram(1024, 80, 24000, 240, 1024, 0, 12000)
    assert fe(torch.zeros(1, 300, device=dev)).shape == (1, 80, 1)       # shorter than the padding: zero frames, one padded row
    with pytest.raises(cube.CubeVocError):
        cube.MelSpectrogram(1024, 80, 24000, 250, 1024, 0, 12000)(torch.zeros(1, 4000, device=dev))   # hop not a multiple of 4


def test_mel_copy_synthesis_chain(dev, neb_arch):
    """wav -> device mel -> HiFi-GAN (the hifigan/inference.py:26-45 copy-synthesis chain) stays on the GPU and matches
    the same chain through the CPU oracles."""
    import tts_cube_b200 as cube
    from oracle import mel_ref as M
    sd, cfg, _ = neb_arch
    y = M.test_signal(1, 16 * 256, seed=12)
    args = (1024, 80, 22050, 256, 1024, 0, 8000)
    mel = cube.mel_spectrogram(y.to(dev), *args)
    g = _gen(cfg, sd, dev, 1)
    with torch.no_grad():
        wav = g(mel).cpu()
    ref = H.generator_forward(sd, cfg, M.hifigan_mel_spectrogram(y, *args))
    assert wav.shape == ref.shape
    assert float((wav - ref).abs().max()) <= TOL


_BITS_SCRIPT = """
import hashlib, sys, torch
sys.path[:0] = [%r, %r]
from conftest import neb_weights
from oracle import hifigan_ref as H
import tts_cube_b200 as cube
sd, cfg, _ = neb_weights()
g = cube.CubeGenerator(cfg, math=1).to("cuda:0"); g.load_state_dict(sd); g.eval()
mel = H.synthetic_mel(3, 70, seed=5)
with torch.no_grad():
    y = g(mel.to("cuda:0"), n_frames=[70, 9, 41]).cpu().contiguous()
print("SHA", hashlib.sha256(y.numpy().tobytes()).hexdigest(), float(y.abs().max()))
"""


def test_packed_step_epilogue_is_bit_identical():
    """tc_rbstep_kernel<.., PK> only regroups the epilogue's fp32 operations into packed instructions and turns selects into
    branches around the stores: on the trained generator (ragged batch) the waveform must not change by one bit."""
    import os
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    script = _BITS_SCRIPT % (here, os.path.dirname(here))
    out = {}
    for pk in ("0", "1"):
        r = subprocess.run([sys.executable, "-c", script], env=dict(os.environ, CUBE_RB_PK=pk), capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, (r.stdout + r.stderr)[-1500:]
        line = [ln for ln in r.stdout.splitlines() if ln.startswith("SHA")][-1].split()
        out[pk] = line[1]
        assert float(line[2]) > 0.01
    assert out["0"] == out["1"]


# ------------------------------------------------ kernel variants behind env switches ------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("env,select", [
    pytest.param({"CUBE_TC_FUSED": "0"}, "student and tcgen05 and not 862", id="student_unfused_pair"),
    pytest.param({"CUBE_TC_FUSED": "0", "CUBE_TC_CG2": "1"}, "student and tcgen05 and not full_length", id="student_cta_pair"),
    pytest.param({"CUBE_TC_WIN": "0"}, "hifigan and tcgen05 and not full_size and not loudness", id="hifigan_no_window"),
    pytest.param({"CUBE_TC_RBFUSE": "0"}, "hifigan and tcgen05 and not loudness", id="hifigan_unfused_resblock_steps"),
    pytest.param({"CUBE_TC_WIDE": "2"}, "hifigan and tcgen05 and not loudness", id="hifigan_two_subtile_128_stage_forced"),
    pytest.param({"CUBE_RB_PK": "1"}, "hifigan and tcgen05 and not loudness and not full_size and not full_length", id="hifigan_packed_step_epilogue"),
    pytest.param({"CUBE_TC_LEAN": "0"}, "hifigan and tcgen05 and not loudness and not full_size", id="hifigan_generic_issue_loop"),
    pytest.param({"CUBE_TC_LEAN": "0"}, "student and tcgen05 and not full_length and not 862", id="student_generic_issue_loop"),
    pytest.param({"CUBE_TC_FP8": "0"}, "student and tcgen05", id="student_pair_fp16x3"),
    pytest.param({"CUBE_TC_AONCE": "1"}, "student and tcgen05", id="student_pair_a_once"),
    pytest.param({"CUBE_TC_AONCE": "1", "CUBE_TC_FP8": "0"}, "student and tcgen05 and not 862", id="student_pair_a_once_fp16x3"),
    pytest.param({"CUBE_TC_FP8": "0", "CUBE_TC_PAIR": "0"}, "student and tcgen05 and not 862", id="student_single_cta_fp16x3"),
    pytest.param({"CUBE_TC_PAIR": "0"}, "student and tcgen05 and not full_length", id="student_single_cta_fp8"),
])
def test_variants_in_subprocess(env, select):
    """The library reads its kernel-selection switches once per process, so the non-default variants (gate + res/skip
    pair instead of the fused block kernel, CTA-pair MMA, per-tap staging instead of window mode) are exercised by
    re-running the matching parity tests in a child process with the switch set."""
    import os
    import subprocess
    import sys
    e = dict(os.environ, **env)
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-k",
                        f"({select}) and not subprocess"], env=e, capture_output=True, text=True, timeout=600)
    tail = (r.stdout or "")[-1500:] + (r.stderr or "")[-500:]
    assert r.returncode == 0, tail
    assert " passed" in r.stdout, tail
