"""Pin the CPU oracles against outputs of the UNMODIFIED reference (tests/golden/*.npz, produced by
oracle/make_goldens.py in the build container).  CPU only."""
import math

import numpy as np
import pytest
import torch

from conftest import golden_cfg, golden_weights, load_golden
from oracle import clarinet_ref as C, heads_ref as W, hifigan_ref as H


@pytest.mark.parametrize("name", ["hifigan_mini.npz", "hifigan_mini_rb2.npz"])
def test_hifigan_oracle_matches_reference_mini(name):
    d = load_golden(name)
    y = H.generator_forward(golden_weights(d), golden_cfg(d), torch.from_numpy(d["mel"]))
    assert y.shape == d["wav"].shape
    assert float(np.abs(y.numpy() - d["wav"]).max()) <= 1e-6
    assert float(np.abs(d["wav"]).max()) > 0.3  # the fixture is loud: the check is not vacuous


def test_hifigan_oracle_matches_reference_trained(neb):
    sd, cfg = neb
    d = load_golden("hifigan_neb.npz")
    y = H.generator_forward(sd, cfg, torch.from_numpy(d["mel"]))
    assert float(np.abs(y.numpy() - d["wav"]).max()) <= 1e-6
    assert np.array_equal(H.wav_to_int16(y).squeeze(1).numpy(), d["wav_int16"])


def test_hifigan_length_law():
    # SURVEY Appendix B: F=100 -> 24096 (neb rates); F=50 -> 12064 (config_v1)
    assert H.out_len(H.CONFIG_NEB, 100) == 24096
    assert H.out_len(H.CONFIG_V1, 50) == 12064
    assert H.out_len(H.CONFIG_V1, 919) == 220624


def test_hifigan_ragged_equals_alone():
    d = load_golden("hifigan_mini.npz")
    sd, cfg = golden_weights(d), golden_cfg(d)
    mel = torch.from_numpy(d["mel"])
    y = H.generator_forward_ragged(sd, cfg, mel, [13, 7])
    alone = H.generator_forward(sd, cfg, mel[1:2, :, :7])
    assert torch.equal(y[1, :, : alone.shape[2]], alone[0])
    assert float(y[1, :, alone.shape[2]:].abs().max()) == 0.0


def test_heads_oracle_matches_reference():
    d = load_golden("heads.npz")
    x = torch.from_numpy(d["mulaw_x"])
    assert np.array_equal(W.mulaw_encode(x).numpy(), d["mulaw_q"])
    assert np.array_equal(W.mulaw_decode_table().numpy(), d["mulaw_table"])
    # the reference's embedded vector (cube/networks/loss.py:312) and SURVEY Appendix B answers
    assert W.mulaw_encode(torch.tensor([1, 0.9, 0, -0.9, -1.0])).tolist() == [255, 253, 128, 2, 0]
    assert np.array_equal(W.mulaw_encode(torch.from_numpy(d["mulaw_nb_x"])).numpy(), d["mulaw_nb_q"])
    # the edge table reproduces encode bit for bit, including the 765 hardest inputs
    edges = d["mulaw_edges"]
    assert np.all(np.diff(edges) > 0)
    assert np.array_equal(W.mulaw_encode_by_edges(x, edges).numpy(), d["mulaw_q"])
    assert np.array_equal(W.mulaw_encode_by_edges(torch.from_numpy(d["mulaw_nb_x"]), edges).numpy(), d["mulaw_nb_q"])
    # encode(decode(k)) == k for all 256 codes
    assert W.mulaw_encode(W.mulaw_decode_table()).tolist() == list(range(256))
    xr = torch.from_numpy(d["raw_x"])
    assert np.array_equal(W.raw_encode(xr).numpy(), d["raw_q"])
    assert np.array_equal(W.raw_decode(torch.arange(256)).numpy(), d["raw_table"])
    xm = W.mol_sample(torch.from_numpy(d["mol_y"]), torch.from_numpy(d["mol_u_mix"]), torch.from_numpy(d["mol_u_x"]))
    assert np.array_equal(xm.numpy(), d["mol_x"])
    xg = W.gaussian_sample(torch.from_numpy(d["gau_y"]), torch.from_numpy(d["gau_eps"]))
    assert np.array_equal(xg.numpy(), d["gau_x"])


def test_upsamplers_match_reference():
    d = load_golden("upsample2.npz")
    tsd = golden_weights(d)
    mel = torch.from_numpy(d["mel"])
    c = C.upsample_mel(tsd, mel)
    assert c.shape == d["c_up"].shape
    assert float(np.abs(c.numpy() - d["c_up"]).max()) <= 1e-6
    assert np.array_equal(W.upsample_repeat(mel[:, :4], 3).numpy(), d["rep3"])
    assert float(np.abs(W.upsample_linear(mel[:, :4], 3).numpy() - d["lin3"]).max()) <= 1e-6


def test_clarinet_checkpoints_strict_and_regression(clarinet_weights):
    ssd, tsd, trained = clarinet_weights
    C.check_state_dict(ssd, "student")
    C.check_state_dict(tsd, "teacher")
    assert C.student_blocks_of(ssd) == [6, 6, 6, 24] and C.teacher_blocks_of(tsd) == 24
    if not trained:
        pytest.skip("shipped checkpoints not staged: regression snapshot needs them")
    d = load_golden("clarinet_regress.npz")
    x = C.vocode_student(ssd, tsd, torch.from_numpy(d["mel"]), torch.from_numpy(d["z"]))
    assert float(np.abs(x.numpy() - d["wav"]).max()) <= 1e-5


def test_clarinet_self_consistency_probe(clarinet_weights):
    """SURVEY Appendix C.1: the forward code is not in the reference, so the restatement's free
    choices are checked for self-consistency - student samples must be far likelier under the
    teacher with dilation 3^(i mod 6) and sqrt(.5) residual scaling than without."""
    ssd, tsd, trained = clarinet_weights
    if not trained:
        pytest.skip("needs the shipped checkpoints")
    torch.manual_seed(0)
    mel = C.synthetic_mel01(1, 14, seed=21)
    c_up = C.upsample_mel(tsd, mel)
    z = torch.randn(1, 1, c_up.shape[2], generator=torch.Generator().manual_seed(5))
    nll = {}
    for name, base, rs in (("3^n", 3, math.sqrt(0.5)), ("2^n", 2, math.sqrt(0.5)), ("3^n,noscale", 3, 1.0)):
        x = C.student_forward(ssd, z, c_up, dil_base=base, res_scale=rs)
        nll[name] = C.teacher_nll(tsd, x, c_up, dil_base=base, res_scale=rs)
    assert nll["3^n"] < nll["2^n"] - 0.3, nll
    assert nll["3^n"] < nll["3^n,noscale"] - 3.0, nll
    assert nll["3^n"] < -1.0, nll


@pytest.mark.parametrize("head", ["mol", "gm"])
def test_wavernn_oracle_matches_reference(head):
    """Path W4: the restatement replays the reference WaveRNN (seeded weights, seeded draws) sample for sample."""
    from oracle import wavernn_ref as R
    d = load_golden(f"wavernn_{head}.npz")
    sd = golden_weights(d)
    draws = {k[2:]: torch.from_numpy(d[k]) for k in d.files if k.startswith("d:")}
    x = R.wavernn_inference(sd, torch.from_numpy(d["mel"]), torch.from_numpy(d["x_low"]), int(d["upsample"]),
                            int(d["upsample_low"]), head, draws)
    assert x.shape == d["x"].shape
    assert float(np.abs(x.numpy() - d["x"]).max()) <= 2e-6
    assert float(np.abs(d["x"]).max()) > 0.2


def test_wavernn_fold_unfold():
    """Path W5 (cube/networks/vocoder.py:109-131): fold one utterance into chunks with left context and back."""
    from oracle import wavernn_ref as R
    mel = torch.arange(1 * 43 * 80, dtype=torch.float).reshape(1, 43, 80)
    xl = torch.arange(430, dtype=torch.float).reshape(1, 430)
    m, x = R.fold_batch(mel, xl, upsample_low=10, num_batches=20)
    assert m.shape == (20, 3, 80) and x.shape == (20, 31)
    assert float(m[0, 0, 0]) == -5.0 and torch.equal(m[1, 0], mel[0, 1]) and torch.equal(m[3, 1:], mel[0, 6:8])
    assert float(x[0, :10].abs().max()) == 0.0 and torch.equal(x[1, :10], xl[0, 11:21])
    y = torch.arange(20 * 300, dtype=torch.float).reshape(20, 300)
    assert R.unfold_batch(y, 100).shape == (1, 20 * 200)


def test_mel_oracle_matches_reference():
    """oracle/mel_ref.py vs the unmodified hifigan/meldataset.py:mel_spectrogram run in the build container
    (tests/golden/mel_hifigan.npz), with the oracle's OWN Slaney filter bank against the torchaudio one the golden used."""
    from oracle import mel_ref as M
    d = load_golden("mel_hifigan.npz")
    for tag in "ab":
        a = [int(v) for v in d[f"args_{tag}"]]
        basis = M.slaney_mel_basis(a[2], a[0], a[1], a[5], a[6])
        assert float(np.abs(basis - d[f"basis_{tag}"]).max()) <= 2e-7
        # every filter has unit area in Hz (Slaney normalisation) up to the sampling of the triangle on the FFT grid
        area = basis.sum(1) * (a[2] / a[0])
        assert float(np.abs(area[5:-1] - 1.0).max()) < 0.1
        mel = M.hifigan_mel_spectrogram(torch.from_numpy(d[f"y_{tag}"]), *a).numpy()
        assert mel.shape == d[f"mel_{tag}"].shape
        assert float(np.abs(mel - d[f"mel_{tag}"]).max()) <= 5e-5


def test_mel_cube_flavour_properties():
    """MelVocoder restatement: frame law of librosa center=True, log10 floor -5 on silence, pre-emphasis = lfilter([1,-.97])."""
    from oracle import mel_ref as M
    y = M.test_signal(1, 5000, seed=3)[0]
    m = M.cube_melspectrogram(y, 22050, 80, 256)
    assert tuple(m.shape) == (1 + 5000 // 256, 80)
    z = M.cube_melspectrogram(torch.zeros(3000), 22050, 80, 256)
    assert float(z.max()) == -5.0 and float(z.min()) == -5.0
    yp = y.clone()
    yp[1:] = y[1:] - 0.97 * y[:-1]
    assert torch.allclose(M.cube_melspectrogram(y, 22050, 80, 256, use_preemphasis=True), M.cube_melspectrogram(yp, 22050, 80, 256))


def test_teacher_generate_is_consistent_with_teacher_forcing():
    """configs[0] path of the oracle: autoregressive sampling (truncated-window recompute) reproduces itself under
    teacher forcing - x[t+1] = mean_t + 0.8 eps_t exp(log_std_t) with (mean, log_std) from ONE causal pass over the
    finished waveform (cube/networks/loss.py:50-52 for the head)."""
    tsd = C.random_state_dict("teacher", 6, blocks=[3])
    mel = C.synthetic_mel01(1, 1, seed=3)
    c_up = C.upsample_mel(tsd, mel)[:, :, :96]
    eps = torch.randn(1, 96, generator=torch.Generator().manual_seed(2))
    x = C.teacher_generate(tsd, c_up, eps)
    assert x.shape == (1, 1, 96) and float(x[0, 0, 0]) == 0.0 and bool(torch.isfinite(x).all())
    w = {k: v.float() for k, v in C.fold_weight_norm(tsd).items()}
    ml = C.wavenet_forward(w, "", 3, x, c_up)
    want = ml[:, 0, :-1] + 0.8 * eps[:, :-1] * torch.exp(ml[:, 1, :-1])
    assert float((x[:, 0, 1:] - want).abs().max()) <= 1e-5
    assert float(x.abs().max()) > 1e-3


def test_upsamplenet_oracle_matches_reference():
    """cube/networks/modules.py:317-343: the restatement equals the reference-run golden bit for bit on the CPU code path
    the golden was made with.  ATen's conv and tanh round differently under another oneDNN ISA or vector width (both
    follow the host CPU), which moves outputs by up to two ulps of their peak; the tolerance is twice that."""
    from oracle import wavernn_ref as R
    d = load_golden("upsamplenet.npz")
    sd = golden_weights(d)
    y = R.upsamplenet_forward(sd, torch.from_numpy(d["c"]), [int(s) for s in d["scales"]], int(d["kernel_size"]))
    assert y.shape == d["y"].shape == (2, 24, 9 * 16)
    assert float((y - torch.from_numpy(d["y"])).abs().max()) <= 4 * float(np.spacing(np.abs(d["y"]).max()))
