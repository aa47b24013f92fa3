"""CPU: the oracle restatement against the committed golden fixtures generated from the imported unmodified reference
(oracle/make_golden.py): (a) the codec cases shared with the GPU tests and (b) the pins (tests/golden/pin_*) of every
restated module, made from the reference's outputs for the inputs these tests rebuild from seeds."""
import hashlib
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN_CASES, case_inputs, load_golden, state_dicts
from oracle import facodec_oracle as O
from oracle import make_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# The fixtures were made on one host CPU; on another, oneDNN may pick other kernels (other summation orders), so floats
# are compared with a tight tolerance and near-tied VQ decisions of the long cases may flip.
ATOL = 2e-5


def _close(a, b, name):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, name
    assert np.abs(a - b).max() <= ATOL * max(1.0, np.abs(b).max()), f"{name}: max diff {np.abs(a - b).max()}"


def _close_pinned(got, g, name):
    """got against a pin: its full shape, and the elements make_golden.sample kept."""
    got = got.detach().numpy() if torch.is_tensor(got) else np.asarray(got)
    assert got.shape == tuple(g[name + "_shape"]), name
    _close(make_golden.sample(got), g[name], name)


def _pin(name):
    return dict(np.load(os.path.join(ROOT, "tests", "golden", name), allow_pickle=False))


def test_case_table():
    from oracle import make_golden
    assert make_golden.CASES == GOLDEN_CASES
    for name in GOLDEN_CASES:
        assert os.path.exists(os.path.join(os.path.dirname(__file__), "golden", name + ".npz"))


def test_synth_is_host_independent():
    """Synthetic checkpoints must be the same bits everywhere (golden fixtures depend on it)."""
    from facodec_b200 import synth
    sd = synth.synth_encoder(1)
    h = hashlib.sha256()
    for k in ("block.0.conv.conv.weight_g", "block.1.block.0.block.1.conv.conv.weight_v", "block.6.alpha"):
        h.update(sd[k].numpy().tobytes())
    assert h.hexdigest() == "db65aa08d774396d996e318b9407e70d4417e942368011e08c72c2d351e27314"
    w = synth.synth_waves(1, 1000, seed=3)
    assert abs(float(w.abs().max()) - 1.0) < 1e-7


@pytest.mark.parametrize("name", ["b2_t7200", "b1_t7000_ragged", "b3_t1500_short", "b2_t6000_fullwaves", "b1_t96000"])
def test_oracle_matches_golden(name):
    c = GOLDEN_CASES[name]
    g = load_golden(name)
    sds = state_dicts(c["wseed"])
    x, kw = case_inputs(c)
    with torch.no_grad():
        z = O.encoder_forward(sds["encoder"], x)
        q = O.quantizer_forward(sds["quantizer"], z, x, n_c=c["n_c"], return_codes=True, **kw)
        y = O.decoder_forward(sds["decoder"], q[0])
    _close(z, g["z"], "z")
    _close(q[0], g["outs"], "outs")
    _close(q[4], g["timbre"], "timbre")
    _close(y, g["y"], "y")
    for k, t in zip(("codes_p", "codes_c", "codes_r"), q[5]):
        assert (t.numpy() != g[k]).mean() < 0.02, k
    assert abs(float(q[2]) - float(g["commitment"])) <= 1e-5 * abs(float(g["commitment"]))
    if "z_p" in g:
        for k, t in zip(("z_p", "z_c", "z_r"), q[1]):
            _close(t, g[k], k)


def test_oracle_matches_imported_reference():
    """Pins the restatement to the real thing: the unmodified reference's codec forward (pin_codec.npz) on one more case."""
    c = make_golden.PIN_CODEC
    g = _pin("pin_codec.npz")
    sds = state_dicts(c["wseed"])
    x, _ = case_inputs(c)
    with torch.no_grad():
        z, q, y = O.codec_forward(sds, x, n_c=c["n_c"])
    for k, t in (("z", z), ("outs", q[0]), ("timbre", q[4]), ("y", y), ("z_p", q[1][0]), ("z_c", q[1][1]), ("z_r", q[1][2])):
        _close_pinned(t, g, k)
    for k, t in zip(("codes_p", "codes_c", "codes_r"), q[5]):
        assert np.array_equal(t.numpy(), g[k]), k
    _close(q[2], g["commitment"], "commitment")
    _close(q[3], g["codebook"], "codebook")


def test_fvq_rvq_and_alias_free_match_reference():
    """quantize/rvq.py ResidualVQ with seeded weights and alias_free_torch.Activation1d(Identity) (pin_rvq_altfree.npz)."""
    r = make_golden.PIN_RVQ
    g = _pin("pin_rvq_altfree.npz")
    sd = make_golden.seeded_tensors(g["names"], make_golden.parse_shapes(g["shapes"]), r["wseed"])
    layers = []
    for i in range(r["num_quantizers"]):
        p = f"layers.{i}."
        w = {n: torch._weight_norm(sd[p + n + ".weight_v"], sd[p + n + ".weight_g"], 0) for n in ("in_proj", "out_proj")}
        layers.append(dict(in_w=w["in_proj"], in_b=sd[p + "in_proj.bias"], out_w=w["out_proj"], out_b=sd[p + "out_proj.bias"],
                           codebook=sd[p + "_codebook.weight"]))
    gen = torch.Generator().manual_seed(r["xseed"])
    x = torch.randn(2, r["dim"], r["T"], generator=gen)
    xx = torch.randn(2, 5, 50, generator=gen)
    with torch.no_grad():
        b = O.fvq_residual_vq(layers, x)
    assert np.array_equal(b[1].numpy(), g["indices"])
    _close_pinned(b[0], g, "quantized")
    _close(make_golden.sample(b[3].numpy()), g["all_quantized"], "all_quantized")
    _close_pinned(O.alias_free_act(xx, lambda u: u), g, "act")


def test_reflect_pad_short_branch():
    """encodec.py:96-113: length <= pad => zero-extend, reflect, truncate."""
    x = torch.arange(1, 4, dtype=torch.float32).reshape(1, 1, 3)
    y = O._pad1d_reflect(x, 5, 0)
    assert y.shape[-1] == 8
    assert y.flatten().tolist() == [0.0, 0.0, 0.0, 3.0, 2.0, 1.0, 2.0, 3.0]


# ---------------------------------------------------------------------------------------------------------------
# round 2: voice-conversion path (modules/redecoder.py), predictor heads (modules/quantize.py:29-125), dataset mel
# ---------------------------------------------------------------------------------------------------------------
from conftest import REDEC_CASES  # noqa: E402


def test_redecoder_case_table():
    from oracle import make_golden
    assert make_golden.REDEC_CASES == REDEC_CASES
    for name in REDEC_CASES:
        assert os.path.exists(os.path.join(os.path.dirname(__file__), "golden", name + ".npz"))


@pytest.mark.parametrize("name", list(REDEC_CASES))
def test_redecoder_oracle_matches_golden(name):
    from facodec_b200 import synth
    c = REDEC_CASES[name]
    g = load_golden(name)
    src = load_golden(c["src"])
    sds = synth.synth_redecoder_state_dicts(c["wseed"])
    cp, cc, timbre = (torch.from_numpy(src[k]) for k in ("codes_p", "codes_c", "timbre"))
    with torch.no_grad():
        z = O.redecoder_forward(sds["encoder"], cp, cc, timbre, use_p_code=c["use_p"], n_c=c["n_c"])
        y = O.decoder_forward(sds["decoder"], z, causal=False, lstm=0)
    _close(z, g["z"], "z")
    _close(y, g["y"], "y")


def test_redecoder_oracle_matches_imported_reference():
    """modules/redecoder.py:35-48 + the non-causal, LSTM-free Decoder of build_model(stage='redecoder') (pin_redecoder.npz)."""
    from facodec_b200 import synth
    g = _pin("pin_redecoder.npz")
    sds = synth.synth_redecoder_state_dicts(2)
    gen = torch.Generator().manual_seed(5)
    cp = torch.randint(0, 1024, (2, 1, 13), generator=gen)
    cc = torch.randint(0, 1024, (2, 2, 13), generator=gen)
    timbre = torch.randn(2, 1024, generator=gen)
    for use_p, n_c in ((False, 1), (True, 2)):
        with torch.no_grad():
            z = O.redecoder_forward(sds["encoder"], cp, cc, timbre, use_p_code=use_p, n_c=n_c)
            y = O.decoder_forward(sds["decoder"], z, causal=False, lstm=0)
        _close_pinned(z, g, f"z_{int(use_p)}{n_c}")
        _close_pinned(y, g, f"y_{int(use_p)}{n_c}")


def test_predictor_heads_and_snakebeta_match_imported_reference():
    """SnakeBeta (modules/quantize.py:29-88) inside Activation1d, the heads' ResidualUnit (:90-104) and CNNLSTM (:106-125) of
    the unmodified reference (pin_heads.npz): outputs, and a state_dict surface that synth's checkpoints fill but for the
    registered filter buffers."""
    from facodec_b200 import synth
    g = _pin("pin_heads.npz")
    gen = torch.Generator().manual_seed(9)
    alpha = torch.randn(6, generator=gen) * 0.3
    beta = torch.randn(6, generator=gen) * 0.3
    x = torch.randn(2, 6, 40, generator=gen)
    with torch.no_grad():
        _close(O.snake_beta(x, alpha, beta), g["snake"], "snake")
        _close(O.alias_free_act(x, lambda u: O.snake_beta(u, alpha, beta)), g["snake_act"], "snake_act")
    for i, (indim, outdim, heads, glob) in enumerate(((64, 10, 2, False), (32, 7, 1, True))):
        sd = synth.synth_cnnlstm(3, indim, outdim, heads)
        keys = set(g[f"keys_{i}"].tolist())
        assert set(sd) <= keys and all(k.endswith("filter") for k in keys - set(sd))
        xx = torch.randn(2, indim, 33, generator=gen)
        with torch.no_grad():
            b = O.cnnlstm_forward(sd, xx, heads, global_pred=glob)
        assert len(b) == heads and f"head_{i}_{heads}" not in g
        for h, v in enumerate(b):
            _close(v, g[f"head_{i}_{h}"], f"head_{i}_{h}")


def test_dataset_mel_matches_imported_meldataset():
    """meldataset.py:37-47 preprocess (torchaudio MelSpectrogram with its default sample_rate = 16000) of the unmodified
    reference (pin_dataset_mel.npz, with the window and filterbank it used), against the restatement fed with those and
    with synth's host-independent window and 16 kHz filterbank."""
    from facodec_b200 import synth
    g = _pin("pin_dataset_mel.npz")
    ref = torch.from_numpy(g["mel"])
    win_ref = torch.from_numpy(g["window"])
    fb_ref = torch.zeros(int(np.prod(g["fb_shape"])))
    fb_ref[torch.from_numpy(g["fb_index"]).long()] = torch.from_numpy(g["fb_value"])
    fb_ref = fb_ref.reshape(tuple(g["fb_shape"]))
    w = synth.synth_waves(1, 5000, seed=3)[0, 0]
    with torch.no_grad():
        _close(O.dataset_mel(w, win_ref, fb_ref), ref, "mel")
        fb = synth.melscale_fbanks_htk(sample_rate=16000, f_max=8000.0)
        assert float((fb - fb_ref).abs().max()) <= 1e-5      # fp64-then-round vs torchaudio fp32 evaluation
        got = O.dataset_mel(w, synth.hann_window_periodic(1200), fb)
    assert tuple(ref.shape) == (1, 80, 5000 // 300 + 1)
    assert float((got - ref).abs().max()) <= 2e-5


def test_dac_code_file_matches_imported_dacfile(tmp_path):
    """dac/model/base.py:15-54: files written here are byte-identical to the reference class's (pin_codefile.dac), and the
    reference's file loads here (codes, every metadata field)."""
    from facodec_b200 import codefile
    ref_path = os.path.join(ROOT, "tests", "golden", "pin_codefile.dac")
    g = torch.Generator().manual_seed(9)
    codes = [torch.randint(0, 1024, (2, n, 37), generator=g) for n in (1, 2, 3)]
    mine = codefile.from_forward(codes, original_length=37 * 300, input_db=torch.tensor([-23.5, -17.25]))
    pa = mine.save(tmp_path / "mine")
    assert pa.suffix == ".dac" and open(pa, "rb").read() == open(ref_path, "rb").read()
    for f in (codefile.DACFile.load(pa), codefile.DACFile.load(ref_path)):
        assert torch.equal(f.codes, codefile.pack_codes(codes))
        assert (f.chunk_length, f.original_length, f.channels, f.sample_rate, f.padding, f.dac_version) == (37, 11100, 1, 24000, True, "1.0.0")
        assert np.array_equal(np.asarray(f.input_db), np.array([-23.5, -17.25], np.float32))
        for u, v in zip(codefile.unpack_codes(f.codes, n_c=2), codes):
            assert torch.equal(u, v)


def _loss_signals(B=2, T=4800, seed=11):
    from facodec_b200 import synth
    return synth.synth_loss_pair(B, T, seed)


def test_reconstruction_loss_matches_imported_losses_py():
    """losses.py:65-89 of the unmodified reference on a second seeded pair, odd length (pin_recon_loss.npz)."""
    g = _pin("pin_recon_loss.npz")
    x, G_x = _loss_signals(int(g["B"]), int(g["T"]), int(g["seed"]))
    with torch.no_grad():
        got = O.reconstruction_loss(x, G_x)
    assert got.dim() == 0
    assert abs(float(got) - float(g["loss"])) <= 2e-6 * abs(float(g["loss"]))


def test_reconstruction_loss_golden():
    """tests/golden/recon_loss.npz: loss + 13 terms the imported reference modules gave for the seeded pair (oracle/make_golden.py)."""
    import warnings
    warnings.simplefilter("ignore")
    gold = np.load(os.path.join(ROOT, "tests", "golden", "recon_loss.npz"))
    x, G_x = _loss_signals(int(gold["B"]), int(gold["T"]), int(gold["seed"]))
    with torch.no_grad():
        L, terms = O.reconstruction_loss(x, G_x, return_terms=True)
    assert abs(float(L) - float(gold["loss"])) <= 2e-6 * abs(float(gold["loss"]))
    assert np.allclose(terms.numpy(), gold["terms"], rtol=2e-6, atol=0)


@pytest.mark.parametrize("timbre_norm", [True, False])
def test_fa_predictors_match_imported_reference(timbre_norm):
    """FApredictors (modules/quantize.py:456-619) of the unmodified reference with build_model's flags and seeded parameters,
    both forward variants (pin_fa_predictors.npz): the restatement over the same state_dict, output by output."""
    g = _pin("pin_fa_predictors.npz")
    p = f"tn{int(timbre_norm)}_"
    sd = make_golden.seeded_tensors(g[p + "names"], make_golden.parse_shapes(g[p + "shapes"]), 4)
    flat = torch.from_numpy(g[p + "buffers"])
    for k, s in zip(g[p + "buffer_names"], make_golden.parse_shapes(g[p + "buffer_shapes"])):
        n = int(np.prod(s))
        sd[str(k)], flat = flat[:n].reshape(s), flat[n:]
    assert flat.numel() == 0
    gen = torch.Generator().manual_seed(6)
    lat = [torch.randn(2, 32, 19, generator=gen) for _ in range(3 if timbre_norm else 4)]
    timbre = torch.randn(2, 32, generator=gen) if timbre_norm else None
    with torch.no_grad():
        got = O.fa_predictors_forward(sd, lat, timbre, timbre_norm=timbre_norm, **make_golden.PIN_FAP_FLAGS)
    none = set(g[p + "none"].tolist())
    outs = {k: v for d in got for k, v in d.items()}
    assert {k for k, v in outs.items() if v is None} == none
    assert {p + k for k in outs if k not in none} == {k[:-len("_shape")] for k in g if k.startswith(p) and k.endswith("_shape")}
    for k, v in outs.items():
        if v is not None:
            _close_pinned(v, g, p + k)


def test_slaney_mel_filterbank_against_torchaudio():
    """The restated librosa.filters.mel (Slaney scale + area norm; librosa itself is not installed) against torchaudio's
    independent Slaney implementation, for the geometries train.py:155-163 uses."""
    import torchaudio
    for w, nm in ((32, 5), (64, 10), (256, 40), (512, 80), (2048, 320), (2048, 150)):
        mine = O.librosa_mel_filters(24000, w, nm, 0.0, None)
        ref = torchaudio.functional.melscale_fbanks(w // 2 + 1, 0.0, 12000.0, nm, 24000, norm="slaney", mel_scale="slaney").T
        assert mine.shape == ref.shape == (nm, w // 2 + 1)
        assert float((mine - ref).abs().max()) <= 2e-6 * max(1.0, float(ref.abs().max())), (w, nm)


def test_dac_spectral_losses_restatement_properties():
    """dac/nn/loss.py MultiScaleSTFTLoss / MelSpectrogramLoss restatements (parity unpinned: audiotools absent): zero for
    identical signals, the magnitude path equals a direct torch.stft evaluation, train.py's mel configuration runs."""
    from facodec_b200 import synth
    x, y = synth.synth_loss_pair(2, 3000, seed=3)
    assert float(O.multiscale_stft_loss(x, x)) == 0.0
    assert float(O.mel_spectrogram_loss(x, x)) == 0.0
    st = torch.stft(x[:, 0], 512, hop_length=128, window=torch.hann_window(512), return_complex=True)
    sy = torch.stft(y[:, 0], 512, hop_length=128, window=torch.hann_window(512), return_complex=True)
    direct = (st.abs() - sy.abs()).abs().mean()
    got = O.multiscale_stft_loss(x, y, window_lengths=(512,), log_weight=0.0)
    assert abs(float(got) - float(direct)) <= 1e-6 * float(direct)
    L = O.mel_spectrogram_loss(x, y, 24000, n_mels=[5, 10, 20, 40, 80, 160, 320], window_lengths=[32, 64, 128, 256, 512, 1024, 2048],
                               mel_fmin=[0] * 7, mel_fmax=[None] * 7, pow=1.0, mag_weight=0.0)
    assert torch.isfinite(L) and float(L) > 0
