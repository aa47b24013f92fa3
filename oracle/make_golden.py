"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/*.npz by running the
*unmodified imported reference* (oracle/ref_import.py) on CPU; needs a checkout
of the reference at ref_import.REFERENCE_ROOT.
Run:  python -m oracle.make_golden [pins | recon_loss | redecoder]

Weights come from facodec_b200.synth.synth_state_dicts(seed) (host-independent
bits) loaded into the reference modules with load_state_dict, exactly as
reconstruct.py:30-37 loads a checkpoint; waves from synth.synth_waves
(PseudoDataset law).  Nothing but the case table, seeds and the reference's
own outputs goes into the fixtures, so any box can regenerate the inputs and
compare.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

from facodec_b200 import synth  # noqa: E402
from oracle import ref_import  # noqa: E402

GOLDEN_DIR = os.path.join(os.path.dirname(HERE), "tests", "golden")

# name -> (weight seed, wave seed, batch, samples, n_c, full_waves?)
CASES = {
    "b2_t7200": dict(wseed=0, xseed=114514, B=2, T=7200, n_c=2),
    "b1_t96000": dict(wseed=0, xseed=114514, B=1, T=96000, n_c=2),      # BASELINE configs[0]
    "b1_t7000_ragged": dict(wseed=0, xseed=7, B=1, T=7000, n_c=2),      # T % 300 != 0
    "b3_t1500_short": dict(wseed=1, xseed=9, B=3, T=1500, n_c=1),       # reflect-pad short-input branch
    "b2_t6000_fullwaves": dict(wseed=1, xseed=11, B=2, T=6000, n_c=2, full=9000, lens=(9000, 4800)),
}


def run_case(model, c):
    x = synth.synth_waves(c["B"], c["T"], seed=c["xseed"])
    kw = {}
    if "full" in c:
        kw["full_waves"] = synth.synth_waves(c["B"], c["full"], seed=c["xseed"] + 1).squeeze(1)
        kw["wave_lens"] = torch.tensor(c["lens"], dtype=torch.int64)
    with torch.no_grad():
        z = model.encoder(x)
        q = model.quantizer(z, x, n_c=c["n_c"], return_codes=True, **kw)
        y = model.decoder(q[0])
    out = dict(z=z, outs=q[0], z_p=q[1][0], z_c=q[1][1], z_r=q[1][2], commitment=q[2],
               codebook=q[3], timbre=q[4], codes_p=q[5][0], codes_c=q[5][1], codes_r=q[5][2], y=y)
    return {k: v.numpy() for k, v in out.items()}


# Voice-conversion fixtures (reconstruct_redecoder.py:108-122): codes + timbre of a codec fixture -> redecoder.encoder ->
# redecoder.decoder.  name -> (source codec fixture, redecoder weight seed, use_p_code, n_c)
REDEC_CASES = {
    "redec_b2_t7200_vc": dict(src="b2_t7200", wseed=0, use_p=False, n_c=1),      # the call reconstruct_redecoder.py makes
    "redec_b2_t7200_full": dict(src="b2_t7200", wseed=0, use_p=True, n_c=2),      # every embedding table
    "redec_b3_t1500_short": dict(src="b3_t1500_short", wseed=1, use_p=True, n_c=1),   # 5 frames: non-causal short-input pads
}


def run_redec_case(model, c):
    g = dict(np.load(os.path.join(GOLDEN_DIR, c["src"] + ".npz")))
    cp, cc, timbre = (torch.from_numpy(g[k]) for k in ("codes_p", "codes_c", "timbre"))
    with torch.no_grad():
        z = model.encoder(cp, cc, timbre, use_p_code=c["use_p"], n_c=c["n_c"])
        y = model.decoder(z)
    return dict(z=z.numpy(), y=y.numpy())


def vq_margin_report(sd, prefix, latents):
    """top-1 / top-2 gap of every decision of one VectorQuantize (dac/nn/quantize.py:78-94): returns the per-frame margin
    dist[2nd] - dist[1st] of the reference's own distance matrix (fp32).  Used by scripts/vq_margins.py to report how
    far the benchmark batch's decisions are from a tie."""
    import torch.nn.functional as F
    w_in = torch._weight_norm(sd[prefix + ".in_proj.weight_v"], sd[prefix + ".in_proj.weight_g"], 0)
    z_e = F.conv1d(latents, w_in, sd[prefix + ".in_proj.bias"])
    b, d, t = z_e.shape
    enc = F.normalize(z_e.permute(0, 2, 1).reshape(b * t, d))
    cb = F.normalize(sd[prefix + ".codebook.weight"])
    dist = enc.pow(2).sum(1, keepdim=True) - 2 * enc @ cb.t() + cb.pow(2).sum(1, keepdim=True).t()
    top2 = torch.topk(-dist, 2, dim=1).values
    return (top2[:, 0] - top2[:, 1]).reshape(b, t)


def main():
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    model = ref_import.build_reference_model(0)
    loaded = None
    for name, c in CASES.items():
        if loaded != c["wseed"]:
            sds = synth.synth_state_dicts(c["wseed"])
            for k in ("encoder", "quantizer", "decoder"):
                model[k].load_state_dict(sds[k])
            loaded = c["wseed"]
        out = run_case(model, c)
        # z_p/z_c/z_r are large; keep float32 for the small cases only
        if c["B"] * c["T"] > 20000:
            for k in ("z_p", "z_c", "z_r"):
                out.pop(k)
        path = os.path.join(GOLDEN_DIR, name + ".npz")
        np.savez_compressed(path, **out)
        print(name, {k: v.shape for k, v in out.items()}, os.path.getsize(path) // 1024, "KiB")
    main_redecoder()


def main_redecoder():
    model = ref_import.build_reference_redecoder(0)
    loaded = None
    for name, c in REDEC_CASES.items():
        if loaded != c["wseed"]:
            sds = synth.synth_redecoder_state_dicts(c["wseed"])
            for k in ("encoder", "decoder"):
                model[k].load_state_dict(sds[k])
            loaded = c["wseed"]
        out = run_redec_case(model, c)
        path = os.path.join(GOLDEN_DIR, name + ".npz")
        np.savez_compressed(path, **out)
        print(name, {k: v.shape for k, v in out.items()}, os.path.getsize(path) // 1024, "KiB")


RECON_LOSS_CASE = dict(B=2, T=4800, seed=11)


def main_recon_loss():
    """tests/golden/recon_loss.npz: losses.py:65-89 reconstruction_loss of the imported reference for one seeded pair, plus
    its 13 components (mse; l1, l2 per scale) formed with the same torchaudio transforms the reference constructs."""
    import warnings
    warnings.simplefilter("ignore")
    from torchaudio.transforms import MelSpectrogram
    ref_import.import_reference()
    import losses as ref_losses
    c = RECON_LOSS_CASE
    x, G_x = synth.synth_loss_pair(c["B"], c["T"], c["seed"])
    with torch.no_grad():
        loss = ref_losses.reconstruction_loss(x, G_x)
        terms = [torch.nn.functional.mse_loss(x, G_x)]
        for i in range(6, 12):
            s = 2 ** i
            melspec = MelSpectrogram(sample_rate=16000, n_fft=max(s, 512), win_length=s, hop_length=s // 4, n_mels=64)
            S_x, S_G = melspec(x), melspec(G_x)
            terms.append((S_x - S_G).abs().mean())
            terms.append((((torch.log(S_x.abs() + 1e-7) - torch.log(S_G.abs() + 1e-7)) ** 2).mean(dim=-2) ** 0.5).mean())
    path = os.path.join(GOLDEN_DIR, "recon_loss.npz")
    np.savez(path, loss=np.float32(loss), terms=torch.stack(terms).numpy(), B=c["B"], T=c["T"], seed=c["seed"])
    print("recon_loss", float(loss), [float(t) for t in terms])


# ---------------------------------------------------------------------------------------------------------------
# Pins of the restatement: what the imported reference modules return for the inputs of tests/test_oracle.py, stored
# under tests/golden/pin_*, so that those tests compare against the reference on any box.
# ---------------------------------------------------------------------------------------------------------------
SAMPLE_N = 2048


def sample(a, n=SAMPLE_N):
    """A fixed, seeded subset of the (flattened) elements of a large array; arrays of at most n elements stay whole."""
    flat = np.asarray(a).reshape(-1)
    if flat.size <= n:
        return flat
    return flat[np.sort(np.random.RandomState(0).choice(flat.size, n, replace=False))]


def pinned(**arrays):
    """name -> sample(array) plus name + '_shape' -> its full shape."""
    out = {}
    for k, v in arrays.items():
        v = v.detach().numpy() if torch.is_tensor(v) else np.asarray(v)
        out[k] = sample(v)
        out[k + "_shape"] = np.array(v.shape, np.int64)
    return out


def seeded_tensors(names, shapes, seed):
    """Host-independent stand-in weights: N(0, 1 / fan_in) per tensor, drawn in the order given."""
    g = torch.Generator().manual_seed(seed)
    out = {}
    for k, s in zip(names, shapes):
        s = tuple(int(d) for d in s)
        fan_in = int(np.prod(s[1:])) if len(s) > 1 else 1
        out[k] = torch.randn(s, generator=g) / float(np.sqrt(fan_in))
    return out


def shape_strings(tensors):
    return np.array([",".join(str(d) for d in t.shape) for t in tensors])


def parse_shapes(strings):
    return [tuple(int(d) for d in s.split(",") if d) for s in strings]


PIN_CODEC = dict(wseed=1, xseed=21, B=2, T=4500, n_c=2)
PIN_RVQ = dict(num_quantizers=4, codebook_size=10, dim=1024, codebook_dim=8, commitment=0.25, wseed=3, xseed=3, T=17)
PIN_RECON_LOSS = dict(B=3, T=7000, seed=5)
PIN_FAP_FLAGS = dict(use_gr_content_f0=False, use_gr_prosody_phone=False, use_gr_residual_f0=True, use_gr_residual_phone=True,
                     use_gr_timbre_content=True, use_gr_timbre_prosody=False, use_gr_x_timbre=True, norm_f0=True)   # modules/commons.py:311-322 + config.yml


def pin_path(name):
    return os.path.join(GOLDEN_DIR, name)


def main_pins():
    import warnings
    warnings.simplefilter("ignore")
    ref_import.import_reference()
    saved = {}

    # codec: encoder -> quantizer -> decoder of build_model(config.yml) with synthetic weights
    c = PIN_CODEC
    model = ref_import.build_reference_model(0)
    sds = synth.synth_state_dicts(c["wseed"])
    for k in ("encoder", "quantizer", "decoder"):
        model[k].load_state_dict(sds[k])
    x = synth.synth_waves(c["B"], c["T"], seed=c["xseed"])
    with torch.no_grad():
        z = model.encoder(x)
        q = model.quantizer(z, x, n_c=c["n_c"], return_codes=True)
        y = model.decoder(q[0])
    saved["pin_codec.npz"] = dict(pinned(z=z, outs=q[0], timbre=q[4], y=y, z_p=q[1][0], z_c=q[1][1], z_r=q[1][2]),
                                  codes_p=q[5][0].numpy(), codes_c=q[5][1].numpy(), codes_r=q[5][2].numpy(),
                                  commitment=q[2].numpy(), codebook=q[3].numpy())

    # quantize/rvq.py ResidualVQ with seeded weights, and alias_free_torch.Activation1d(Identity)
    from quantize.rvq import ResidualVQ as RefRVQ
    from alias_free_torch import Activation1d as RefAct
    r = PIN_RVQ
    rvq = RefRVQ(num_quantizers=r["num_quantizers"], codebook_size=r["codebook_size"], dim=r["dim"],
                 codebook_dim=r["codebook_dim"], commitment=r["commitment"]).eval()
    names = list(rvq.state_dict())
    shapes = shape_strings(rvq.state_dict().values())
    rvq.load_state_dict(seeded_tensors(names, parse_shapes(shapes), r["wseed"]))
    g = torch.Generator().manual_seed(r["xseed"])
    x = torch.randn(2, r["dim"], r["T"], generator=g)
    xx = torch.randn(2, 5, 50, generator=g)
    with torch.no_grad():
        a = rvq(x)
        act = RefAct(activation=torch.nn.Identity())(xx)
    saved["pin_rvq_altfree.npz"] = dict(pinned(quantized=a[0], act=act), names=np.array(names), shapes=shapes,
                                        indices=a[1].numpy(), all_quantized=sample(a[3].numpy()))

    # modules/redecoder.py encoder + the non-causal, LSTM-free decoder of build_model(stage='redecoder')
    model = ref_import.build_reference_redecoder(0)
    sds = synth.synth_redecoder_state_dicts(2)
    for k in ("encoder", "decoder"):
        model[k].load_state_dict(sds[k])
    g = torch.Generator().manual_seed(5)
    cp = torch.randint(0, 1024, (2, 1, 13), generator=g)
    cc = torch.randint(0, 1024, (2, 2, 13), generator=g)
    timbre = torch.randn(2, 1024, generator=g)
    out = {}
    for use_p, n_c in ((False, 1), (True, 2)):
        with torch.no_grad():
            z = model.encoder(cp, cc, timbre, use_p_code=use_p, n_c=n_c)
            y = model.decoder(z)
        out.update(pinned(**{f"z_{int(use_p)}{n_c}": z, f"y_{int(use_p)}{n_c}": y}))
    saved["pin_redecoder.npz"] = out

    # SnakeBeta inside Activation1d, CNNLSTM heads (modules/quantize.py)
    from modules.quantize import CNNLSTM, SnakeBeta
    g = torch.Generator().manual_seed(9)
    sb = SnakeBeta(6, alpha_logscale=True)
    with torch.no_grad():
        sb.alpha.copy_(torch.randn(6, generator=g) * 0.3)
        sb.beta.copy_(torch.randn(6, generator=g) * 0.3)
    x = torch.randn(2, 6, 40, generator=g)
    with torch.no_grad():
        out = dict(snake=sb(x).numpy(), snake_act=RefAct(activation=sb)(x).numpy())
    for i, (indim, outdim, heads, glob) in enumerate(((64, 10, 2, False), (32, 7, 1, True))):
        m = CNNLSTM(indim, outdim, heads, global_pred=glob).eval()
        m.load_state_dict(synth.synth_cnnlstm(3, indim, outdim, heads), strict=False)
        out[f"keys_{i}"] = np.array(list(m.state_dict()))
        xx = torch.randn(2, indim, 33, generator=g)
        with torch.no_grad():
            for h, t in enumerate(m(xx)):
                out[f"head_{i}_{h}"] = t.numpy()
    saved["pin_heads.npz"] = out

    # meldataset.py preprocess (torchaudio MelSpectrogram): output, window and (sparse) filterbank it used
    import meldataset
    w = synth.synth_waves(1, 5000, seed=3)[0, 0]
    with torch.no_grad():
        ref = meldataset.preprocess(w.numpy())
    fb = meldataset.to_mel.mel_scale.fb
    nz = torch.nonzero(fb.reshape(-1)).reshape(-1)
    saved["pin_dataset_mel.npz"] = dict(mel=ref.numpy(), window=meldataset.to_mel.spectrogram.window.numpy(),
                                        fb_shape=np.array(fb.shape, np.int64), fb_index=nz.numpy().astype(np.int32),
                                        fb_value=fb.reshape(-1)[nz].numpy())

    # losses.py reconstruction_loss
    import losses as ref_losses
    c = PIN_RECON_LOSS
    x, G_x = synth.synth_loss_pair(c["B"], c["T"], c["seed"])
    with torch.no_grad():
        saved["pin_recon_loss.npz"] = dict(loss=ref_losses.reconstruction_loss(x, G_x).numpy(), **c)

    # FApredictors (modules/quantize.py) with build_model's flags, seeded parameters, both forward variants
    from modules.quantize import FApredictors
    out = {}
    for tn in (True, False):
        m = FApredictors(in_dim=32, timbre_norm=tn, use_gr_content_global_f0=True, **PIN_FAP_FLAGS).eval()
        params = dict(m.named_parameters())
        names = list(params)
        shapes = shape_strings(params.values())
        missing, unexpected = m.load_state_dict(seeded_tensors(names, parse_shapes(shapes), 4), strict=False)
        assert not unexpected
        bufs = {k: v for k, v in m.state_dict().items() if k not in params}
        assert sorted(missing) == sorted(bufs)
        g = torch.Generator().manual_seed(6)
        lat = [torch.randn(2, 32, 19, generator=g) for _ in range(3 if tn else 4)]
        with torch.no_grad():
            res = m(lat, torch.randn(2, 32, generator=g)) if tn else m(lat)
        p = f"tn{int(tn)}_"
        out[p + "names"] = np.array(names)
        out[p + "shapes"] = shapes
        out[p + "buffer_names"] = np.array(list(bufs))
        out[p + "buffer_shapes"] = shape_strings(bufs.values())
        out[p + "buffers"] = torch.cat([b.reshape(-1) for b in bufs.values()]).numpy()
        out.update(pinned(**{p + k: v for d in res for k, v in d.items() if v is not None}))
        out[p + "none"] = np.array([k for d in res for k, v in d.items() if v is None])
    saved["pin_fa_predictors.npz"] = out

    for name, arrays in saved.items():
        np.savez_compressed(pin_path(name), **arrays)
        print(name, os.path.getsize(pin_path(name)) // 1024, "KiB")

    # dac/model/base.py DACFile: the bytes its save() writes
    from dac.model.base import DACFile as RefFile
    from facodec_b200 import codefile
    g = torch.Generator().manual_seed(9)
    codes = [torch.randint(0, 1024, (2, n, 37), generator=g) for n in (1, 2, 3)]
    ref = RefFile(codes=codefile.pack_codes(codes), chunk_length=37, original_length=37 * 300,
                  input_db=torch.tensor([-23.5, -17.25]), channels=1, sample_rate=24000, padding=True, dac_version="1.0.0")
    print(ref.save(pin_path("pin_codefile.dac")))


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "pins":
        main_pins()
    elif len(sys.argv) > 1 and sys.argv[1] == "recon_loss":
        main_recon_loss()
    elif len(sys.argv) > 1 and sys.argv[1] == "redecoder":
        main_redecoder()
    else:
        main()
