"""GPU: decoding from codes (fac_dequantize / fac_decode_codes) through FAquantizer.from_codes, Codec.decode_codes,
CodecStream.decode_codes and codefile.decode, against (a) the committed golden fixtures made from the imported reference,
(b) the restatement of ResidualVectorQuantize.from_codes + the forward_v2 tail (tests/from_codes_oracle.py) run live on
the host CPU, (c) the engine's own forward at BASELINE configs[1] size (B = 32 x 4 s).

Bars: z_p / z_c / z_r within 1e-5 max(1, |g|) (they differ from the forward's only by the straight-through rounding
z_e + (z_q - z_e)); outs within 2e-4 (the bar of test_golden_end_to_end); waveform RMS <= 1e-4 (north_star).
"""
import ctypes

import pytest
import torch

from conftest import GOLDEN_CASES, load_golden, state_dicts
from from_codes_oracle import quantizer_from_codes
from oracle import facodec_oracle as O
from test_gpu_parity import RMS_TOL, model_for, rms

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
OUTS_TOL = 2e-4


def _max_rel(a, b):
    a, b = a.detach().double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).abs().max()) / max(1.0, float(b.abs().max()))


def _seeded(B, T, seed):
    g = torch.Generator().manual_seed(seed)
    codes = [torch.randint(0, 1024, (B, n, T), generator=g) for n in (1, 2, 3)]
    return codes, torch.randn(B, 1024, generator=g)


def _dev(codes, timbre):
    return [c.to(DEV) for c in codes], timbre.to(DEV)


@pytest.mark.parametrize("name", list(GOLDEN_CASES))
def test_reference_golden_codes_decode(name, built_lib):
    import facodec_b200 as fb
    c = GOLDEN_CASES[name]
    g = load_golden(name)
    m = model_for(c["wseed"])
    codes, timbre = _dev([torch.from_numpy(g[k]) for k in ("codes_p", "codes_c", "codes_r")], torch.from_numpy(g["timbre"]))
    outs, parts = m.quantizer.from_codes(codes, timbre)
    y = fb.Codec(m).decode_codes(codes, timbre)
    torch.cuda.synchronize()
    if "z_p" in g:
        for k, t in zip(("z_p", "z_c", "z_r"), parts):
            assert _max_rel(t, g[k]) <= 1e-5, (k, _max_rel(t, g[k]))
    assert float((outs.cpu() - torch.from_numpy(g["outs"])).abs().max()) <= OUTS_TOL
    e = rms(y, g["y"])
    print(f"{name}: decode_codes vs reference forward y rms {e:.3e}")
    assert e <= RMS_TOL, e


@pytest.mark.parametrize("n_r", [0, 1, 2, 3])
@pytest.mark.parametrize("n_c", [1, 2])
def test_live_oracle_bitrates(n_c, n_r, built_lib):
    import facodec_b200 as fb
    sds = state_dicts(1)
    m = model_for(1)
    codes, timbre = _seeded(2, 23, seed=100 + 4 * n_c + n_r)
    with torch.no_grad():
        o_ref, parts_ref = quantizer_from_codes(sds["quantizer"], codes, timbre, n_c, n_r)
        y_ref = O.decoder_forward(sds["decoder"], o_ref)
    cd, td = _dev(codes, timbre)
    outs, parts = m.quantizer.from_codes(cd, td, n_c=n_c, n_r=n_r)
    y = fb.Codec(m).decode_codes(cd, td, n_c=n_c, n_r=n_r)
    torch.cuda.synchronize()
    for k, a, b in zip(("z_p", "z_c", "z_r"), parts, parts_ref):
        assert _max_rel(a, b) <= 1e-5, k
    if n_r == 0:
        assert not parts[2].any()
    assert float((outs.cpu() - o_ref).abs().max()) <= OUTS_TOL * max(1.0, float(o_ref.abs().max()))
    assert rms(y, y_ref) <= RMS_TOL


def test_decode_codes_is_decoder_of_from_codes(built_lib):
    import facodec_b200 as fb
    m = model_for(1)
    codes, timbre = _dev(*_seeded(3, 40, seed=5))
    for n_c, n_r in ((2, 3), (1, 0)):
        y = fb.Codec(m).decode_codes(codes, timbre, n_c=n_c, n_r=n_r)
        y2 = m.decoder(m.quantizer.from_codes(codes, timbre, n_c=n_c, n_r=n_r)[0])
        torch.cuda.synchronize()
        assert torch.equal(y, y2), (n_c, n_r)


@pytest.fixture(scope="module")
def config1_forward(built_lib):
    """BASELINE configs[1]: B = 32 utterances x 4 s through the engine's own forward."""
    import facodec_b200 as fb
    from facodec_b200 import synth
    m = model_for(0)
    x = synth.synth_waves(32, 96000, seed=2024).to(DEV)
    y, codes, timbre = fb.Codec(m).forward(x, n_c=2)
    torch.cuda.synchronize()
    return m, y, codes, timbre


def test_round_trip_config1(config1_forward):
    import facodec_b200 as fb
    m, y, codes, timbre = config1_forward
    y2 = fb.Codec(m).decode_codes(codes, timbre)
    torch.cuda.synchronize()
    assert y2.shape == y.shape == (32, 1, 96000)
    e = rms(y2, y)
    print(f"configs[1] round trip: decode_codes(forward codes, timbre) vs forward y: rms {e:.3e}, bit-equal {torch.equal(y, y2)}")
    assert e <= RMS_TOL


def _chunks(total, sizes):
    out, pos, i = [], 0, 0
    while pos < total:
        n = min(sizes[i % len(sizes)], total - pos)
        out.append((pos, n))
        pos += n
        i += 1
    return out


@pytest.mark.parametrize("sizes", [[10, 1, 30, 279], [320], [15, 5]])
def test_stream_decode_codes(config1_forward, sizes):
    """Dequantizing is per frame: every chunk's latents are bit-equal to the offline ones, so the streamed audio is the
    stream decoder's on the offline latents, bit for bit; against the offline decode_codes call the bar is the stream
    decoder's own (test_gpu_stream.py: RMS, bit-equality reported)."""
    import facodec_b200 as fb
    m, _, codes, timbre = config1_forward
    B = 4
    codes = [c[:B] for c in codes]
    timbre = timbre[:B].contiguous()
    T = codes[0].shape[-1]
    y_off = fb.Codec(m).decode_codes(codes, timbre)
    outs_off = m.quantizer.from_codes(codes, timbre)[0]
    with fb.CodecStream(m, B) as s:
        ys, zs = [], []
        for p, n in _chunks(T, sizes):
            chunk = [c[:, :, p:p + n].contiguous() for c in codes]
            zs.append(m.quantizer.from_codes(chunk, timbre)[0])
            ys.append(s.decode_codes(chunk, timbre))
        y_st = torch.cat(ys, dim=2)
    with fb.CodecStream(m, B) as s:
        y_ref = torch.cat([s.decode(outs_off[:, :, p:p + n].contiguous()) for p, n in _chunks(T, sizes)], dim=2)
    torch.cuda.synchronize()
    assert torch.equal(torch.cat(zs, dim=2), outs_off)
    assert torch.equal(y_st, y_ref)
    e = rms(y_st, y_off)
    print(f"stream decode_codes {sizes}: vs offline decode_codes rms {e:.3e}, bit-equal {torch.equal(y_st, y_off)}")
    assert e <= RMS_TOL


def test_dac_file_round_trip(config1_forward, tmp_path):
    import facodec_b200 as fb
    from facodec_b200 import codefile
    m, _, codes, timbre = config1_forward
    codes = [c[:3] for c in codes]
    timbre = timbre[:3].contiguous()
    path = codefile.from_forward(codes, original_length=96000).save(tmp_path / "utt")
    y_file = codefile.decode(m, path, timbre)
    y = fb.Codec(m).decode_codes(codes, timbre)
    torch.cuda.synchronize()
    assert torch.equal(y_file, y)
    y1 = codefile.decode(m, path, timbre, n_r=1)
    assert torch.equal(y1, fb.Codec(m).decode_codes(codes, timbre, n_r=1))


def test_reference_dac_file_decode(built_lib, tmp_path):
    """tests/golden/pin_codefile.dac (written by the reference's DACFile.save) decoded against the live oracle."""
    import os
    from facodec_b200 import codefile
    sds = state_dicts(1)
    m = model_for(1)
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pin_codefile.dac")
    timbre = torch.randn(2, 1024, generator=torch.Generator().manual_seed(3))
    y = codefile.decode(m, path, timbre.to(DEV))
    codes = codefile.unpack_codes(codefile.DACFile.load(path).codes, n_c=2)
    with torch.no_grad():
        y_ref = O.decoder_forward(sds["decoder"], quantizer_from_codes(sds["quantizer"], codes, timbre)[0])
    assert y.shape == y_ref.shape == (2, 1, 37 * 300)
    assert rms(y, y_ref) <= RMS_TOL


def test_per_utterance_conditioning_and_timbre_swap(built_lib):
    import facodec_b200 as fb
    m = model_for(1)
    codes, timbre = _dev(*_seeded(3, 30, seed=9))
    codec = fb.Codec(m)
    y = codec.decode_codes(codes, timbre)
    outs = m.quantizer.from_codes(codes, timbre)[0]
    for b in range(3):
        yb = codec.decode_codes([c[b:b + 1] for c in codes], timbre[b:b + 1])
        ob = m.quantizer.from_codes([c[b:b + 1] for c in codes], timbre[b:b + 1])[0]
        assert float((ob - outs[b:b + 1]).abs().max()) <= 1e-5
        assert rms(yb, y[b:b + 1]) <= 0.1 * RMS_TOL, b
        print(f"utterance {b}: alone vs in batch: outs bit-equal {torch.equal(ob, outs[b:b + 1])}, y bit-equal {torch.equal(yb, y[b:b + 1])}")
    perm = [1, 0, 2]
    ys = codec.decode_codes(codes, timbre[perm].contiguous())
    torch.cuda.synchronize()
    assert torch.equal(ys[2], y[2])
    for b in (0, 1):
        assert float((ys[b] - y[b]).abs().max()) > 1e-3, b
        other = codec.decode_codes([c[b:b + 1] for c in codes], timbre[perm[b]:perm[b] + 1])
        assert rms(other, ys[b:b + 1]) <= 0.1 * RMS_TOL


def test_python_error_paths(built_lib):
    import facodec_b200 as fb
    m = model_for(1)
    codes, timbre = _seeded(2, 12, seed=4)
    cd, td = _dev(codes, timbre)
    with pytest.raises(fb.FacError):
        m.quantizer.from_codes(codes, timbre)                     # CPU tensors
    with pytest.raises(fb.FacError):
        fb.Codec(m).decode_codes(cd, timbre)                      # timbre on another device
    with pytest.raises(fb.FacError):
        fb.Codec(m).decode_codes([cd[0], cd[1], codes[2]], td)
    for v in (1024, -1):
        bad = [c.clone() for c in cd]
        bad[1][1, 0, 7] = v
        with pytest.raises(IndexError):
            fb.Codec(m).decode_codes(bad, td)
        with pytest.raises(IndexError):
            m.quantizer.from_codes(bad, td)


def _raw(L, h, codes, timbre, outs, n_c=2, n_r=3, n_c_rows=2, n_r_rows=3, y=None):
    p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
    s = ctypes.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)
    B, _, T = codes[0].shape
    if y is not None:
        return L.fac_decode_codes(h, p(codes[0]), p(codes[1]), n_c_rows, n_c, p(codes[2]), n_r_rows, n_r, p(timbre), B, T, p(y), s)
    return L.fac_dequantize(h, p(codes[0]), p(codes[1]), n_c_rows, n_c, p(codes[2]), n_r_rows, n_r, p(timbre), B, T, p(outs),
                            None, None, None, s)


def test_c_abi_state_and_arguments(built_lib):
    from facodec_b200 import _lib
    L = _lib.load()
    codes, timbre = _dev(*_seeded(2, 12, seed=6))
    outs = torch.empty(2, 1024, 12, device=DEV)
    y = torch.empty(2, 1, 3600, device=DEV)
    h = ctypes.c_void_p()
    assert L.fac_create(ctypes.byref(h), 0) == 0
    try:
        assert _raw(L, h, codes, timbre, outs) == -2                       # FAC_ERR_STATE: no quantizer weights
        assert _raw(L, h, codes, timbre, None, y=y) == -2
        with pytest.raises(_lib.FacError):
            _lib.check(h, _raw(L, h, codes, timbre, outs), "fac_dequantize")
    finally:
        L.fac_destroy(h)
    m = model_for(1)
    m.quantizer._prep(codes[0])                                             # weights on the device
    L, h = m.quantizer._engine.L, m.quantizer._engine.handle
    for kw in (dict(n_c=0), dict(n_c=2, n_c_rows=1), dict(n_c_rows=3, n_c=1), dict(n_r=3, n_r_rows=2), dict(n_r_rows=4, n_r=1)):
        assert _raw(L, h, codes, timbre, outs, **kw) == -1, kw
    assert _raw(L, h, [codes[0], codes[1], None], timbre, outs, n_r=1) == -1
    assert _raw(L, h, [codes[0], codes[1], None], timbre, outs, n_r=0, n_r_rows=0) == 0


def test_c_abi_out_of_range_codes_give_nan_frames(built_lib):
    """The C-ABI's contract (Python rejects such codes before launch): a code outside [0, 1024) is never used as an
    address and makes every channel of exactly that frame's outs NaN; all other frames are unchanged."""
    from facodec_b200 import _lib
    m = model_for(1)
    codes, timbre = _dev(*_seeded(2, 21, seed=8))
    m.quantizer._prep(codes[0])
    L, h = m.quantizer._engine.L, m.quantizer._engine.handle
    clean = torch.empty(2, 1024, 21, device=DEV)
    _lib.check(h, _raw(L, h, codes, timbre, clean), "fac_dequantize")
    bad = [c.clone() for c in codes]
    bad[1][0, 0, 5] = 1024
    bad[2][1, 2, 9] = -1
    bad[0][1, 0, 20] = 1 << 40
    outs = torch.empty_like(clean)
    _lib.check(h, _raw(L, h, bad, timbre, outs), "fac_dequantize")
    torch.cuda.synchronize()
    nan_frames = {(0, 5), (1, 9), (1, 20)}
    for b in range(2):
        for t in range(21):
            if (b, t) in nan_frames:
                assert torch.isnan(outs[b, :, t]).all(), (b, t)
            else:
                assert torch.equal(outs[b, :, t], clean[b, :, t]), (b, t)
