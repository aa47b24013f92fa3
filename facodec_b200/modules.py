"""Reference-facing call surface:  model.encoder(x) / model.quantizer(z, wave, ...) /
model.decoder(z)  on the Munch returned by build_model (reference modules/commons.py:283-348),
backed by the C-ABI library (include/facodec_b200.h).  PyTorch here is plumbing only: it owns
the device tensors and the CUDA stream; all arithmetic happens in libfacodec_b200.so.

Drop-in contract (SURVEY.md section 8b):
* ``Encoder`` / ``FAquantizer`` / ``Decoder`` are nn.Modules whose ``state_dict()`` /
  ``load_state_dict()`` use the reference's key names (legacy weight-norm ``weight_g`` /
  ``weight_v`` included), so reference checkpoints load unchanged (reconstruct.py:30-34).
* forward signatures and returns are those of dac/model/dac.py:103-104, :164-165 and
  modules/quantize.py:375-454 (forward_v2).  Inference only (eval mode, no autograd): the
  training-time branches (quantizer dropout, random residual mask) are out of scope.
* There is no CPU fallback: CPU tensors or a missing library raise.
"""
import ctypes
import os
from collections import OrderedDict

import torch
from torch import nn

from . import _lib, synth

MOD_ENCODER, MOD_QUANTIZER, MOD_DECODER, MOD_REDECODER, MOD_REDEC_DECODER = 0, 1, 2, 3, 4


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream(device=None):
    """The current CUDA stream OF THE TENSORS' DEVICE (not of whatever device happens to be current)."""
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class Engine:
    """One fac_handle (one CUDA device).  The three modules of a build_model() share it so that
    codec_forward can run encoder -> quantizer -> decoder inside one C call."""

    def __init__(self):
        self.L = _lib.load()
        self.handle = None
        self.device_index = None
        self.loaded_version = {}
        self.modules = {}

    def _ensure(self, device):
        if device.type != "cuda":
            raise _lib.FacError("facodec_b200 runs on CUDA tensors only (no CPU fallback); got " + str(device))
        idx = device.index if device.index is not None else torch.cuda.current_device()
        if self.handle is None:
            h = ctypes.c_void_p()
            rc = self.L.fac_create(ctypes.byref(h), idx)
            if rc < 0:
                raise _lib.FacError(f"fac_create(device={idx}) failed with status {rc}")
            self.handle, self.device_index = h, idx
            # measurement aid: FACODEC_B200_OPTS="name=value,name=value" applies fac_set_option at creation
            for kv in filter(None, os.environ.get("FACODEC_B200_OPTS", "").split(",")):
                name, _, val = kv.partition("=")
                _lib.check(self.handle, self.L.fac_set_option(self.handle, name.strip().encode(), int(val)), "fac_set_option")
        elif idx != self.device_index:
            raise _lib.FacError("engine is bound to cuda:%d, got cuda:%d" % (self.device_index, idx))

    def set_option(self, name, value, device=None):
        """fac_set_option, e.g. ("tensor_cores", 0|1|2)."""
        self._ensure(device or torch.device("cuda", torch.cuda.current_device()))
        _lib.check(self.handle, self.L.fac_set_option(self.handle, name.encode(), int(value)), "fac_set_option")

    def register(self, module_id, module):
        self.modules[module_id] = module

    def sync_weights(self, device):
        """(Re)uploads the weights of every registered module whose parameters changed."""
        self._ensure(device)
        dirty = [m for m, mod in self.modules.items() if self.loaded_version.get(m) != mod._version_tag()]
        if not dirty:
            return
        # fac_finalize repacks everything it holds, so push all registered modules again
        for m, mod in self.modules.items():
            for key, t in mod.state_dict().items():
                t = t.detach().to("cpu", torch.float32).contiguous()
                shape = (ctypes.c_int64 * max(t.dim(), 1))(*t.shape)
                rc = self.L.fac_load_tensor(self.handle, m, key.encode(), _ptr(t), shape, t.dim())
                _lib.check(self.handle, rc, "fac_load_tensor(%s)" % key)
        _lib.check(self.handle, self.L.fac_finalize(self.handle), "fac_finalize")
        for m, mod in self.modules.items():
            self.loaded_version[m] = mod._version_tag()

    def __del__(self):
        try:
            if self.handle is not None:
                self.L.fac_destroy(self.handle)
        except Exception:
            pass


class _RefKeyModule(nn.Module):
    """nn.Module whose parameters are stored flat but exposed under the reference's dotted keys."""

    _module_id = None
    _buffer_keys = ()

    def __init__(self, init_sd, engine=None, module_id=None):
        super().__init__()
        if module_id is not None:
            self._module_id = module_id
        self._keys = list(init_sd.keys())
        self._p = nn.ParameterDict()
        for k, v in init_sd.items():
            if k in self._buffer_keys:
                self.register_buffer(self._safe(k), v.clone(), persistent=True)
            else:
                self._p[self._safe(k)] = nn.Parameter(v.clone(), requires_grad=False)
        self._load_count = 0
        self._engine = engine if engine is not None else Engine()
        self._engine.register(self._module_id, self)

    @staticmethod
    def _safe(k):
        return k.replace(".", "/")

    def _get(self, k):
        s = self._safe(k)
        return self._p[s] if s in self._p else getattr(self, s)

    def _version_tag(self):
        return (self._load_count,) + tuple(self._get(k)._version for k in self._keys)

    def state_dict(self, *args, destination=None, prefix="", keep_vars=False, **kw):
        out = destination if destination is not None else OrderedDict()
        for k in self._keys:
            t = self._get(k)
            out[prefix + k] = t if keep_vars else t.detach()
        return out

    def load_state_dict(self, state_dict, strict=True, assign=False):
        missing = [k for k in self._keys if k not in state_dict]
        unexpected = [k for k in state_dict if k not in self._keys]
        if strict and (missing or unexpected):
            raise RuntimeError("Error(s) in loading state_dict for %s: missing %s unexpected %s"
                               % (type(self).__name__, missing[:5], unexpected[:5]))
        with torch.no_grad():
            for k in self._keys:
                if k in state_dict:
                    dst = self._get(k)
                    src = state_dict[k]
                    if tuple(src.shape) != tuple(dst.shape):
                        raise RuntimeError("size mismatch for %s: %s vs %s" % (k, tuple(src.shape), tuple(dst.shape)))
                    dst.copy_(src)
        self._load_count += 1
        return torch.nn.modules.module._IncompatibleKeys(missing, unexpected)

    def _prep(self, *tensors):
        """Every tensor argument must live on the engine's CUDA device: a CPU tensor or one on another GPU would hand the
        kernels a foreign pointer (illegal address, sticky context error) instead of the promised FacError."""
        if self.training:
            raise NotImplementedError("facodec_b200 implements the eval-mode forward only; call .eval()")
        dev = tensors[0].device
        self._engine.sync_weights(dev)
        for t in tensors[1:]:
            if t is None:
                continue
            if t.device.type != "cuda" or (t.device.index if t.device.index is not None else torch.cuda.current_device()) != self._engine.device_index:
                raise _lib.FacError("all inputs must be on cuda:%d (no CPU fallback, no cross-device copies); got %s"
                                    % (self._engine.device_index, t.device))
        return self._engine.L, self._engine.handle


def _f32c(t):
    return t.detach().to(torch.float32).contiguous()


CODEBOOK_SIZE = 1024


def _codes_args(codes, timbre, n_c=None, n_r=None):
    """Checks a ``[codes_p [B,1,T'], codes_c [B,1|2,T'], codes_r [B,0..3,T'] or None]`` list and ``timbre [B,1024]`` before
    anything reaches the library; ``n_c`` / ``n_r`` (leading codebooks used) default to the rows given.  Returns
    (codes_p, codes_c, codes_r or None, n_c, n_r, timbre) as contiguous int64 / float32 tensors on their own device."""
    if len(codes) != 3:
        raise ValueError("codes must be [codes_p, codes_c, codes_r]")
    cp, cc, cr = codes
    for name, t in (("codes_p", cp), ("codes_c", cc), ("codes_r", cr)):
        if t is None and name == "codes_r":
            continue
        if not torch.is_tensor(t) or t.dtype.is_floating_point or t.dtype.is_complex or t.dtype == torch.bool:
            raise TypeError("%s must be an integer tensor" % name)
        if t.dim() != 3:
            raise ValueError("%s must be [B, rows, T'], got %s" % (name, tuple(t.shape)))
    B, T = cp.shape[0], cp.shape[2]
    rows_r = 0 if cr is None else cr.shape[1]
    if cp.shape[1] != 1 or not (1 <= cc.shape[1] <= 2) or rows_r > 3:
        raise ValueError("codes need 1 prosody, 1-2 content and 0-3 residual rows; got %d, %d, %d"
                         % (cp.shape[1], cc.shape[1], rows_r))
    for name, t in (("codes_c", cc), ("codes_r", cr)):
        if t is not None and (t.shape[0] != B or t.shape[2] != T):
            raise ValueError("%s is %s but codes_p is %s: B and T' must agree" % (name, tuple(t.shape), tuple(cp.shape)))
    if B == 0 or T == 0:
        raise ValueError("empty codes %s" % (tuple(cp.shape),))
    n_c = cc.shape[1] if n_c is None else int(n_c)
    n_r = rows_r if n_r is None else int(n_r)
    if not (1 <= n_c <= cc.shape[1]) or not (0 <= n_r <= rows_r):
        raise ValueError("need 1 <= n_c <= %d content rows and 0 <= n_r <= %d residual rows; got n_c=%d, n_r=%d"
                         % (cc.shape[1], rows_r, n_c, n_r))
    if not torch.is_tensor(timbre) or tuple(timbre.shape) != (B, 1024):
        raise ValueError("timbre must be [%d, 1024], got %s" % (B, tuple(timbre.shape) if torch.is_tensor(timbre) else type(timbre)))
    for t in (cc, cr, timbre):
        if t is not None and t.device != cp.device:
            raise _lib.FacError("codes and timbre must be on one device (no cross-device copies); got %s and %s"
                                % (cp.device, t.device))
    used = [cp, cc[:, :n_c]] + ([cr[:, :n_r]] if n_r else [])
    bad = None
    for t in used:
        b = ((t < 0) | (t >= CODEBOOK_SIZE)).any()
        bad = b if bad is None else bad | b
    if bool(bad):
        raise IndexError("codes out of range: every code must be in [0, %d)" % CODEBOOK_SIZE)
    cp, cc = (t.detach().to(torch.int64).contiguous() for t in (cp, cc))
    cr = None if cr is None else cr.detach().to(torch.int64).contiguous()
    return cp, cc, cr, n_c, n_r, _f32c(timbre)


class Encoder(_RefKeyModule):
    """dac/model/dac.py:69-104 Encoder(d_model=64, strides=[2,5,5,6], d_latent=1024, causal=True, lstm=2)."""
    _module_id = MOD_ENCODER

    def __init__(self, d_model=64, strides=(2, 5, 5, 6), d_latent=1024, causal=True, lstm=2, engine=None):
        if (d_model, tuple(strides), d_latent, bool(causal), lstm) != (64, (2, 5, 5, 6), 1024, True, 2):
            raise NotImplementedError("only the configs/config.yml encoder geometry is built")
        super().__init__(synth.synth_encoder(1), engine)
        self.enc_dim = 1024

    def forward(self, x):
        L, h = self._prep(x)
        x = _f32c(x)
        B, C, T = x.shape
        assert C == 1, "encoder expects [B,1,T]"
        z = torch.empty(B, 1024, L.fac_encode_frames(T), device=x.device, dtype=torch.float32)
        _lib.check(h, L.fac_encode(h, _ptr(x), B, T, _ptr(z), _stream(x.device)), "fac_encode")
        return z


class Decoder(_RefKeyModule):
    """dac/model/dac.py:131-165 Decoder(1024, 1536, [6,5,5,2], causal, lstm): the codec's decoder (causal=True, lstm=2,
    configs/config.yml) or the redecoder model's (causal=False, lstm=0, configs/config_redecoder.yml)."""
    _module_id = MOD_DECODER

    def __init__(self, input_channel=1024, channels=1536, rates=(6, 5, 5, 2), d_out=1, causal=True, lstm=2, engine=None):
        if (input_channel, channels, tuple(rates), d_out) != (1024, 1536, (6, 5, 5, 2), 1) or \
                (bool(causal), int(lstm)) not in ((True, 2), (False, 0)):
            raise NotImplementedError("built: the config.yml decoder (causal, lstm=2) and the config_redecoder.yml one "
                                      "(non-causal, lstm=0)")
        super().__init__(synth.synth_decoder(3, lstm=int(lstm)), engine, module_id=MOD_DECODER if causal else MOD_REDEC_DECODER)
        self.causal = bool(causal)

    def forward(self, z):
        L, h = self._prep(z)
        z = _f32c(z)
        B, C, Tf = z.shape
        assert C == 1024
        y = torch.empty(B, 1, Tf * 300, device=z.device, dtype=torch.float32)
        fn = L.fac_decode if self.causal else L.fac_redecoder_decode
        _lib.check(h, fn(h, _ptr(z), B, Tf, _ptr(y), _stream(z.device)), "fac_decode")
        return y


class Redecoder(_RefKeyModule):
    """modules/redecoder.py:5-48 Redecoder(args) with args.encoder_type == 'wavenet' (wavenet_embed_dim 512, 1 prosody + 2
    content codebooks): forward(p_code, c_code, timbre_vec, use_p_code=True, use_c_code=True, n_c=2) -> [B, 1024, T]."""
    _module_id = MOD_REDECODER

    def __init__(self, args=None, engine=None):
        def g(name, default):
            if args is None:
                return default
            return args[name] if isinstance(args, dict) and name in args else getattr(args, name, default)
        if (g("encoder_type", "wavenet"), g("wavenet_embed_dim", 512), g("n_p_codebooks", 1), g("n_c_codebooks", 2),
                bool(g("decoder_causal", False))) != ("wavenet", 512, 1, 2, False):
            raise NotImplementedError("only the configs/config_redecoder.yml geometry (wavenet, 512, 1 + 2 codebooks, non-causal)")
        super().__init__(synth.synth_redecoder(7), engine)
        self.n_p_codebooks, self.n_c_codebooks, self.codebook_size, self.embed_dim = 1, 2, 1024, 512
        self.encoder_type = "wavenet"

    def forward(self, p_code, c_code, timbre_vec, use_p_code=True, use_c_code=True, n_c=2):
        L, h = self._prep(p_code, c_code, timbre_vec)
        cp = p_code.detach().to(torch.int64).contiguous()
        cc = c_code.detach().to(torch.int64).contiguous()
        tv = _f32c(timbre_vec)
        B, _, T = cp.shape
        if cc.shape[1] < n_c:
            raise IndexError("c_code has %d codebooks, n_c = %d" % (cc.shape[1], n_c))
        z = torch.empty(B, 1024, T, device=cp.device, dtype=torch.float32)
        rc = L.fac_redecode(h, _ptr(cp), _ptr(cc), cc.shape[1], _ptr(tv), B, T, int(bool(use_p_code)), int(bool(use_c_code)),
                            int(n_c), _ptr(z), _stream(cp.device))
        _lib.check(h, rc, "fac_redecode")
        return z


class FAquantizer(_RefKeyModule):
    """modules/quantize.py:156-454 FAquantizer(..., separate_prosody_encoder=True, timbre_norm=True);
    forward == forward_v2 (:375-454)."""
    _module_id = MOD_QUANTIZER
    _buffer_keys = ("to_mel.spectrogram.window", "to_mel.mel_scale.fb")

    def __init__(self, in_dim=1024, n_p_codebooks=1, n_c_codebooks=2, n_t_codebooks=2, n_r_codebooks=3,
                 codebook_size=1024, codebook_dim=8, quantizer_dropout=0.5, causal=True,
                 separate_prosody_encoder=True, timbre_norm=True, engine=None):
        cfg = (in_dim, n_p_codebooks, n_c_codebooks, n_r_codebooks, codebook_size, codebook_dim, bool(causal),
               bool(separate_prosody_encoder), bool(timbre_norm))
        if cfg != (1024, 1, 2, 3, 1024, 8, True, True, True):
            raise NotImplementedError("only the configs/config.yml quantizer geometry is built")
        super().__init__(synth.synth_quantizer(2), engine)
        self.hop_length = 300
        self.is_timbre_norm = True

    def forward(self, x, wave_segments, n_c=1, n_t=2, full_waves=None, wave_lens=None, return_codes=False):
        L, h = self._prep(x, wave_segments, full_waves)
        if not (1 <= int(n_c) <= 2):
            raise ValueError("n_c must be 1 or 2 (content codebooks)")
        x = _f32c(x)
        wave = _f32c(wave_segments)
        B, C, Tz = x.shape
        T = wave.shape[-1]
        Tq = min(T // 300, Tz)
        dev = x.device
        outs = torch.empty(B, 1024, Tq, device=dev)
        zp, zc, zr = (torch.empty(B, 1024, Tq, device=dev) for _ in range(3))
        losses = torch.empty(2, device=dev)
        timbre = torch.empty(B, 1024, device=dev)
        cp = torch.empty(B, 1, Tq, device=dev, dtype=torch.int64)
        cc = torch.empty(B, n_c, Tq, device=dev, dtype=torch.int64)
        cr = torch.empty(B, 3, Tq, device=dev, dtype=torch.int64)
        fw = wl = None
        tfull = 0
        if full_waves is not None:
            fw = _f32c(full_waves)
            wl = wave_lens.detach().to(dev, torch.int64).contiguous()
            tfull = fw.shape[-1]
        rc = L.fac_quantize(h, _ptr(x), _ptr(wave), B, T, Tz, int(n_c), _ptr(fw), tfull, _ptr(wl), _ptr(outs), _ptr(zp),
                            _ptr(zc), _ptr(zr), _ptr(losses), _ptr(timbre), _ptr(cp), _ptr(cc), _ptr(cr), _stream(dev))
        _lib.check(h, rc, "fac_quantize")
        quantized = [zp, zc, zr]
        if return_codes:
            return outs, quantized, losses[0], losses[1], timbre, [cp, cc, cr]
        return outs, quantized, losses[0], losses[1], timbre

    forward_v2 = forward

    def from_codes(self, codes, timbre, n_c=None, n_r=None):
        """Codes back to the decoder's input: ResidualVectorQuantize.from_codes (dac/nn/quantize.py:200-220) of the
        prosody, content and residual quantizers, then the forward_v2 tail (modules/quantize.py:435-449),
        LayerNorm(z_p + z_c + z_r) * gamma + beta with (gamma, beta) = timbre_linear(timbre).

        ``codes`` is the ``[codes_p, codes_c, codes_r]`` list ``forward(..., return_codes=True)`` returns and ``timbre``
        [B, 1024] its timbre (or another utterance's: timbre conversion).  ``n_c`` / ``n_r`` use only the leading content /
        residual codebooks (a lower bitrate; ``n_r = 0`` leaves z_r = 0); they default to the rows given.  Returns
        ``(outs, [z_p, z_c, z_r])``, each [B, 1024, T'].  Not named ``decode``: the reference's ``decode`` takes another
        code layout and cannot run under configs/config.yml."""
        return self._dequantize(codes, timbre, n_c, n_r, parts=True)

    def _dequantize(self, codes, timbre, n_c, n_r, parts):
        cp, cc, cr, n_c, n_r, tv = _codes_args(codes, timbre, n_c, n_r)
        L, h = self._prep(cp, cc, cr, tv)
        B, _, T = cp.shape
        dev = cp.device
        outs = torch.empty(B, 1024, T, device=dev)
        zp, zc, zr = (torch.empty(B, 1024, T, device=dev) for _ in range(3)) if parts else (None, None, None)
        rc = L.fac_dequantize(h, _ptr(cp), _ptr(cc), cc.shape[1], n_c, _ptr(cr), 0 if cr is None else cr.shape[1], n_r,
                              _ptr(tv), B, T, _ptr(outs), _ptr(zp), _ptr(zc), _ptr(zr), _stream(dev))
        _lib.check(h, rc, "fac_dequantize")
        return outs, [zp, zc, zr]


class Munch(dict):
    """Attribute dict (the reference returns munch.Munch from build_model)."""
    __getattr__ = dict.__getitem__
    __setattr__ = dict.__setitem__


class Codec:
    """reconstruct.py:56-61 as one C call: encoder -> quantizer(n_c) -> decoder, latents resident."""

    def __init__(self, model):
        self.model = model
        self.engine = model.encoder._engine

    def forward(self, x, n_c=2):
        """x [B,1,T] on the GPU -> (y [B,1,T'], [codes_p, codes_c, codes_r], timbre)."""
        e = self.engine
        for m in (self.model.encoder, self.model.quantizer, self.model.decoder):
            if m.training:
                raise NotImplementedError("eval mode only")
        e.sync_weights(x.device)
        x = _f32c(x)
        B, _, T = x.shape
        Tq = min(T // 300, e.L.fac_encode_frames(T))
        dev = x.device
        y = torch.empty(B, 1, Tq * 300, device=dev)
        cp = torch.empty(B, 1, Tq, device=dev, dtype=torch.int64)
        cc = torch.empty(B, n_c, Tq, device=dev, dtype=torch.int64)
        cr = torch.empty(B, 3, Tq, device=dev, dtype=torch.int64)
        timbre = torch.empty(B, 1024, device=dev)
        rc = e.L.fac_codec_forward(e.handle, _ptr(x), B, T, n_c, _ptr(y), _ptr(cp), _ptr(cc), _ptr(cr), _ptr(timbre), _stream(dev))
        _lib.check(e.handle, rc, "fac_codec_forward")
        return y, [cp, cc, cr], timbre

    def decode_codes(self, codes, timbre, n_c=None, n_r=None):
        """Codes + timbre -> audio in one C call: model.decoder(model.quantizer.from_codes(codes, timbre, n_c, n_r)[0])
        with the latents kept on the device.  codes = [codes_p, codes_c, codes_r] as ``forward`` returns them,
        timbre [B, 1024] -> y [B, 1, 300 T']."""
        if self.model.decoder.training:
            raise NotImplementedError("eval mode only")
        cp, cc, cr, n_c, n_r, tv = _codes_args(codes, timbre, n_c, n_r)
        L, h = self.model.quantizer._prep(cp, cc, cr, tv)
        B, _, T = cp.shape
        y = torch.empty(B, 1, T * 300, device=cp.device)
        rc = L.fac_decode_codes(h, _ptr(cp), _ptr(cc), cc.shape[1], n_c, _ptr(cr), 0 if cr is None else cr.shape[1], n_r,
                                _ptr(tv), B, T, _ptr(y), _stream(cp.device))
        _lib.check(h, rc, "fac_decode_codes")
        return y

    def forward_host(self, x_host, n_c=2, out=None):
        """End-to-end with HOST tensors (pinned recommended): H2D, forward, D2H inside the call.
        x_host [B,1,T] float32 CPU -> (y_host [B,1,T'], [codes_p, codes_c, codes_r]) CPU tensors."""
        e = self.engine
        dev = torch.device("cuda", torch.cuda.current_device() if e.device_index is None else e.device_index)
        e.sync_weights(dev)
        assert x_host.device.type == "cpu" and x_host.dtype == torch.float32 and x_host.is_contiguous()
        B, _, T = x_host.shape
        Tq = min(T // 300, e.L.fac_encode_frames(T))
        if out is None:
            pin = torch.cuda.is_available()
            out = (torch.empty(B, 1, Tq * 300, pin_memory=pin),
                   torch.empty(B, 1, Tq, dtype=torch.int64, pin_memory=pin),
                   torch.empty(B, n_c, Tq, dtype=torch.int64, pin_memory=pin),
                   torch.empty(B, 3, Tq, dtype=torch.int64, pin_memory=pin))
        y, cp, cc, cr = out
        with torch.cuda.device(dev):
            rc = e.L.fac_codec_forward_host(e.handle, _ptr(x_host), B, T, n_c, _ptr(y), _ptr(cp), _ptr(cc), _ptr(cr), _stream(dev))
        _lib.check(e.handle, rc, "fac_codec_forward_host")
        return y, [cp, cc, cr]

    def forward_graphed(self, x, n_c=2):
        """The same call replayed from a CUDA graph (one graph per (B, T, n_c, device), captured on first use after one
        eager call has sized the workspace): for latency-bound shapes (B = 1: 115 launches, two of them cooperative LSTM
        layers, plus the forked quantizer front) the launches leave the host in one go.  Returns the graph's OWN output
        tensors: they are overwritten by the next replay of the same shape -- clone what must survive."""
        x = _f32c(x)
        key = (tuple(x.shape), int(n_c), x.device.index)
        if not hasattr(self, "_graphs"):
            self._graphs = {}
        ent = self._graphs.get(key)
        if ent is None:
            self.forward(x, n_c)                                  # sizes the workspace, creates the side stream (not capturable)
            torch.cuda.synchronize(x.device)
            sx = x.clone()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                out = self.forward(sx, n_c)
            ent = self._graphs[key] = (g, sx, out, self.launch_count())
        g, sx, out, _ = ent
        sx.copy_(x)
        g.replay()
        return out

    def launch_count(self):
        return self.engine.L.fac_last_launch_count(self.engine.handle)


class CodecStream:
    """Chunked (streaming) use of the causal encoder / decoder of a build_model() Munch (README.md:105-107): feeding an
    utterance in pieces gives the results of ONE offline model.encoder(x) / model.decoder(z) call (dac/model/dac.py:103-104,
    :164-165).  The conv left context and the SLSTM (h, c) states live on the device between calls (fac_stream_*)."""

    def __init__(self, model, batch, device=None):
        self.model = model
        self.engine = model.encoder._engine
        dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.engine.sync_weights(dev)
        self.device = torch.device("cuda", self.engine.device_index)
        self.batch = int(batch)
        sid = self.engine.L.fac_stream_begin(self.engine.handle, self.batch)
        _lib.check(self.engine.handle, sid, "fac_stream_begin")
        self.sid = sid

    def _check(self, t):
        if t.device.type != "cuda" or (t.device.index if t.device.index is not None else torch.cuda.current_device()) != self.engine.device_index:
            raise _lib.FacError("stream inputs must be on cuda:%d (no CPU fallback); got %s" % (self.engine.device_index, t.device))
        if self.sid is None:
            raise _lib.FacError("stream is closed")

    def encode(self, x):
        """x chunk [B,1,T] (T a multiple of 300; first chunk >= 3000 samples) -> z chunk [B,1024,T/300]."""
        self._check(x)
        x = _f32c(x)
        B, C, T = x.shape
        assert C == 1 and B == self.batch
        z = torch.empty(B, 1024, max(T // 300, 0), device=x.device, dtype=torch.float32)
        e = self.engine
        _lib.check(e.handle, e.L.fac_stream_encode(e.handle, self.sid, _ptr(x), T, _ptr(z), _stream(x.device)), "fac_stream_encode")
        return z

    def decode(self, z):
        """z chunk [B,1024,Fc] (first chunk >= 10 frames) -> y chunk [B,1,300*Fc]."""
        self._check(z)
        z = _f32c(z)
        B, C, Fc = z.shape
        assert C == 1024 and B == self.batch
        y = torch.empty(B, 1, Fc * 300, device=z.device, dtype=torch.float32)
        e = self.engine
        _lib.check(e.handle, e.L.fac_stream_decode(e.handle, self.sid, _ptr(z), Fc, _ptr(y), _stream(z.device)), "fac_stream_decode")
        return y

    def decode_codes(self, codes_chunk, timbre):
        """A chunk of codes ([codes_p, codes_c, codes_r], Fc frames; the first chunk >= 10 frames) and the utterance's
        timbre [B, 1024] -> y chunk [B, 1, 300 Fc].  Dequantizing is per frame, so the chunks together give exactly what
        one offline ``Codec.decode_codes`` call gives."""
        self._check(codes_chunk[0])
        z, _ = self.model.quantizer._dequantize(codes_chunk, timbre, None, None, parts=False)
        return self.decode(z)

    def close(self):
        if self.sid is not None and self.engine.handle is not None:
            self.engine.L.fac_stream_end(self.engine.handle, self.sid)
        self.sid = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class VoiceConverter:
    """reconstruct_redecoder.py:118-121 as one C call: z = model.encoder(codes[0], codes[1], timbre, use_p_code, n_c);
    wave = model.decoder(z) on a build_model(stage='redecoder') Munch, latents resident."""

    def __init__(self, model):
        self.model = model
        self.engine = model.encoder._engine

    def convert(self, codes, timbre, use_p_code=False, use_c_code=True, n_c=1):
        e = self.engine
        dev = codes[0].device
        e.sync_weights(dev)
        cp = codes[0].detach().to(torch.int64).contiguous()
        cc = codes[1].detach().to(torch.int64).contiguous()
        tv = _f32c(timbre)
        B, _, T = cp.shape
        y = torch.empty(B, 1, T * 300, device=dev)
        rc = e.L.fac_voice_convert(e.handle, _ptr(cp), _ptr(cc), cc.shape[1], _ptr(tv), B, T, int(bool(use_p_code)),
                                   int(bool(use_c_code)), int(n_c), _ptr(y), _stream(dev))
        _lib.check(e.handle, rc, "fac_voice_convert")
        return y


class _HeadLinear(nn.Module):
    """A plain nn.Linear(indim, outdim) run through the head machinery (kind "linear" of fac_head_finalize)."""

    def __init__(self, indim, outdim, seed=0, engine=None):
        super().__init__()
        self.indim, self.outdim = int(indim), int(outdim)
        g = synth._Gen(900 + seed)
        b = 1.0 / (indim ** 0.5)
        self.weight = nn.Parameter(g.uniform((outdim, indim), b), requires_grad=False)
        self.bias = nn.Parameter(g.uniform((outdim,), b), requires_grad=False)
        self._engine = engine if engine is not None else Engine()
        self._head_id = None
        self._tag = None

    def _sync(self, device):
        e = self._engine
        e._ensure(device)
        tag = (self.weight._version, self.bias._version)
        if self._tag == tag:
            return
        L, h = e.L, e.handle
        if self._head_id is None:
            self._head_id = _lib.check(h, L.fac_head_begin(h), "fac_head_begin")
        for k, p in (("linear.weight", self.weight), ("linear.bias", self.bias)):
            t = p.detach().to("cpu", torch.float32).contiguous()
            shape = (ctypes.c_int64 * t.dim())(*t.shape)
            _lib.check(h, L.fac_head_tensor(h, self._head_id, k.encode(), _ptr(t), shape, t.dim()), "fac_head_tensor(%s)" % k)
        _lib.check(h, L.fac_head_finalize(h, self._head_id, self.indim, self.outdim, 1, 2), "fac_head_finalize")
        self._tag = tag

    def forward(self, x):
        self._sync(x.device)
        e = self._engine
        x = _f32c(x)
        rows = x.numel() // self.indim
        out = torch.empty(tuple(x.shape[:-1]) + (self.outdim,), device=x.device)
        arr = (ctypes.c_void_p * 1)(out.data_ptr())
        _lib.check(e.handle, e.L.fac_head_forward(e.handle, self._head_id, _ptr(x), rows, 1, arr, _stream(x.device)), "fac_head_forward")
        return out


class FApredictors(nn.Module):
    """modules/quantize.py:456-619 FApredictors, forward only (training-side in the reference; the GradientReversal layers are
    identities in the forward pass): the f0 / phone / timbre predictors and their reversal counterparts over the quantizer's
    latents -- CNNLSTM heads (fac_head_*), one nn.Linear (timbre_predictor under timbre_norm) and the latent sums
    (fac_add3).  Same constructor flags, same state_dict keys (``rev_*_predictor.1.*`` for the heads inside nn.Sequential),
    same ``(preds, rev_preds)`` dicts; ``forward`` is ``forward_v2(quantized, timbre)`` when ``timbre_norm`` (config.yml),
    else the 4-latent ``forward(quantized)``."""

    def __init__(self, in_dim=1024, use_gr_content_f0=False, use_gr_prosody_phone=False, use_gr_residual_f0=False,
                 use_gr_residual_phone=False, use_gr_timbre_content=True, use_gr_timbre_prosody=True, use_gr_x_timbre=False,
                 norm_f0=True, timbre_norm=False, use_gr_content_global_f0=False, n_speakers=20000, engine=None):
        super().__init__()
        eng = engine if engine is not None else Engine()
        self._engine = eng
        self.in_dim = int(in_dim)
        self.flags = dict(use_gr_content_f0=use_gr_content_f0, use_gr_prosody_phone=use_gr_prosody_phone,
                          use_gr_residual_f0=use_gr_residual_f0, use_gr_residual_phone=use_gr_residual_phone,
                          use_gr_timbre_content=use_gr_timbre_content, use_gr_timbre_prosody=use_gr_timbre_prosody,
                          use_gr_x_timbre=use_gr_x_timbre, norm_f0=norm_f0, timbre_norm=timbre_norm)
        parts = OrderedDict()
        parts["f0_predictor"] = CNNLSTM(in_dim, 1, 2, seed=1, engine=eng)
        parts["phone_predictor"] = CNNLSTM(in_dim, 1024, 1, seed=2, engine=eng)
        parts["timbre_predictor"] = (_HeadLinear(in_dim, n_speakers, seed=3, engine=eng) if timbre_norm
                                     else CNNLSTM(in_dim, n_speakers, 1, global_pred=True, seed=3, engine=eng))
        parts["rev_f0_predictor.1"] = CNNLSTM(in_dim, 1, 2, seed=4, engine=eng)
        parts["rev_content_predictor.1"] = CNNLSTM(in_dim, 1024, 1, seed=5, engine=eng)
        parts["rev_timbre_predictor.1"] = CNNLSTM(in_dim, n_speakers, 1, global_pred=True, seed=6, engine=eng)
        if timbre_norm:
            parts["global_f0_predictor"] = _HeadLinear(in_dim, 1, seed=7, engine=eng)           # built, unused by forward (as in the reference)
        if use_gr_content_global_f0:
            parts["rev_global_f0_predictor.1"] = CNNLSTM(in_dim, 1, 1, global_pred=True, seed=8, engine=eng)
        self._parts = parts
        self._mods = nn.ModuleList(list(parts.values()))
        if timbre_norm:
            self.forward = self.forward_v2

    # ---- reference state_dict surface ----
    def state_dict(self, *a, prefix="", **kw):
        out = OrderedDict()
        for name, m in self._parts.items():
            if isinstance(m, _HeadLinear):
                out[prefix + name + ".weight"] = m.weight.detach()
                out[prefix + name + ".bias"] = m.bias.detach()
            else:
                out.update(m.state_dict(prefix=prefix + name + "."))
        return out

    def load_state_dict(self, sd, strict=True, assign=False):
        for name, m in self._parts.items():
            sub = {k[len(name) + 1:]: v for k, v in sd.items() if k.startswith(name + ".")}
            if isinstance(m, _HeadLinear):
                if strict and ("weight" not in sub or "bias" not in sub):
                    raise RuntimeError("missing keys: %s.weight / bias" % name)
                with torch.no_grad():
                    if "weight" in sub:
                        m.weight.copy_(sub["weight"])
                    if "bias" in sub:
                        m.bias.copy_(sub["bias"])
            else:
                m.load_state_dict(sub, strict=strict)

    def _sum(self, terms):
        """Left-to-right sum of 1-3 latents, as the reference accumulates them into zeros_like()."""
        if len(terms) == 1:
            return terms[0]
        e = self._engine
        a = [_f32c(t) for t in terms]
        out = torch.empty_like(a[0])
        _lib.check(e.handle, e.L.fac_add3(e.handle, _ptr(a[0]), _ptr(a[1]), _ptr(a[2]) if len(a) > 2 else None, a[0].numel(), _ptr(out),
                                          _stream(out.device)), "fac_add3")
        return out

    def _check(self, t):
        if self.training:
            raise NotImplementedError("eval mode only")
        if t.device.type != "cuda":
            raise _lib.FacError("FApredictors runs on CUDA tensors only (no CPU fallback)")
        self._engine._ensure(t.device)

    def forward_v2(self, quantized, timbre):
        """modules/quantize.py:564-619: quantized = [prosody, content, residual] latents [B, in_dim, T], timbre [B, in_dim]."""
        f = self.flags
        p, c, r = quantized[0], quantized[1], quantized[2]
        self._check(p)
        P = self._parts
        content_pred = P["phone_predictor"](c)[0]
        spk_pred = P["timbre_predictor"](timbre)
        f0_pred, uv_pred = P["f0_predictor"](p)
        pro_terms = ([c] if f["use_gr_content_f0"] else []) + ([r] if f["use_gr_residual_f0"] else [])
        con_terms = ([p] if f["use_gr_prosody_phone"] else []) + ([r] if f["use_gr_residual_phone"] else [])
        zeros = None
        if not pro_terms or not con_terms:
            zeros = torch.zeros_like(p)
        rev_f0_pred, rev_uv_pred = P["rev_f0_predictor.1"](self._sum(pro_terms) if pro_terms else zeros)
        rev_content_pred = P["rev_content_predictor.1"](self._sum(con_terms) if con_terms else zeros)[0]
        x_spk_pred = P["rev_timbre_predictor.1"](self._sum([p, c, r]))[0] if f["use_gr_x_timbre"] else None
        preds = {"f0": f0_pred, "uv": uv_pred, "content": content_pred, "timbre": spk_pred}
        rev_preds = {"rev_f0": rev_f0_pred, "rev_uv": rev_uv_pred, "rev_content": rev_content_pred, "x_timbre": x_spk_pred}
        return preds, rev_preds

    def forward(self, quantized):
        """modules/quantize.py:507-563 (timbre_norm = False): quantized = [prosody, content, timbre, residual] latents."""
        f = self.flags
        p, c, t, r = quantized[0], quantized[1], quantized[2], quantized[3]
        self._check(p)
        P = self._parts
        content_pred = P["phone_predictor"](c)[0]
        if f["norm_f0"]:
            spk_pred = P["timbre_predictor"](t)[0]
            f0_pred, uv_pred = P["f0_predictor"](p)
        else:
            spk_pred = P["timbre_predictor"](self._sum([t, p]))[0]
            f0_pred, uv_pred = P["f0_predictor"](self._sum([p, t]))
        pro_terms = ([c] if f["use_gr_content_f0"] else []) + ([t] if f["use_gr_timbre_prosody"] else []) + ([r] if f["use_gr_residual_f0"] else [])
        con_terms = ([p] if f["use_gr_prosody_phone"] else []) + ([t] if f["use_gr_timbre_content"] else []) + ([r] if f["use_gr_residual_phone"] else [])
        zeros = torch.zeros_like(p) if (not pro_terms or not con_terms) else None
        rev_f0_pred, rev_uv_pred = P["rev_f0_predictor.1"](self._sum(pro_terms) if pro_terms else zeros)
        rev_content_pred = P["rev_content_predictor.1"](self._sum(con_terms) if con_terms else zeros)[0]
        x_terms = [p, c, r] if f["norm_f0"] else [c, r]
        x_spk_pred = P["rev_timbre_predictor.1"](self._sum(x_terms))[0] if f["use_gr_x_timbre"] else None
        preds = {"f0": f0_pred, "uv": uv_pred, "content": content_pred, "timbre": spk_pred}
        rev_preds = {"rev_f0": rev_f0_pred, "rev_uv": rev_uv_pred, "rev_content": rev_content_pred, "x_timbre": x_spk_pred}
        return preds, rev_preds


def build_model(args=None, stage="codec", with_predictors=False):
    """Mirror of modules/commons.py:283-348 build_model(args, stage='codec') for the hot-path
    modules: returns Munch(encoder, quantizer, decoder) (the discriminator is training-only and out of scope).
    ``with_predictors=True`` adds ``fa_predictors`` (forward only) with the flags of modules/commons.py:311-322; it is
    opt-in because its two 20 000-way speaker heads are 160 MB of weights no inference call touches.
    ``args`` may be the reference's recursive_munch(config['model_params']) or None.
    stage='redecoder' returns the voice-conversion model Munch(encoder=Redecoder, decoder=Decoder(non-causal, no LSTM))."""
    if stage == "redecoder":
        # modules/commons.py:385-412: Munch(encoder=Redecoder(args), decoder=Decoder(causal=args.decoder_causal, lstm=args.decoder_lstm))
        eng = Engine()

        def ga(name, default):
            if args is None:
                return default
            return args[name] if isinstance(args, dict) and name in args else getattr(args, name, default)
        return Munch(encoder=Redecoder(args, engine=eng),
                     decoder=Decoder(input_channel=1024, channels=1536, rates=(6, 5, 5, 2), causal=ga("decoder_causal", False),
                                     lstm=ga("decoder_lstm", 0), engine=eng))
    if stage != "codec":
        raise NotImplementedError("built stages: 'codec' and 'redecoder'")

    def g(obj, name, default):
        if obj is None:
            return default
        return obj[name] if isinstance(obj, dict) and name in obj else getattr(obj, name, default)

    dac = g(args, "DAC", None)
    eng = Engine()
    encoder = Encoder(d_model=g(dac, "encoder_dim", 64), strides=tuple(g(dac, "encoder_rates", (2, 5, 5, 6))),
                      d_latent=1024, causal=g(args, "causal", True), lstm=g(args, "lstm", 2), engine=eng)
    quantizer = FAquantizer(in_dim=1024, n_p_codebooks=1, n_c_codebooks=g(args, "n_c_codebooks", 2), n_t_codebooks=2,
                            n_r_codebooks=3, codebook_size=1024, codebook_dim=8, quantizer_dropout=0.5,
                            causal=g(args, "causal", True),
                            separate_prosody_encoder=g(args, "separate_prosody_encoder", True),
                            timbre_norm=g(args, "timbre_norm", True), engine=eng)
    decoder = Decoder(input_channel=1024, channels=g(dac, "decoder_dim", 1536),
                      rates=tuple(g(dac, "decoder_rates", (6, 5, 5, 2))), causal=g(args, "causal", True),
                      lstm=g(args, "lstm", 2), engine=eng)
    out = Munch(encoder=encoder, quantizer=quantizer, decoder=decoder)
    if with_predictors:
        out["fa_predictors"] = FApredictors(in_dim=1024, use_gr_content_f0=g(args, "use_gr_content_f0", False),
                                            use_gr_prosody_phone=g(args, "use_gr_prosody_phone", False), use_gr_residual_f0=True,
                                            use_gr_residual_phone=True, use_gr_timbre_content=True,
                                            use_gr_timbre_prosody=g(args, "use_gr_timbre_prosody", False), use_gr_x_timbre=True,
                                            norm_f0=g(args, "norm_f0", True), timbre_norm=g(args, "timbre_norm", True),
                                            use_gr_content_global_f0=g(args, "use_gr_content_global_f0", True), engine=eng)
    return out


class ResidualVQ(nn.Module):
    """quantize/rvq.py:12-87 ResidualVQ over quantize/fvq.py:16-116 FactorizedVectorQuantize
    (eval forward), dim=1024 -> codebook_dim=8, 2**codebook_size entries (must be 1024).
    state_dict keys follow the reference: layers.{i}.in_proj.weight_g/_v/bias, out_proj..., _codebook.weight."""

    def __init__(self, *, num_quantizers, codebook_size=10, dim=1024, codebook_dim=8, commitment=0.25, seed=0, **kw):
        super().__init__()
        if dim != 1024 or codebook_dim != 8 or 2 ** int(codebook_size) != 1024 or not (1 <= num_quantizers <= 8):
            raise NotImplementedError("built for dim=1024, codebook_dim=8, 2**10 entries, <= 8 quantizers")
        self.num_quantizers = num_quantizers
        g = synth._Gen(1000 + seed)
        sd = OrderedDict()
        for i in range(num_quantizers):
            tmp = {}
            synth._conv(g, tmp, "in_proj", 8, 1024, 1)
            synth._conv(g, tmp, "out_proj", 1024, 8, 1)
            for k, v in tmp.items():
                v = v.squeeze(-1) if k.endswith("weight_v") else (v.reshape(-1, 1) if k.endswith("weight_g") else v)
                sd[f"layers.{i}.{k}"] = v
            sd[f"layers.{i}._codebook.weight"] = g.normal((1024, 8))
        self._keys = list(sd.keys())
        self._p = nn.ParameterDict({k.replace(".", "/"): nn.Parameter(v, requires_grad=False) for k, v in sd.items()})
        self._engine = Engine()
        self._rvq_id = None
        self._tag = None

    def state_dict(self, *a, prefix="", **kw):
        return OrderedDict((prefix + k, self._p[k.replace(".", "/")].detach()) for k in self._keys)

    def load_state_dict(self, sd, strict=True, assign=False):
        with torch.no_grad():
            for k in self._keys:
                self._p[k.replace(".", "/")].copy_(sd[k])
        self._tag = None

    def _folded(self, i, name):
        v = self._p[f"layers/{i}/{name}/weight_v"].detach().cpu().double()
        g = self._p[f"layers/{i}/{name}/weight_g"].detach().cpu().double()
        # weight_norm(nn.Linear) default dim=0: per output row
        w = (v * (g / v.norm(dim=1, keepdim=True))).float().contiguous()
        return w

    def _sync(self, device):
        e = self._engine
        e._ensure(device)
        tag = tuple(p._version for p in self._p.values())
        if self._tag == tag:
            return
        n = self.num_quantizers
        keep = []

        def arr(ts):
            keep.extend(ts)
            return (ctypes.c_void_p * n)(*[t.data_ptr() for t in ts])
        in_w = arr([self._folded(i, "in_proj") for i in range(n)])
        in_b = arr([self._p[f"layers/{i}/in_proj/bias"].detach().cpu().contiguous() for i in range(n)])
        out_w = arr([self._folded(i, "out_proj") for i in range(n)])
        out_b = arr([self._p[f"layers/{i}/out_proj/bias"].detach().cpu().contiguous() for i in range(n)])
        cb = arr([self._p[f"layers/{i}/_codebook/weight"].detach().cpu().contiguous() for i in range(n)])
        if self._rvq_id is not None:
            e.L.fac_rvq_destroy(e.handle, self._rvq_id)      # weights changed: release the previous device arena
        rid = e.L.fac_rvq_create(e.handle, n, in_w, in_b, out_w, out_b, cb)
        _lib.check(e.handle, rid, "fac_rvq_create")
        self._rvq_id, self._tag = rid, tag

    def forward(self, x, n_quantizers=None, channels_last=False, return_all=True):
        """x [B,1024,T] -> (quantized_out, indices [N,B,T], losses [N] (zeros in eval), all_quantized [N,B,1024,T])."""
        if self.training:
            raise NotImplementedError("eval mode only")
        if n_quantizers is not None and n_quantizers != self.num_quantizers:
            raise NotImplementedError("n_quantizers must equal num_quantizers")
        self._sync(x.device)
        e = self._engine
        x = _f32c(x)
        if channels_last:
            B, T, D = x.shape
        else:
            B, D, T = x.shape
        n = self.num_quantizers
        q = torch.empty_like(x)
        idx = torch.empty(n, B, T, device=x.device, dtype=torch.int64)
        allq = torch.empty((n,) + tuple(x.shape), device=x.device) if return_all else None
        rc = e.L.fac_rvq_forward(e.handle, self._rvq_id, _ptr(x), B, T, 1 if channels_last else 0, _ptr(q), _ptr(idx),
                                 _ptr(allq), _stream())
        _lib.check(e.handle, rc, "fac_rvq_forward")
        return q, idx, torch.zeros(n, device=x.device), allq


class Activation1d(nn.Module):
    """alias_free_torch/act.py:7-29 Activation1d(activation, up_ratio=2, down_ratio=2, 12, 12) with
    activation = SnakeBeta(alpha_logscale) (modules/quantize.py:29-88) or identity (activation=None)."""

    def __init__(self, channels=None, alpha_logscale=True, identity=False):
        super().__init__()
        self.identity = identity
        self.alpha_logscale = alpha_logscale
        if not identity:
            init = torch.zeros(channels) if alpha_logscale else torch.ones(channels)
            self.alpha = nn.Parameter(init.clone(), requires_grad=False)
            self.beta = nn.Parameter(init.clone(), requires_grad=False)
        self._engine = Engine()

    def forward(self, x):
        e = self._engine
        e._ensure(x.device)
        x = _f32c(x)
        B, C, T = x.shape
        y = torch.empty_like(x)
        a = b = None
        if not self.identity:
            a = (torch.exp(self.alpha) if self.alpha_logscale else self.alpha).detach().to(x.device, torch.float32).contiguous()
            b = (torch.exp(self.beta) if self.alpha_logscale else self.beta).detach().to(x.device, torch.float32).contiguous()
        rc = e.L.fac_alias_free_act(e.handle, _ptr(x), B, C, T, 0 if self.identity else 1, _ptr(a), _ptr(b), _ptr(y), _stream())
        _lib.check(e.handle, rc, "fac_alias_free_act")
        return y



class CNNLSTM(nn.Module):
    """modules/quantize.py:106-125 CNNLSTM(indim, outdim, head, global_pred=False), forward only (the FApredictors heads are
    training-side in the reference: SURVEY.md 8f rank 1).  state_dict keys follow the reference, including the registered
    Kaiser-sinc filter buffers of every Activation1d (accepted on load, regenerated on save).  forward(x [B, indim, T]) ->
    list of ``head`` tensors [B, T, outdim] ([B, outdim] when global_pred)."""

    def __init__(self, indim, outdim, head, global_pred=False, seed=0, engine=None):
        super().__init__()
        self.indim, self.outdim, self.nheads, self.global_pred = int(indim), int(outdim), int(head), bool(global_pred)
        sd = synth.synth_cnnlstm(500 + seed, self.indim, self.outdim, self.nheads)
        self._keys = list(sd.keys())
        self._p = nn.ParameterDict({k.replace(".", "/"): nn.Parameter(v, requires_grad=False) for k, v in sd.items()})
        self._engine = engine if engine is not None else Engine()
        self._head_id = None
        self._tag = None

    @staticmethod
    def _filter():
        from math import pi
        ks, half = 12, 6
        A = 2.285 * (half - 1) * pi * (4 * 0.3) + 7.95
        beta = 0.1102 * (A - 8.7) if A > 50.0 else (0.5842 * (A - 21) ** 0.4 + 0.07886 * (A - 21.0) if A >= 21.0 else 0.0)
        win = torch.kaiser_window(ks, beta=beta, periodic=False)
        time = torch.arange(-half, half) + 0.5
        f = 2 * 0.25 * win * torch.sinc(2 * 0.25 * time)
        return (f / f.sum()).view(1, 1, ks)

    def state_dict(self, *a, prefix="", **kw):
        out = OrderedDict()
        for k in self._keys:
            out[prefix + k] = self._p[k.replace(".", "/")].detach()
            if k.endswith("act.beta"):
                base = k[:-len("act.beta")]
                out[prefix + base + "upsample.filter"] = self._filter()
                out[prefix + base + "downsample.lowpass.filter"] = self._filter()
        return out

    def load_state_dict(self, sd, strict=True, assign=False):
        missing = [k for k in self._keys if k not in sd]
        if strict and missing:
            raise RuntimeError("missing keys: %s" % missing[:5])
        with torch.no_grad():
            for k in self._keys:
                if k in sd:
                    self._p[k.replace(".", "/")].copy_(sd[k])
        self._tag = None

    def _sync(self, device):
        e = self._engine
        e._ensure(device)
        tag = tuple(p._version for p in self._p.values())
        if self._tag == tag:
            return
        L, h = e.L, e.handle
        if self._head_id is None:
            self._head_id = _lib.check(h, L.fac_head_begin(h), "fac_head_begin")
        for k in self._keys:
            t = self._p[k.replace(".", "/")].detach().to("cpu", torch.float32).contiguous()
            shape = (ctypes.c_int64 * max(t.dim(), 1))(*t.shape)
            _lib.check(h, L.fac_head_tensor(h, self._head_id, k.encode(), _ptr(t), shape, t.dim()), "fac_head_tensor(%s)" % k)
        _lib.check(h, L.fac_head_finalize(h, self._head_id, self.indim, self.outdim, self.nheads, int(self.global_pred)),
                   "fac_head_finalize")
        self._tag = tag

    def forward(self, x):
        if self.training:
            raise NotImplementedError("eval mode only")
        self._sync(x.device)
        e = self._engine
        x = _f32c(x)
        B, C, T = x.shape
        assert C == self.indim
        shape = (B, self.outdim) if self.global_pred else (B, T, self.outdim)
        outs = [torch.empty(shape, device=x.device) for _ in range(self.nheads)]
        arr = (ctypes.c_void_p * self.nheads)(*[o.data_ptr() for o in outs])
        rc = e.L.fac_head_forward(e.handle, self._head_id, _ptr(x), B, T, arr, _stream(x.device))
        _lib.check(e.handle, rc, "fac_head_forward")
        return outs
