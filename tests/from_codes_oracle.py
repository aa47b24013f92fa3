"""TEST INFRASTRUCTURE ONLY -- CPU restatement of decoding from codes, over the reference's ``state_dict`` in the style of
``oracle/facodec_oracle.py``: ResidualVectorQuantize.from_codes (dac/nn/quantize.py:200-220) per group, then the
FAquantizer.forward_v2 tail (modules/quantize.py:435-449) composed as ``quantizer_forward`` does (:346-356 of the oracle).

Pinned by tests/golden/pin_from_codes.npz, which scripts/make_golden_from_codes.py makes from the imported unmodified
reference's own ``from_codes`` / ``timbre_linear`` / ``timbre_norm`` / ``decoder`` for the inputs ``pin_inputs`` rebuilds
from seeds.  Nothing here reads the reference.
"""
import torch
import torch.nn.functional as F

from oracle.facodec_oracle import _wn_weight

# weight seed (synth.synth_state_dicts), input seed, batch, frames, (n_c, n_r) cases; n_r = 0 has no reference from_codes
PIN_FROM_CODES = dict(wseed=1, seed=31, B=2, T=15, cases=((2, 3), (2, 1), (1, 3), (2, 0)))


def pin_inputs(c=PIN_FROM_CODES):
    """Seeded [codes_p, codes_c, codes_r] (all rows of every group) and timbre [B, 1024]."""
    g = torch.Generator().manual_seed(c["seed"])
    codes = [torch.randint(0, 1024, (c["B"], n, c["T"]), generator=g) for n in (1, 2, 3)]
    timbre = torch.randn(c["B"], 1024, generator=g)
    return codes, timbre


def case_key(n_c, n_r):
    return f"c{n_c}r{n_r}"


def residual_vq_from_codes(sd, prefix, codes):
    """ResidualVectorQuantize.from_codes, dac/nn/quantize.py:200-220: z_q = 0 + sum_i out_proj_i(codebook_i[codes[:, i]])
    over the rows given (decode_code = F.embedding on the raw codebook, transposed to [B, 8, T])."""
    z_q = 0.0
    for i in range(codes.shape[1]):
        p = f"{prefix}.quantizers.{i}"
        z_p_i = F.embedding(codes[:, i, :], sd[p + ".codebook.weight"]).transpose(1, 2)
        z_q = z_q + F.conv1d(z_p_i, _wn_weight(sd, p + ".out_proj"), sd[p + ".out_proj.bias"])
    return z_q


def quantizer_from_codes(sd, codes, timbre, n_c=None, n_r=None):
    """codes = [codes_p [B,1,T], codes_c [B,>=n_c,T], codes_r [B,>=n_r,T] or None], timbre [B,1024] ->
    (outs [B,1024,T], [z_p, z_c, z_r]): the leading n_c / n_r codebooks, z_r = 0 when n_r = 0; then
    LayerNorm(no affine, eps 1e-5) * gamma + beta with (gamma, beta) = timbre_linear(timbre), as forward_v2."""
    cp, cc, cr = codes
    n_c = cc.shape[1] if n_c is None else n_c
    n_r = (0 if cr is None else cr.shape[1]) if n_r is None else n_r
    z_p = residual_vq_from_codes(sd, "prosody_quantizer", cp)
    z_c = residual_vq_from_codes(sd, "content_quantizer", cc[:, :n_c])
    z_r = residual_vq_from_codes(sd, "residual_quantizer", cr[:, :n_r]) if n_r else torch.zeros_like(z_p)
    outs = 0 + z_p
    outs = outs + z_c
    outs = outs + z_r
    style = F.linear(timbre, sd["timbre_linear.weight"], sd["timbre_linear.bias"]).unsqueeze(2)
    gamma, beta = style.chunk(2, 1)
    o = outs.transpose(1, 2)
    o = F.layer_norm(o, (o.shape[-1],), None, None, 1e-5)
    o = o.transpose(1, 2)
    return o * gamma + beta, [z_p, z_c, z_r]
