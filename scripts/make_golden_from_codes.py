"""Writes tests/golden/pin_from_codes.npz (and nothing else) from the imported unmodified reference on the CPU; needs a
checkout of the reference at oracle.ref_import.REFERENCE_ROOT.

    python scripts/make_golden_from_codes.py

Model: build_reference_model(0) (configs/config.yml) loaded with synth.synth_state_dicts(wseed).  Inputs: the seeded codes
and timbre of tests/from_codes_oracle.pin_inputs.  Per (n_c, n_r) case: z_p / z_c / z_r from the reference's own
prosody_quantizer / content_quantizer / residual_quantizer.from_codes (dac/nn/quantize.py:200-220), outs from its
timbre_linear and timbre_norm applied in forward_v2 order (modules/quantize.py:435-449), y = model.decoder(outs).  With
n_r = 0 the residual from_codes is skipped (torch.cat([]) raises there) and z_r is 0.  Stored as make_golden.pinned does.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from facodec_b200 import synth  # noqa: E402
from from_codes_oracle import PIN_FROM_CODES, case_key, pin_inputs  # noqa: E402
from oracle import ref_import  # noqa: E402
from oracle.make_golden import GOLDEN_DIR, pinned  # noqa: E402


def main():
    import warnings
    warnings.simplefilter("ignore")
    c = PIN_FROM_CODES
    model = ref_import.build_reference_model(0)
    sds = synth.synth_state_dicts(c["wseed"])
    for k in ("quantizer", "decoder"):
        model[k].load_state_dict(sds[k])
    q = model.quantizer
    (cp, cc, cr), timbre = pin_inputs(c)
    out = {}
    with torch.no_grad():
        for n_c, n_r in c["cases"]:
            z_p = q.prosody_quantizer.from_codes(cp)[0]
            z_c = q.content_quantizer.from_codes(cc[:, :n_c])[0]
            outs = 0 + z_p
            outs = outs + z_c
            if n_r:
                z_r = q.residual_quantizer.from_codes(cr[:, :n_r])[0]
                outs += z_r
            else:
                z_r = torch.zeros_like(z_p)
            style = q.timbre_linear(timbre).unsqueeze(2)
            gamma, beta = style.chunk(2, 1)
            outs = q.timbre_norm(outs.transpose(1, 2)).transpose(1, 2)
            outs = outs * gamma + beta
            y = model.decoder(outs)
            p = case_key(n_c, n_r) + "_"
            out.update(pinned(**{p + "z_p": z_p, p + "z_c": z_c, p + "z_r": z_r, p + "outs": outs, p + "y": y}))
    path = os.path.join(GOLDEN_DIR, "pin_from_codes.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
