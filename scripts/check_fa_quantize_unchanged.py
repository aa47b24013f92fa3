"""Checks that two trees of this project compute the same quantizer forward, bit for bit: each tree (its own
facodec_b200 package with its library built in place) runs model.quantizer on the same seeded BASELINE configs[1] batch
(B = 32 utterances x 4 s, synth weights of seed 0) in a subprocess of its own, and outs, z_p / z_c / z_r, timbre and the
three code tensors are compared with torch.equal.  Used to show that a refactor of fa_quantize_kernel changed nothing.

    python scripts/check_fa_quantize_unchanged.py OTHER_TREE [THIS_TREE]
"""
import os
import subprocess
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

RUN = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
import facodec_b200 as fb
from facodec_b200 import synth
assert fb.__file__.startswith(sys.argv[1]), fb.__file__
torch.cuda.set_device(0)
sds = synth.synth_state_dicts(0)
m = fb.build_model()
for k in ("encoder", "quantizer", "decoder"):
    m[k].load_state_dict(sds[k]); m[k].eval()
x = synth.synth_waves(32, 96000, seed=2024).cuda()
z = m.encoder(x)
q = m.quantizer(z, x, n_c=2, return_codes=True)
torch.cuda.synchronize()
out = dict(z=z, outs=q[0], z_p=q[1][0], z_c=q[1][1], z_r=q[1][2], timbre=q[4], codes_p=q[5][0], codes_c=q[5][1], codes_r=q[5][2])
torch.save({k: v.cpu() for k, v in out.items()}, sys.argv[2])
"""


def run(tree, path):
    subprocess.check_call([sys.executable, "-c", RUN, os.path.abspath(tree), path])
    return torch.load(path)


def main():
    other = sys.argv[1]
    this = sys.argv[2] if len(sys.argv) > 2 else ROOT
    with tempfile.TemporaryDirectory() as d:
        a = run(other, os.path.join(d, "other.pt"))
        b = run(this, os.path.join(d, "this.pt"))
    ok = True
    for k in a:
        eq = torch.equal(a[k], b[k])
        ok &= eq
        print(f"{k:8s} {tuple(b[k].shape)} torch.equal {eq}")
    print("quantizer forward at configs[1] (B=32 x 4 s): %s" % ("IDENTICAL" if ok else "DIFFERENT"))
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
