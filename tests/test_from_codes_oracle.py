"""CPU: decoding from codes.  (a) The restatement (tests/from_codes_oracle.py) against what the imported unmodified
reference's from_codes / timbre_linear / timbre_norm / decoder returned (pin_from_codes.npz); (b) the reference-written
.dac file unpacks into the codec's three groups; (c) the Python layer rejects bad codes before anything reaches the
library."""
import os

import numpy as np
import pytest
import torch

from conftest import state_dicts
from from_codes_oracle import PIN_FROM_CODES, case_key, pin_inputs, quantizer_from_codes
from oracle import facodec_oracle as O
from oracle import make_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ATOL = 2e-5          # as tests/test_oracle.py: the pins were made on one host CPU


def _close_pinned(got, g, name):
    got = got.detach().numpy()
    assert got.shape == tuple(g[name + "_shape"]), name
    a, b = make_golden.sample(got), g[name]
    assert np.abs(a - b).max() <= ATOL * max(1.0, np.abs(b).max()), f"{name}: max diff {np.abs(a - b).max()}"


@pytest.mark.parametrize("n_c,n_r", PIN_FROM_CODES["cases"])
def test_from_codes_oracle_matches_imported_reference(n_c, n_r):
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "pin_from_codes.npz")))
    sds = state_dicts(PIN_FROM_CODES["wseed"])
    codes, timbre = pin_inputs()
    with torch.no_grad():
        outs, (z_p, z_c, z_r) = quantizer_from_codes(sds["quantizer"], codes, timbre, n_c, n_r)
        y = O.decoder_forward(sds["decoder"], outs)
    p = case_key(n_c, n_r) + "_"
    for name, t in (("z_p", z_p), ("z_c", z_c), ("z_r", z_r), ("outs", outs), ("y", y)):
        _close_pinned(t, g, p + name)
    if n_r == 0:
        assert not z_r.any()


def test_reference_dac_file_unpacks_into_three_groups():
    from facodec_b200 import codefile
    f = codefile.DACFile.load(os.path.join(ROOT, "tests", "golden", "pin_codefile.dac"))
    groups = codefile.unpack_codes(f.codes, n_c=2)
    assert [t.shape[1] for t in groups] == [1, 2, 3]
    assert all(t.dtype == torch.int64 and t.shape[0] == 2 and t.shape[2] == 37 for t in groups)


class _NoLibrary:
    def __getattr__(self, name):
        raise AssertionError("reached the library: " + name)


@pytest.fixture
def quantizer(built_lib):
    import facodec_b200 as fb
    q = fb.FAquantizer().eval()
    q._engine.L = _NoLibrary()          # validation must fail before any library call
    return q


def _codes(B=2, T=15):
    codes, _ = pin_inputs(dict(PIN_FROM_CODES, B=B, T=T))
    return codes, torch.randn(B, 1024)


def test_wrong_row_counts_rejected(quantizer):
    (cp, cc, cr), tv = _codes()
    for bad in ([cp.repeat(1, 2, 1), cc, cr], [cp, cc.repeat(1, 2, 1), cr], [cp, cc, cr.repeat(1, 2, 1)],
                [cp, cc[:, :0], cr]):
        with pytest.raises(ValueError):
            quantizer.from_codes(bad, tv)
    for n_c, n_r in ((3, 3), (0, 3), (2, 4), (2, -1)):
        with pytest.raises(ValueError):
            quantizer.from_codes([cp, cc, cr], tv, n_c=n_c, n_r=n_r)
    with pytest.raises(ValueError):
        quantizer.from_codes([cp, cc[:, :1], cr], tv, n_c=2)
    with pytest.raises(ValueError):
        quantizer.from_codes([cp, cc, cr], tv[:1])
    with pytest.raises(ValueError):
        quantizer.from_codes([cp, cc, cr], tv[:, :512])
    with pytest.raises(TypeError):
        quantizer.from_codes([cp.float(), cc, cr], tv)


def test_mismatched_frames_rejected(quantizer):
    (cp, cc, cr), tv = _codes()
    with pytest.raises(ValueError):
        quantizer.from_codes([cp, cc[:, :, :14], cr], tv)
    with pytest.raises(ValueError):
        quantizer.from_codes([cp, cc, cr[:, :, 1:]], tv)
    with pytest.raises(ValueError):
        quantizer.from_codes([cp, cc[:1], cr], tv)


@pytest.mark.parametrize("value", [1024, 5000, -1])
@pytest.mark.parametrize("group", [0, 1, 2])
def test_out_of_range_codes_raise_index_error(quantizer, value, group):
    codes, tv = _codes()
    codes[group][-1, -1, 3] = value
    with pytest.raises(IndexError):
        quantizer.from_codes(codes, tv)


def test_unused_rows_are_not_checked(quantizer):
    """Only the n_c / n_r leading rows are decoded; codes in the others are never read."""
    from facodec_b200 import FacError
    (cp, cc, cr), tv = _codes()
    cc[:, 1] = 1024
    cr[:, 2] = -1
    with pytest.raises(FacError):                 # passes validation, then refuses the CPU tensors
        quantizer.from_codes([cp, cc, cr], tv, n_c=1, n_r=2)


def test_cpu_tensors_raise_fac_error(built_lib):
    import facodec_b200 as fb
    (cp, cc, cr), tv = _codes()
    q = fb.FAquantizer().eval()
    with pytest.raises(fb.FacError):
        q.from_codes([cp, cc, cr], tv)
