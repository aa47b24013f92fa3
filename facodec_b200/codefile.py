"""On-disk code format: the reference's ``.dac`` file (dac/model/base.py:15-54 ``DACFile``).

A ``.dac`` file is ``np.save`` of one dict: ``codes`` as uint16 ``[B, n_codebooks, frames]`` plus a ``metadata`` dict
(``input_db`` float32 array, ``original_length``, ``sample_rate``, ``chunk_length``, ``channels``, ``padding``,
``dac_version`` = "1.0.0").  This module writes byte-identical files and reads the reference's (tests/test_oracle.py
checks both directions against the imported class).  The codec's three code tensors (prosody ``[B, 1, T']``, content
``[B, n_c, T']``, residual ``[B, 3, T']``, modules/quantize.py:451-454) are stacked along the codebook axis in that order.
Host-side numpy only: there is no arithmetic here to put on the GPU.
"""
from dataclasses import dataclass
from pathlib import Path
from typing import Sequence

import numpy as np
import torch

SUPPORTED_VERSIONS = ["1.0.0"]          # dac/model/base.py:12
HOP_LENGTH = 300                        # samples per frame (config.yml encoder rates 2*5*5*6)


@dataclass
class DACFile:
    """Same fields, ``save`` and ``load`` as dac/model/base.py:15-54."""
    codes: torch.Tensor
    chunk_length: int
    original_length: int
    input_db: torch.Tensor
    channels: int
    sample_rate: int
    padding: bool
    dac_version: str

    # the order of the metadata entries is part of the byte format (np.save pickles the dict)
    _META_ORDER = ("input_db", "original_length", "sample_rate", "chunk_length", "channels", "padding", "dac_version")

    def _metadata(self):
        db = self.input_db.detach().cpu().numpy() if torch.is_tensor(self.input_db) else np.asarray(self.input_db)
        values = dict(input_db=db.astype(np.float32), original_length=self.original_length, sample_rate=self.sample_rate,
                      chunk_length=self.chunk_length, channels=self.channels, padding=self.padding,
                      dac_version=SUPPORTED_VERSIONS[-1])
        return {k: values[k] for k in self._META_ORDER}

    def save(self, path):
        """Writes ``<path>.dac`` (the suffix is forced, as the reference does) and returns the path."""
        grid = self.codes.detach().cpu().numpy()
        if grid.size and (grid.min() < 0 or grid.max() > np.iinfo(np.uint16).max):
            raise ValueError("codes do not fit the format's uint16")
        target = Path(path).with_suffix(".dac")
        with open(target, "wb") as fh:
            np.save(fh, {"codes": grid.astype(np.uint16), "metadata": self._metadata()})
        return target

    @classmethod
    def load(cls, path):
        """Reads a ``.dac`` file written here or by the reference; refuses unknown format versions."""
        blob = np.load(path, allow_pickle=True)[()]
        meta = dict(blob["metadata"])
        if meta.get("dac_version", None) not in SUPPORTED_VERSIONS:
            raise RuntimeError(f"Given file {path} can't be loaded with this version of descript-audio-codec.")
        return cls(codes=torch.from_numpy(blob["codes"].astype(int)), **meta)


def pack_codes(codes: Sequence[torch.Tensor]) -> torch.Tensor:
    """[codes_p [B,1,T'], codes_c [B,n_c,T'], codes_r [B,3,T']] -> one ``[B, 1 + n_c + 3, T']`` int64 tensor."""
    return torch.cat([c.detach().cpu().to(torch.int64) for c in codes], dim=1)


def unpack_codes(packed: torch.Tensor, n_c: int = 2):
    """Inverse of :func:`pack_codes` (the residual quantizer always has 3 codebooks, modules/quantize.py:416-418)."""
    if packed.dim() != 3 or packed.shape[1] != 1 + n_c + 3:
        raise ValueError(f"expected [B, {1 + n_c + 3}, T'] codes, got {tuple(packed.shape)}")
    return [packed[:, :1], packed[:, 1:1 + n_c], packed[:, 1 + n_c:]]


def from_forward(codes: Sequence[torch.Tensor], original_length: int, sample_rate: int = 24000, input_db=None,
                 chunk_length: int = None, channels: int = 1, padding: bool = True) -> DACFile:
    """A :class:`DACFile` for the ``codes`` list ``model.quantizer(..., return_codes=True)`` returns."""
    packed = pack_codes(codes)
    if input_db is None:
        input_db = torch.zeros(packed.shape[0], dtype=torch.float32)
    return DACFile(codes=packed, chunk_length=packed.shape[-1] if chunk_length is None else chunk_length,
                   original_length=int(original_length), input_db=input_db, channels=channels, sample_rate=sample_rate,
                   padding=padding, dac_version=SUPPORTED_VERSIONS[-1])


def decode(model, dac_or_path, timbre, n_c: int = 2, n_r: int = None) -> torch.Tensor:
    """Audio from a ``.dac`` file (a path or a loaded :class:`DACFile`) of a build_model() Munch: unpack the codes (``n_c``
    content rows per the file's layout), move them to ``timbre``'s device and run ``Codec(model).decode_codes``.  The
    format holds codes only, so the timbre [B, 1024] (one vector per utterance, e.g. the forward's own) is an argument;
    ``n_r`` residual codebooks are used (default: all in the file).  Returns y [B, 1, 300 T']."""
    from .modules import Codec
    f = dac_or_path if isinstance(dac_or_path, DACFile) else DACFile.load(dac_or_path)
    codes = [c.to(timbre.device) for c in unpack_codes(f.codes, n_c=n_c)]
    return Codec(model).decode_codes(codes, timbre, n_c=n_c, n_r=n_r)
