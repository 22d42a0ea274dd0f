"""Butterworth filterbank design (host side), mirrored from micloc/filterbank.py.

`evolve` keeps the reference's return layout (F x T x M) and runs on the host with
scipy (it is only used to prepare live-demo frames); inside the Xylo chain the
band filters run on the device as SOS cascades (csrc/micloc_staged.cuh:k_chain_blk).
"""
from __future__ import annotations

from typing import List

import numpy as np
from scipy.signal import butter, lfilter


class Filterbank:
    def __init__(self, ba_list: List):
        self.ba_list = ba_list

    def evolve(self, sig_in: np.ndarray) -> np.ndarray:
        sig_in = np.asarray(sig_in)
        if sig_in.ndim == 1:
            sig_in = sig_in.reshape(-1, 1)
        return np.asarray([lfilter(b, a, sig_in, axis=0) for b, a in self.ba_list])

    __call__ = evolve

    def __len__(self):
        return len(self.ba_list)


class ButterworthFilterbank(Filterbank):
    """One butter(order, band, 'bandpass') per band (micloc/filterbank.py:49-84)."""

    def __init__(self, freq_bands: List, order: int, fs: float):
        self.order, self.fs = order, fs
        fb = np.asarray(freq_bands, dtype=np.float64)
        self.freq_bands = fb.reshape(1, -1) if fb.ndim == 1 else fb
        ba_list, self.sos_list = [], []
        for band in self.freq_bands:
            ba_list.append(butter(order, band, btype="bandpass", output="ba", fs=fs))
            self.sos_list.append(butter(order, band, btype="bandpass", output="sos", fs=fs))
        super().__init__(ba_list=ba_list)
