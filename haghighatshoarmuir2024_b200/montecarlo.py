"""Batched Monte-Carlo localisation sweep: the driver loop of
paper_plots/target_snn_localization.py:431-467 (11 SNRs x num_sim random-DoA trials,
one clip per trial) re-stated as batches of independent clips per frequency band.

Clips are synthesised ON THE DEVICE by the library's own kernels (micloc_synth_clips)
exactly as SNNBeamformer.apply_to_template builds them
(micloc/snn_beamformer.py:243-275: per-microphone delay, linear interpolation of the
sampled source clamped at t_min, AWGN at the requested SNR), then go through the
fused CUDA chain of one `SnnEngine` per band; only DoA indices, per-DoA power and a
DoA histogram come back.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch
from scipy.signal import butter, hilbert

from . import _native as N
from .engine import ChainSpec, SnnEngine, neuron_alpha_params

SPEED_OF_SOUND = 340.0            # micloc/array_geometry.py:14


@dataclass
class BandSetup:
    band: Sequence[float]
    tau: float
    bf_mat: np.ndarray            # [2M, G]
    bf_hilbert: Optional[np.ndarray] = None   # [M, G] complex: steering of the Hilbert beamformer arm (run_band_hilbert)


def stht_kernel(fs: float, kernel_duration: float) -> np.ndarray:
    """micloc/snn_beamformer.py:45-53."""
    K = int(fs * kernel_duration)
    impulse = np.zeros(K)
    impulse[0] = 1
    return np.fft.fftshift(np.imag(hilbert(impulse)))


def band_chain_spec(num_mic: int, fs: float, kernel: np.ndarray, band, tau: float, T: int,
                    bipolar: bool = True) -> ChainSpec:
    """Constants SNNBeamformer derives for one band (micloc/snn_beamformer.py:58-80, 342-361)."""
    sos = butter(2, band, btype="bandpass", analog=False, output="sos", fs=fs)
    robust_width = max(int(fs / band[1]) // 2, 1)
    _, a, c, L = neuron_alpha_params(np.arange(T) / fs, [tau, tau])
    return ChainSpec(num_mic=num_mic, stht_kernel=kernel, sos=sos, robust_width=robust_width, bipolar=bipolar,
                     neuron_decay=a, neuron_scale=c, neuron_len=L)


def synthesize_clips(r_vec, theta_vec, fs: float, T: int, doa, snr_lin=None, source=None, source_index=None,
                     sine_freq: float = 0.0, gain=None, mode: int = 0, seed: int = 0, dtype: torch.dtype = torch.float32,
                     int16_peak: float = 12000.0, device: int = 0) -> torch.Tensor:
    """Synthetic array clips [B, T, M] on the GPU with the library's synthesis kernels (micloc_synth_clips).

    mode 0 restates SNNBeamformer.apply_to_template (micloc/snn_beamformer.py:243-275), mode 1
    signal_multiple_targets (paper_plots/multiple_targets_snn.py:87-159).  `doa` [B] or [B, n_targets] radians;
    `source` None = sine of `sine_freq`, else a float table [T] or [S, T] on the clip grid (+ `source_index` [B]);
    `snr_lin` [B] linear SNR per clip (None = noiseless); dtype float32 or int16 (peak `int16_peak` per clip)."""
    dev = torch.device("cuda", device)
    lib = N.lib()
    doa_t = torch.as_tensor(np.asarray(doa, dtype=np.float64))
    if doa_t.dim() == 1:
        doa_t = doa_t.unsqueeze(1)
    B, K = doa_t.shape
    r = np.ascontiguousarray(r_vec, dtype=np.float64)
    th = np.ascontiguousarray(theta_vec, dtype=np.float64)
    M = len(r)
    cfg = N.SynthConfig()
    cfg.num_mic, cfg.r_vec, cfg.theta_vec = M, r.ctypes.data_as(N._dp), th.ctypes.data_as(N._dp)
    cfg.fs, cfg.speed, cfg.clip_len, cfg.n_targets, cfg.mode = float(fs), SPEED_OF_SOUND, int(T), int(K), int(mode)
    cfg.source_kind, cfg.sine_freq = (1, float(sine_freq)) if source is None else (0, 0.0)
    src = idx = None
    if source is not None:
        src = torch.as_tensor(np.asarray(source, dtype=np.float32)).reshape(-1, T).contiguous().to(dev)
        if source_index is not None:
            idx = torch.as_tensor(np.asarray(source_index, dtype=np.int32)).contiguous().to(dev)
            if idx.numel() != B or int(idx.max()) >= src.shape[0]:
                raise ValueError("source_index must hold one valid row per clip")
    gn = None if gain is None else torch.as_tensor(np.asarray(gain, dtype=np.float32)).reshape(B, K).contiguous().to(dev)
    sn = None if snr_lin is None else torch.as_tensor(np.asarray(snr_lin, dtype=np.float32)).reshape(B).contiguous().to(dev)
    out16 = None
    if dtype == torch.int16:
        out16 = torch.empty((B, T, M), dtype=torch.int16, device=dev)
    elif dtype != torch.float32:
        raise ValueError("dtype must be float32 or int16")
    out = torch.empty((B, T, M), dtype=torch.float32, device=dev)
    p_ = lambda t: None if t is None else C.c_void_p(t.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    chunk = 65535
    for b0 in range(0, B, chunk):
        b1 = min(B, b0 + chunk)
        d = doa_t[b0:b1].contiguous().to(dev)
        scratch = torch.empty(2 * (b1 - b0), dtype=torch.float64, device=dev)
        sl = lambda t: None if t is None else t[b0:b1]
        N.check(lib.micloc_synth_clips(C.byref(cfg), b1 - b0, p_(src), p_(sl(idx)), p_(d), p_(sl(gn)), p_(sl(sn)),
                                       int(seed) + b0, p_(out[b0:b1]), p_(sl(out16)), float(int16_peak), p_(scratch),
                                       device, st))
    return out if out16 is None else out16


class SnrSweep:
    """One engine per band on one GPU + on-device clip synthesis."""

    def __init__(self, bands: List[BandSetup], r_vec, theta_vec, fs: float, kernel_duration: float, T: int,
                 device: int = 0, bipolar: bool = True):
        self.fs, self.T = float(fs), int(T)
        self.device = torch.device("cuda", device)
        self.r_vec = np.asarray(r_vec, dtype=np.float64)
        self.theta_vec = np.asarray(theta_vec, dtype=np.float64)
        self.M = len(self.r_vec)
        self.kernel = stht_kernel(fs, kernel_duration)
        self.bands = bands
        self.specs = [band_chain_spec(self.M, fs, self.kernel, b.band, b.tau, T, bipolar) for b in bands]
        self.engines = [SnnEngine(s, b.bf_mat, device=device) for s, b in zip(self.specs, bands)]
        for eng, b in zip(self.engines, bands):
            if b.bf_hilbert is not None:
                eng.set_hilbert_bf(b.bf_hilbert)
        self.G = bands[0].bf_mat.shape[1]

    # ------------------------------------------------------------------
    def synthesize(self, band_idx: int, B: int, seed: int, snr_db_grid: Sequence[float],
                   dtype: torch.dtype = torch.float32):
        """B noisy single-target clips for band `band_idx`: sine at the band's upper edge
        (freq_design, target_snn_localization.py:439-441), DoA ~ U[0, 2 pi) (:452), SNR cycling
        through `snr_db_grid` minus the bandwidth correction (:382, :449).
        Returns (audio [B,T,M] device tensor, doa_true [B] float64 numpy, snr_index [B])."""
        band = self.bands[band_idx].band
        rng = np.random.default_rng(int(seed))
        doa = rng.uniform(0.0, 2 * np.pi, size=B)
        snr_idx = np.arange(B) % len(snr_db_grid)
        corr = 10 * np.log10((self.fs / 2) / (band[1] - band[0]))
        snr = 10 ** ((np.asarray(snr_db_grid, dtype=np.float64)[snr_idx] - corr) / 10)
        out = synthesize_clips(self.r_vec, self.theta_vec, self.fs, self.T, doa, snr_lin=snr, sine_freq=float(band[1]),
                               mode=0, seed=int(seed), dtype=dtype, device=self.device.index or 0)
        return out, doa, snr_idx

    # ------------------------------------------------------------------
    def run_band(self, band_idx: int, audio: torch.Tensor, want_spikes: bool = False, want_power: bool = True,
                 hist: Optional[torch.Tensor] = None, refine: bool = True) -> Dict[str, torch.Tensor]:
        """One band's batch through the fused kernel.  refine=False keeps the call stream-ordered (no read-back of the
        RZCC overflow flags); the caller then runs `self.engines[band_idx].refine(audio, out)` once per step."""
        eng = self.engines[band_idx]
        out = eng.run(audio, want_spikes=want_spikes, want_power=want_power, fused=True, refine=refine)
        if hist is not None:
            self.histogram(out["doa"], hist)
        return out

    def run_band_hilbert(self, band_idx: int, audio: torch.Tensor, hist: Optional[torch.Tensor] = None
                         ) -> Dict[str, torch.Tensor]:
        """The same batch through the Hilbert beamformer on the band's engine (its STHT and band-pass; steering
        `bf_hilbert` of the band): dict(doa, power); stream-ordered."""
        if self.bands[band_idx].bf_hilbert is None:
            raise ValueError(f"band {band_idx} has no bf_hilbert")
        out = self.engines[band_idx].hilbert(audio, want=("doa", "power"))
        if hist is not None:
            self.histogram(out["doa"], hist)
        return out

    def histogram(self, doa: torch.Tensor, hist: torch.Tensor) -> None:
        """hist[g] += count(doa == g) with the library's own kernel (int64 [G] on this GPU)."""
        assert hist.dtype == torch.int64 and hist.numel() == self.G and hist.device == doa.device
        st = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        N.check(N.lib().micloc_doa_histogram(C.c_void_p(doa.data_ptr()), doa.numel(), self.G,
                                             C.c_void_p(hist.data_ptr()), self.device.index or 0, st))

    def doa_error(self, doa_idx: np.ndarray, doa_true: np.ndarray, doa_list: np.ndarray) -> np.ndarray:
        """arcsin|sin(est - true)| (target_snn_localization.py:466)."""
        return np.arcsin(np.abs(np.sin(doa_list[doa_idx] - doa_true)))
