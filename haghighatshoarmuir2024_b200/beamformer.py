"""Beamformer: drop-in for the non-spiking Hilbert beamformer of micloc/beamformer.py.

`apply_to_signal` (micloc/beamformer.py:260-292) runs STHT + band-pass + complex
projection on the GPU (micloc_hilbert_beamform) and returns complex128 `T x G`.
`localize` and `design_from_template` take batches through micloc_hilbert_localize, which
gets power, DoA and the design covariance from one Gram matrix of the analytic signal per
clip and never forms the dense `T x G` output.  `HilbertStreamBatch` (and the one-band
`Beamformer.stream_batch`) runs the same chain over many live recordings, state carried
from frame to frame (micloc_hilbert_streams_*).
"""
from __future__ import annotations

import ctypes as C
from numbers import Number
from typing import Dict, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch
from scipy.linalg import eigh
from scipy.signal import butter, hilbert

from . import _native as N
from .array_geometry import ArrayGeometry
from .engine import ChainSpec, SnnEngine, _SlotBatch, _activity, _check_frames, _ptr, _stream_ptr

Fs = 48_000


class Beamformer:
    def __init__(self, geometry: ArrayGeometry, kernel_duration: float, freq_range: List, fs: float = Fs,
                 device: int = 0):
        self.geometry = geometry
        self.kernel_duration = kernel_duration
        self.fs = fs
        ker_len = int(fs * kernel_duration)
        impulse = np.zeros(ker_len)
        impulse[0] = 1
        self.kernel = np.fft.fftshift(np.imag(hilbert(impulse)))
        self.freq_range = np.asarray(freq_range)
        try:
            f_low, f_high = freq_range
            if f_low > f_high:
                raise Exception()
        except Exception:
            raise ValueError("freq_range should be a vector consisting of two frequencies f_low < f_high!")
        self.bandpass_filter = butter(2, freq_range, btype="bandpass", analog=False, output="ba", fs=fs)
        self.bandpass_sos = butter(2, freq_range, btype="bandpass", analog=False, output="sos", fs=fs)
        self.device = device
        self.verbose = True
        self._eng = None
        self._hbf = None            # the engine's Hilbert steering matrix

    def _engine(self) -> SnnEngine:
        if self._eng is None:
            M = len(self.geometry)
            # the spike/neuron constants are unused by the Hilbert path; any valid values do
            spec = ChainSpec(num_mic=M, stht_kernel=self.kernel, sos=self.bandpass_sos, robust_width=1,
                             bipolar=False, neuron_decay=0.5, neuron_scale=1.0, neuron_len=1)
            self._eng = SnnEngine(spec, np.zeros((2 * M, 1)), device=self.device)
        return self._eng

    def _hilbert_engine(self, bf_mat: np.ndarray) -> SnnEngine:
        """The engine with bf_mat [M, G] as its Hilbert steering matrix, uploaded only when it changed."""
        eng = self._engine()
        if self._hbf is None or self._hbf.shape != bf_mat.shape or not np.array_equal(self._hbf, bf_mat):
            eng.set_hilbert_bf(bf_mat)
            self._hbf = bf_mat.copy()
        return eng

    def hilbert_signal(self, sig_in: np.ndarray) -> np.ndarray:
        """Band-passed analytic signal `T x M` complex128 (beamformer.py:281-287)."""
        eng = self._engine()
        x = torch.from_numpy(np.ascontiguousarray(sig_in, dtype=np.float32)).to(eng.device)
        z = eng.run_taps(x, want=("z",))["z"][0].cpu().numpy().astype(np.float64)
        M = len(self.geometry)
        return z[:, :M] + 1j * z[:, M:]

    def design_from_template(self, template: Tuple[np.ndarray, np.ndarray], doa_list: np.ndarray,
                             interference_removal: bool = False):
        """(bf_mat `M x G` complex, list of covariance matrices) (beamformer.py:73-192)."""
        try:
            time_temp, sig_temp = template
        except Exception:
            raise ValueError("input template should be a tuple containing (time_in, sig_in) of the template signal!")
        time_interp = np.arange(np.min(time_temp), np.max(time_temp), step=1 / self.fs)
        sig_temp = np.interp(time_interp, time_temp, sig_temp)
        time_temp = time_interp
        if self.verbose:
            print()
            print("+" * 150)
            print(" designing beamforming matrices for various DoAs ".center(150, "+"))
            print("+" * 150)
        eng = self._engine()
        time_temp = np.asarray(time_temp, dtype=np.float64)
        T = len(time_temp)
        # the analytic signal roll(x, K/2) + j STHT(x) without band-pass (upstream band-passes a copy it never uses,
        # beamformer.py:136-137), covariance over its stable part: one batched device call per chunk of DoAs
        t_start = min(len(self.kernel), T // 2)
        chunk = max(1, min(len(doa_list), (256 << 20) // max(1, 4 * T * len(self.geometry))))
        cov_mat_list = []
        for d0 in range(0, len(doa_list), chunk):
            sig = np.empty((min(chunk, len(doa_list) - d0), T, len(self.geometry)), dtype=np.float32)
            for i, doa in enumerate(doa_list[d0:d0 + chunk]):
                delays = self.geometry.delays(theta=doa, normalized=True)
                td = time_temp.reshape(-1, 1) - delays.reshape(1, -1)
                td[td < time_temp.min()] = time_temp.min()
                sig[i] = np.interp(td.ravel(), time_temp, sig_temp).reshape(td.shape)
            x = torch.from_numpy(sig).to(eng.device)
            cov = eng.hilbert(x, t_start=t_start, bandpass=False, want=("cov",))["cov"].cpu().numpy()
            cov_mat_list.extend(cov / (T - t_start))
        bf_mat = []
        if not interference_removal:
            for Cm in cov_mat_list:
                U, _, _ = np.linalg.svd(Cm)
                bf_mat.append(U[:, 0])
        else:
            C_sum = 0
            for Cm in cov_mat_list:
                C_sum = C_sum + Cm
            C_sum = C_sum + np.diag(np.mean(np.diag(C_sum)) * np.ones(C_sum.shape[0])) / 10
            for Cm in cov_mat_list:
                _, vecs = eigh(Cm, C_sum - Cm)   # ascending eigenvalues: last is the largest
                v = vecs[:, -1]
                bf_mat.append(v / np.linalg.norm(v))
        return np.asarray(bf_mat).T, cov_mat_list

    def design_on_device(self, template: Tuple[np.ndarray, np.ndarray], doa_list: np.ndarray,
                         interference_removal: bool = False) -> Tuple[torch.Tensor, torch.Tensor]:
        """(bf complex128 `[M, G]`, cov complex128 `[G, M, M]`) designed on the GPU from the template to the steering
        vectors (micloc_hilbert_design), both device tensors.  cov equals design_from_template's list; every column
        equals the host's up to a phase (the device makes its entry of largest modulus real and positive)."""
        try:
            time_temp, sig_temp = template
        except Exception:
            raise ValueError("input template should be a tuple containing (time_in, sig_in) of the template signal!")
        time_interp = np.arange(np.min(time_temp), np.max(time_temp), step=1 / self.fs)
        sig_interp = np.interp(time_interp, time_temp, sig_temp)
        return self._engine().hilbert_design(self.geometry, time_interp, sig_interp, doa_list,
                                             interference_removal=interference_removal)

    def localize(self, bf_mat: np.ndarray, audio) -> dict:
        """Batched hot path: audio [B,T,M] (CUDA tensor, float32/int16) -> dict(doa [B] int32, power [B,G] float32).

        Equals argmax(mean(|apply_to_signal(bf_mat, x)|**2, axis=0)) per clip without the dense T x G array."""
        bf_mat = np.asarray(bf_mat)
        num_mic, num_grid = bf_mat.shape
        num_chan = audio.shape[-1]
        if num_chan != num_mic:
            raise ValueError(
                f"number of channels in the input siganl {num_chan} should be the same as the number of microphones {num_mic}!")
        return self._hilbert_engine(bf_mat).hilbert(audio, want=("doa", "power"))

    def stream_batch(self, bf_mat: np.ndarray, num_streams: int, max_frame_len: int) -> "HilbertStreamBatch":
        """`num_streams` live recordings through this beamformer's own band-pass chain, no filterbank in front."""
        return HilbertStreamBatch([(self, bf_mat)], num_streams, max_frame_len)

    def apply_to_template(self, bf_mat: np.ndarray, template, snr_db: float) -> np.ndarray:
        """beamformer.py:194-258: delayed + noisy array signal, then apply_to_signal."""
        try:
            time_temp, sig_temp, doa_temp = template
        except Exception:
            raise ValueError(
                "input template should be a tuple containing (time_in, sig_in, doa_in) of the template signal!")
        if isinstance(doa_temp, Number):
            doa_temp = doa_temp * np.ones_like(sig_temp)
        snr = 10 ** (snr_db / 10)
        time_in = np.arange(np.min(time_temp), np.max(time_temp), step=1 / self.fs)
        sig_in = np.interp(time_in, time_temp, sig_temp)
        doa_in = np.interp(time_in, time_temp, doa_temp)
        delays = self.geometry.delays_batch(doa_in)
        delays = delays - delays.min()
        td = time_in.reshape(-1, 1) - delays
        td[td < time_in.min()] = time_in.min()
        sig_vec = np.interp(td.ravel(), time_in, sig_in).reshape(td.shape)
        sig_vec = sig_vec + np.sqrt(np.mean(sig_vec ** 2)) / np.sqrt(snr) * np.random.randn(*sig_vec.shape)
        return self.apply_to_signal(bf_mat=bf_mat, sig_in=sig_vec)

    def apply_to_signal(self, bf_mat: np.ndarray, sig_in: np.ndarray) -> np.ndarray:
        bf_mat = np.asarray(bf_mat)
        num_mic, num_grid = bf_mat.shape
        T, num_chan = np.shape(sig_in)
        if num_chan != num_mic:
            raise ValueError(
                f"number of channels in the input siganl {num_chan} should be the same as the number of microphones {num_mic}!")
        eng = self._engine()
        x = torch.from_numpy(np.ascontiguousarray(sig_in, dtype=np.float32)).to(eng.device).unsqueeze(0)
        y = torch.empty((1, T, num_grid, 2), dtype=torch.float32, device=eng.device)
        bre = np.ascontiguousarray(bf_mat.real, dtype=np.float64)
        bim = np.ascontiguousarray(bf_mat.imag, dtype=np.float64)
        N.check(N.lib().micloc_hilbert_beamform(eng._h, _ptr(x), N.F32, 1, T, bre.ctypes.data_as(N._dp),
                                                bim.ctypes.data_as(N._dp), num_grid, _ptr(y), None, None,
                                                _stream_ptr(eng.device)))
        yh = y[0].cpu().numpy().astype(np.float64)
        return yh[..., 0] + 1j * yh[..., 1]


class HilbertStreamBatch(_SlotBatch):
    """`num_streams` independent live recordings ("slots") through the Hilbert beamformer with its state carried across
    pushes (micloc_hilbert_streams_*).  `bands` is a list of (Beamformer, bf_mat [M, G] complex) of one array and one
    DoA grid; `filterbank` (a ButterworthFilterbank, one band per entry of `bands`) runs in front of them, or, when None,
    the single band takes the raw frames.  N pushed frames give every band's analytic signal of their concatenation
    (after the filterbank, if any), with the stream's causal in-phase delay.  Every pushed sample is final at once
    (latency 0, no flush); `reset(slots)` restarts the listed slots.  The steering matrices are copied at creation."""

    def __init__(self, bands, num_streams: int, max_frame_len: int, filterbank=None, doa_list=None):
        bands = list(bands)
        if not bands:
            raise ValueError("a Hilbert stream batch needs at least one band")
        if filterbank is not None and len(filterbank.sos_list) != len(bands):
            raise ValueError(f"the filterbank has {len(filterbank.sos_list)} bands, the batch {len(bands)}")
        self.bands = bands
        self.engines = [beamf._hilbert_engine(np.asarray(bf_mat)) for beamf, bf_mat in bands]
        self.F = len(bands)
        self.M, self.G = self.engines[0].M, np.asarray(bands[0][1]).shape[1]
        self.C2 = 2 * self.M
        self.filterbank = filterbank
        self.doa_list = None if doa_list is None else np.ascontiguousarray(doa_list, dtype=np.float64)
        lib = N.lib()
        sos = None if filterbank is None else np.ascontiguousarray(filterbank.sos_list, dtype=np.float64)
        ctxs = (C.c_void_p * self.F)(*[e._h.value for e in self.engines])
        h = C.c_void_p()
        N.check(lib.micloc_hilbert_streams_create(
            ctxs, self.F, 0 if sos is None else sos.shape[1], None if sos is None else sos.ctypes.data_as(N._dp),
            None if self.doa_list is None else self.doa_list.ctypes.data_as(N._dp), int(num_streams),
            int(max_frame_len), C.byref(h)))
        self._attach(lib, h, "micloc_hilbert_streams", int(num_streams), int(max_frame_len), self.engines[0].device)
        self._doa_dev = None if self.doa_list is None else torch.from_numpy(self.doa_list).to(self.device)

    def push(self, frames: torch.Tensor, want: Sequence[str] = ("doa", "power"), rel_threshold: float = 0.0001,
             full_scale: Optional[float] = None) -> Dict[str, object]:
        """One frame [num_streams, n, channels] per slot in (int32 / int16 / float32; channels beyond the microphones
        are dropped), this push's n rows out, as device tensors: any of 'z' [F, S, n, 2M], 'cov' [F, S, M, M]
        complex128 (sum conj(s_t) s_t^T), 'power' [F, S, G] (mean |s_t . conj(bf_g)|^2), 'power_grid' [S, G] (sum over
        the bands), 'doa' [S] (its first argmax), 'periodic_ml' / 'trimmed_periodic_ml' [S] (need doa_list) and
        'flags' [S] (bit 1: the trimmed estimator's IndexError).  With a filterbank, also 'sumsq' [S] of the frame,
        'active' [S] (its rms against rel_threshold * full_scale, as Demo.localize) and, when 'doa' is wanted and
        doa_list was given, 'doa_deg' [S] (NaN where inactive).  'n_out' (numpy int64 [S]) is n for every slot.  No
        host synchronisation."""
        frames, dt = _check_frames(frames, self.M, self.device, self.num_streams)
        S, n, ch = frames.shape
        dev = self.device
        mk = lambda name, shape, dtype: torch.empty(shape, dtype=dtype, device=dev) if name in want else None
        out = {"z": mk("z", (self.F, S, n, self.C2), torch.float32),
               "cov": mk("cov", (self.F, S, self.M, self.M, 2), torch.float64),
               "power": mk("power", (self.F, S, self.G), torch.float32),
               "power_grid": mk("power_grid", (S, self.G), torch.float32),
               "doa": mk("doa", (S,), torch.int32),
               "periodic_ml": mk("periodic_ml", (S,), torch.float64),
               "trimmed_periodic_ml": mk("trimmed_periodic_ml", (S,), torch.float64),
               "flags": mk("flags", (S,), torch.int32)}
        sumsq = torch.empty(S, dtype=torch.float64, device=dev) if self.filterbank is not None else None
        n_out = np.zeros(S, dtype=np.int64)
        N.check(self._lib.micloc_hilbert_streams_push(
            self._h, _ptr(frames), dt, n, ch, _ptr(out["z"]), _ptr(out["cov"]), _ptr(out["power"]),
            _ptr(out["power_grid"]), _ptr(out["doa"]), _ptr(out["periodic_ml"]), _ptr(out["trimmed_periodic_ml"]),
            _ptr(sumsq), _ptr(out["flags"]), n_out.ctypes.data_as(C.c_void_p), _stream_ptr(dev)))
        if out["cov"] is not None:
            out["cov"] = torch.view_as_complex(out["cov"])
        out = {k: v for k, v in out.items() if v is not None}
        out["n_out"] = n_out
        if sumsq is not None:
            out["sumsq"] = sumsq
            out["active"], doa_deg = _activity(sumsq, n, self.M, frames.dtype, rel_threshold, full_scale,
                                               out.get("doa"), self._doa_dev)
            if doa_deg is not None:
                out["doa_deg"] = doa_deg
        return out
