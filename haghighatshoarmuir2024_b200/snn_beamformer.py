"""SNNBeamformer: drop-in for micloc/snn_beamformer.py backed by the CUDA hot path.

Same constructor, attributes and method signatures as the reference class
(micloc/snn_beamformer.py:24-422).  `apply_to_signal` returns the dense float64
`T x num_DoA` array the reference returns; `localize` is the batched call a
Monte-Carlo driver should use (audio in, DoA indices out, nothing dense).
"""
from __future__ import annotations

from collections import OrderedDict
from numbers import Number
from typing import Dict, Tuple, Union

import numpy as np
import torch
from scipy.signal import butter, hilbert

from .array_geometry import ArrayGeometry
from .engine import ChainSpec, SnnEngine, neuron_alpha_params
from .spike_encoder import ZeroCrossingSpikeEncoder

Fs = 48_000


class SNNBeamformer:
    def __init__(self, geometry: ArrayGeometry, kernel_duration: float, freq_range: np.ndarray,
                 tau_vec: np.ndarray, bipolar_spikes: bool = False, fs: float = Fs, device: int = 0):
        self.geometry = geometry
        self.fs = fs
        # STHT kernel (snn_beamformer.py:45-53)
        self.kernel_duration = kernel_duration
        self.kernel_length = int(self.fs * self.kernel_duration)
        impulse = np.zeros(self.kernel_length)
        impulse[0] = 1
        self.kernel = np.fft.fftshift(np.imag(hilbert(impulse)))
        self.tau_vec = tau_vec
        # band-pass (snn_beamformer.py:58-72)
        try:
            f_low, f_high = freq_range
            if f_low > f_high:
                raise Exception()
        except Exception:
            raise ValueError("freq_range should be a vector consisting of two frequencies f_low < f_high!")
        self.bandpass_filter = butter(2, freq_range, btype="bandpass", analog=False, output="ba", fs=fs)
        self.bandpass_sos = butter(2, freq_range, btype="bandpass", analog=False, output="sos", fs=fs)
        # RZCC encoder (snn_beamformer.py:74-80)
        robust_width = int(fs / f_high) // 2
        self.bipolar_spikes = bipolar_spikes
        self.spk_encoder = ZeroCrossingSpikeEncoder(fs=self.fs, robust_width=robust_width, bipolar=bipolar_spikes,
                                                    device=device)
        self.device = device
        self.verbose = True
        self._engines: "OrderedDict[tuple, SnnEngine]" = OrderedDict()
        self.max_engines = 4          # contexts kept alive (one per clip length / encoder setting), least recently used first out

    # ------------------------------------------------------------------
    def chain_spec(self, time_vec: np.ndarray) -> ChainSpec:
        _, a, c, L = neuron_alpha_params(time_vec, self.tau_vec)
        return ChainSpec(num_mic=len(self.geometry), stht_kernel=self.kernel, sos=self.bandpass_sos,
                         robust_width=max(int(np.ceil(self.spk_encoder.robust_width)), 1),
                         bipolar=self.spk_encoder.bipolar, neuron_decay=a, neuron_scale=c, neuron_len=L)

    def engine(self, bf_mat: np.ndarray, time_vec: np.ndarray) -> SnnEngine:
        """Context for (neuron kernel implied by time_vec, bf_mat); cached."""
        spec = self.chain_spec(time_vec)
        if self.spk_encoder.robust_width < 1:
            raise ValueError("`distance` must be greater or equal to 1")
        # the encoder's settings are read at evolve time in the reference (callers may change them after construction)
        key = (spec.neuron_len, round(spec.neuron_decay, 15), round(spec.neuron_scale, 18), spec.num_mic,
               spec.robust_width, bool(spec.bipolar))
        eng = self._engines.get(key)
        # the beamforming matrix is a per-call argument: the same array object (unchanged since) skips the hashing
        same_obj = eng is not None and getattr(eng, "_bf_obj", None) is bf_mat and not getattr(bf_mat, "flags", None) is None \
            and not bf_mat.flags.writeable
        if same_obj:
            self._engines.move_to_end(key)
            return eng
        bf = np.ascontiguousarray(bf_mat, dtype=np.float64)
        sig = (bf.shape, hash(bf.tobytes()))
        if eng is None:
            eng = SnnEngine(spec, bf, device=self.device)
            eng._bf_sig = sig
            self._engines[key] = eng
            while len(self._engines) > self.max_engines:          # variable-length frames must not grow GPU memory without bound
                _, old = self._engines.popitem(last=False)
                old.close()
        elif eng._bf_sig != sig:
            eng.set_bf(bf)
            eng._bf_sig = sig
        eng._bf_obj = bf_mat
        self._engines.move_to_end(key)
        return eng

    # ------------------------------------------------------------------
    def _delayed_template(self, time_temp, sig_temp, delays):
        """T x M array of the template delayed per microphone, clamped at t_min (snn_beamformer.py:146-154)."""
        td = time_temp.reshape(1, -1) - np.asarray(delays).reshape(-1, 1)
        td[td < time_temp.min()] = time_temp.min()
        return np.interp(td.ravel(), time_temp, sig_temp).reshape(td.shape).T

    def design_from_template(self, template: Tuple[np.ndarray, np.ndarray], doa_list: np.ndarray) -> np.ndarray:
        """Beamforming matrix `2 num_mic x num_DoA` (snn_beamformer.py:82-211).

        The per-DoA front end (STHT, band-pass, RZCC, neuron filter) and the covariance
        run batched on the GPU; the small eigen-problems stay on the host."""
        try:
            time_temp, sig_temp = template
        except Exception:
            raise ValueError("input template should be a tuple containing (time_in, sig_in) of the template signal!")
        time_temp = np.asarray(time_temp, dtype=np.float64)
        time_interp = np.arange(time_temp.min(), time_temp.max(), step=1 / self.fs)
        sig_interp = np.interp(time_interp, time_temp, sig_temp)
        sig_temp, time_temp = sig_interp, time_interp
        if self.verbose:
            print()
            print("+" * 150)
            print(" designing SNN beamforming matrices for various DoAs ".center(150, "+"))
            print("+" * 150)
        doa_list = np.asarray(doa_list, dtype=np.float64)
        M, T = len(self.geometry), len(time_temp)
        eng = self.engine(np.zeros((2 * M, 1)), time_temp)
        t_start = T // 4
        covs = []
        chunk = max(1, min(len(doa_list), (256 << 20) // (T * M * 4)))
        for g0 in range(0, len(doa_list), chunk):
            clips = np.empty((min(chunk, len(doa_list) - g0), T, M), dtype=np.float32)
            for i, doa in enumerate(doa_list[g0:g0 + chunk]):
                delays = self.geometry.delays(theta=doa, normalized=True)
                delays = delays - delays.min()
                clips[i] = self._delayed_template(time_temp, sig_temp, delays)
            gram = eng.gram(torch.from_numpy(clips).to(eng.device), t_start)
            covs.append(gram.cpu().numpy() / (T - t_start))
        covs = np.concatenate(covs, axis=0)
        bf_mat = []
        for Cm in covs:
            if not self.spk_encoder.bipolar:
                bf_vec = self._find_dc_removed_sing_vec(Cm, rel_prec=0.00000001)
            else:
                d = Cm.shape[0] // 2
                C_diag = (Cm[:d, :d] + Cm[d:, d:]) / 2
                C_off = (Cm[:d, d:] + Cm[d:, :d].T) / 2
                U, _, _ = np.linalg.svd(C_diag + 1j * C_off)
                bf_vec = np.concatenate([np.real(U[:, 0]), np.imag(U[:, 0])])
            bf_mat.append(bf_vec)
        return np.asarray(bf_mat).T

    def design_on_device(self, template: Tuple[np.ndarray, np.ndarray], doa_list: np.ndarray) -> torch.Tensor:
        """Beamforming matrix float64 `[2 num_mic, num_DoA]` on the beamformer's GPU, designed there from the template
        to the steering vectors (micloc_snn_design): the same covariances as design_from_template and the same
        unipolar vectors; bipolar columns equal the host's up to a phase of u = Re + i Im (the device makes the entry
        of largest modulus real and positive).  Only the resampling of the template onto the fs grid runs on the host."""
        try:
            time_temp, sig_temp = template
        except Exception:
            raise ValueError("input template should be a tuple containing (time_in, sig_in) of the template signal!")
        time_temp = np.asarray(time_temp, dtype=np.float64)
        time_interp = np.arange(time_temp.min(), time_temp.max(), step=1 / self.fs)
        sig_interp = np.interp(time_interp, time_temp, sig_temp)
        M = len(self.geometry)
        eng = self.engine(np.zeros((2 * M, 1)), time_interp)
        bf, _ = eng.snn_design(self.geometry, time_interp, sig_interp, doa_list)
        return bf

    def synthesize_from_template(self, template, snr_db: float, rng=None) -> Tuple[np.ndarray, np.ndarray]:
        """(time, `T x num_mic` noisy array signal) exactly as apply_to_template builds it
        (snn_beamformer.py:230-275); `rng=None` uses numpy's global RNG like the reference."""
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
        delays = self.geometry.delays_batch(doa_in).T          # M x T, un-normalised
        delays = delays - delays.min()
        td = time_in.reshape(1, -1) - delays
        td[td < time_in.min()] = time_in.min()
        sig_vec = np.interp(td.ravel(), time_in, sig_in).reshape(td.shape).T
        randn = np.random.randn if rng is None else (lambda *s: rng.standard_normal(s))
        sig_vec = sig_vec + np.sqrt(np.mean(sig_vec ** 2)) / np.sqrt(snr) * randn(*sig_vec.shape)
        return time_in, sig_vec

    def apply_to_template(self, bf_mat: np.ndarray, template, snr_db: float) -> np.ndarray:
        """Beamformed signal for a (time, signal, doa) template at a given SNR (snn_beamformer.py:213-281)."""
        time_in, sig_vec = self.synthesize_from_template(template, snr_db)
        return self.apply_to_signal(bf_mat=bf_mat, sig_in_vec=(time_in, sig_vec))

    def _prepare_signal(self, bf_mat, sig_in_vec):
        time_vec, sig = sig_in_vec
        time_vec = np.asarray(time_vec, dtype=np.float64)
        sig = np.asarray(sig)
        twice_num_mic, _ = np.shape(bf_mat)
        num_mic = twice_num_mic // 2
        T, num_chan = sig.shape
        if num_chan != num_mic:
            raise ValueError(
                f"number of channels in the input siganl {num_chan} should be the same as the number of microphones {num_mic}!")
        if not np.allclose(np.diff(time_vec), 1 / self.fs):   # snn_beamformer.py:309-321
            t_new = np.arange(time_vec[0], time_vec[-1], step=1 / self.fs)
            t_all = np.repeat(time_vec.reshape(1, -1), num_mic, axis=0)
            t_new_all = np.repeat(t_new.reshape(1, -1), num_mic, axis=0)
            sig = np.interp(t_new_all.ravel(), t_all.ravel(), sig.ravel()).reshape(-1, num_mic)
            time_vec = t_new
        return time_vec, sig

    def apply_to_signal(self, bf_mat: np.ndarray, sig_in_vec: Tuple[np.ndarray, np.ndarray]) -> np.ndarray:
        """`T x num_DoA` float64 beamformed membrane signal (snn_beamformer.py:283-370)."""
        time_vec, sig = self._prepare_signal(bf_mat, sig_in_vec)
        eng = self.engine(bf_mat, time_vec)
        x = torch.from_numpy(np.ascontiguousarray(sig, dtype=np.float32)).to(eng.device)
        out = eng.run_taps(x, want=("y",))
        return out["y"][0].cpu().numpy().astype(np.float64)

    def localize(self, bf_mat: np.ndarray, time_vec: np.ndarray, audio, want_spikes: bool = False,
                 fused: bool = True):
        """Batched hot path: audio [B,T,M] (CUDA tensor, float32/int16) -> dict(doa, power, spikes, flags).

        Equals argmax(mean(|apply_to_signal(...)|**2, axis=0)) per clip
        (paper_plots/target_snn_localization.py:462-464) without the dense T x G array."""
        eng = self.engine(bf_mat, time_vec)
        return eng.run(audio, want_spikes=want_spikes, want_power=True, fused=fused)

    def _find_dc_removed_sing_vec(self, C: np.ndarray, rel_prec: float = 0.0001):
        """Top singular vector of PSD C constrained orthogonal to the all-one vector:
        bisection on the secular equation sum_k theta_k^2/(d_k - u) = 0 between the two
        largest singular values (snn_beamformer.py:372-422)."""
        U, D, _ = np.linalg.svd(C)
        theta = U.T @ np.ones(C.shape[0])
        u_min, u_max = D[1], D[0]
        while (u_max - u_min) / u_min >= rel_prec:
            u_mid = (u_min + u_max) / 2
            if np.sum(theta ** 2 / (D - u_mid)) < 0.0:
                u_min = u_mid
            else:
                u_max = u_mid
        root = (u_min + u_max) / 2.0
        vec = U @ (theta / (D - root))
        return vec / np.linalg.norm(vec)
