"""Xylo-quantised integer localisation: drop-in for micloc/xylo_snn_localization.py (class `Demo`)
backed by the CUDA chain of csrc/micloc_xylo.cu.

What is mirrored (reference file:line):
  signal_from_template            micloc/xylo_snn_localization.py:44-71
  Demo.__init__                   :75-171   one SNNBeamformer + bf_mat per band, order-1 filterbank
  Demo._initialize_snn_module     :173-313  block-diagonal weights, [W; -W] for bipolar spikes,
                                            w_rec = -0.1/N, threshold 1, tau * fs / 1000, then
                                            rockpool mapper -> global_quantize -> XyloSim
  Demo.spike_encoding             :315-356
  Demo.xylo_process               :358-377
  Demo.extract_rate               :379-398
  Demo.estimate_doa_from_rate     :400-444

rockpool / xylosim are third-party and absent here; `quantize_network` restates
rockpool.transform.quantize_methods.global_quantize + the mapper's dash computation, and the
device kernel restates XyloSim's hidden-layer integer dynamics (see DESIGN.md, "Xylo": parity
unpinned at that boundary).  The live-demo parts of the reference class (recorder,
visualiser, hardware board) are out of scope.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from numbers import Number
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _native as N
from .array_geometry import ArrayGeometry
from .engine import _SlotBatch, _check_frames, _ptr, _stream_ptr
from .filterbank import ButterworthFilterbank
from .snn_beamformer import SNNBeamformer

MAX_HIDDEN_SPIKES = 31          # spikes per hidden neuron per time step on Xylo-2


def signal_from_template(geometry: ArrayGeometry, template) -> np.ndarray:
    """`T x num_mic` array signal for a (time, signal, doa) template
    (micloc/xylo_snn_localization.py:44-71: delays ADDED, np.interp clamps at both ends)."""
    time_temp, sig_temp, doa_temp = template
    time_temp = np.asarray(time_temp, dtype=np.float64)
    if isinstance(doa_temp, Number):
        doa_temp = doa_temp * np.ones_like(time_temp)
    delays = geometry.delays_batch(np.asarray(doa_temp, dtype=np.float64))   # T x M, un-normalised
    time_delays = time_temp.reshape(-1, 1) + delays
    return np.interp(time_delays.ravel(), time_temp, sig_temp).reshape(*time_delays.shape)


@dataclass
class XyloNetwork:
    """Integer constants of the hidden layer as XyloSim receives them."""
    w_in: np.ndarray            # int8 [N_in, N]
    w_rec: Optional[np.ndarray]  # int8 [N, N] or None when it quantises to all-zero
    threshold: np.ndarray       # int16 [N]
    dash_syn: np.ndarray        # int8 [N]
    dash_mem: np.ndarray        # int8 [N]
    bias: Optional[np.ndarray] = None
    weight_shift_in: int = 0
    weight_shift_rec: int = 0
    max_spikes: int = MAX_HIDDEN_SPIKES
    scale: float = 1.0          # float weight -> integer weight factor (for inspection)


def quantize_network(bf_mats: Sequence[np.ndarray], tau_vecs: np.ndarray, fs: float, bipolar: bool,
                     target_dt: float = 1e-3, threshold: float = 1.0) -> XyloNetwork:
    """Float network of Demo._initialize_snn_module (:186-237) -> Xylo integers.

    Restates rockpool's `mapper` (dash = log2(tau / dt)) and `global_quantize` (one scale
    127 / max(|W_in|, |W_rec|) for input and recurrent weights and the hidden thresholds,
    np.round, dash rounded to the nearest integer)."""
    scale_t = fs / (1.0 / target_dt)                                   # :186-188
    scaled_tau = np.asarray(tau_vecs, dtype=np.float64) * scale_t
    F = len(bf_mats)
    c_in, c_out = bf_mats[0].shape
    weight = np.zeros((F * c_in, F * c_out))
    for ch in range(F):                                                # :203-208
        weight[ch * c_in:(ch + 1) * c_in, ch * c_out:(ch + 1) * c_out] = bf_mats[ch]
    if bipolar:
        weight = np.vstack([weight, -weight])                          # :211-216
    n_hidden = F * c_out
    # the reference stores everything as float32 torch tensors (:218, :227-232)
    w32 = weight.astype(np.float32).astype(np.float64)
    w_rec32 = float(np.float32(-0.1 / n_hidden))
    tau_syn = np.repeat(scaled_tau[:, 0].astype(np.float32).astype(np.float64), c_out)
    tau_mem = np.repeat(scaled_tau[:, 1].astype(np.float32).astype(np.float64), c_out)
    # mapper: dash = log2(tau / dt); global_quantize rounds it
    dash_syn = np.round(np.log2(tau_syn / target_dt)).astype(np.int64)
    dash_mem = np.round(np.log2(tau_mem / target_dt)).astype(np.int64)
    w_max = max(np.abs(w32).max(), abs(w_rec32))
    scale = (2 ** 7 - 1) / w_max if w_max != 0 else 1.0
    w_in_q = np.round(w32 * scale).astype(np.int64)
    w_rec_q = int(np.round(w_rec32 * scale))
    thr_q = int(np.round(threshold * scale))
    if thr_q > 2 ** 15 - 1 or thr_q < 1:
        raise ValueError(f"quantised threshold {thr_q} does not fit Xylo's 16-bit threshold")
    if np.any(dash_syn < 0) or np.any(dash_mem < 0):
        raise ValueError("time constants shorter than dt cannot be mapped to a bit-shift decay")
    w_rec = None
    if w_rec_q != 0:
        w_rec = np.full((n_hidden, n_hidden), w_rec_q, dtype=np.int8)
    return XyloNetwork(w_in=np.ascontiguousarray(w_in_q.astype(np.int8)), w_rec=w_rec,
                       threshold=np.full(n_hidden, thr_q, dtype=np.int16),
                       dash_syn=np.ascontiguousarray(dash_syn.astype(np.int8)),
                       dash_mem=np.ascontiguousarray(dash_mem.astype(np.int8)), scale=float(scale))


class XyloEngine:
    """One `micloc_xylo` context on one GPU (batched; device tensors in and out)."""

    def __init__(self, num_mic: int, stht_kernel: np.ndarray, sos_list: Sequence[np.ndarray],
                 ba_list: Sequence[Tuple[np.ndarray, np.ndarray]], robust_width: int, bipolar: bool,
                 net: XyloNetwork, num_doa: int, device: int = 0):
        if not torch.cuda.is_available():
            raise RuntimeError("XyloEngine needs a CUDA device (B200); there is no CPU fallback")
        self._lib = N.lib()
        self.device = torch.device("cuda", device)
        F = len(sos_list)
        self.M, self.F, self.G = int(num_mic), F, int(num_doa)
        self.N = int(net.w_in.shape[1])
        self.CT = 2 * self.M * F
        self.N_in = self.CT * (2 if bipolar else 1)
        if net.w_in.shape != (self.N_in, self.N):
            raise ValueError(f"w_in should have shape ({self.N_in}, {self.N}); got {net.w_in.shape}")
        self._keep = dict(
            kernel=np.ascontiguousarray(stht_kernel, dtype=np.float64),
            sos=np.ascontiguousarray(np.stack([np.asarray(s, dtype=np.float64).reshape(-1, 6) for s in sos_list])),
            ba_b=np.ascontiguousarray(np.stack([np.asarray(b, dtype=np.float64) / a[0] for b, a in ba_list])),
            ba_a=np.ascontiguousarray(np.stack([np.asarray(a, dtype=np.float64) / a[0] for b, a in ba_list])),
            w_in=np.ascontiguousarray(net.w_in, dtype=np.int8),
            w_rec=None if net.w_rec is None else np.ascontiguousarray(net.w_rec, dtype=np.int8),
            thr=np.ascontiguousarray(net.threshold, dtype=np.int16),
            ds=np.ascontiguousarray(net.dash_syn, dtype=np.int8),
            dm=np.ascontiguousarray(net.dash_mem, dtype=np.int8),
            bias=None if net.bias is None else np.ascontiguousarray(net.bias, dtype=np.int16),
        )
        k = self._keep
        cfg = N.XyloConfig()
        cfg.num_mic = self.M
        cfg.kernel_len = len(k["kernel"])
        cfg.stht_kernel = k["kernel"].ctypes.data_as(N._dp)
        cfg.num_bands = F
        cfg.n_sections = k["sos"].shape[1]
        cfg.sos = k["sos"].ctypes.data_as(N._dp)
        cfg.n_ba = k["ba_b"].shape[1]
        cfg.ba_b = k["ba_b"].ctypes.data_as(N._dp)
        cfg.ba_a = k["ba_a"].ctypes.data_as(N._dp)
        cfg.robust_width = int(robust_width)
        cfg.bipolar = int(bool(bipolar))
        cfg.num_hidden = self.N
        cfg.num_doa = self.G
        cfg.w_in = k["w_in"].ctypes.data_as(C.POINTER(C.c_int8))
        cfg.w_rec = None if k["w_rec"] is None else k["w_rec"].ctypes.data_as(C.POINTER(C.c_int8))
        cfg.threshold = k["thr"].ctypes.data_as(C.POINTER(C.c_int16))
        cfg.dash_syn = k["ds"].ctypes.data_as(C.POINTER(C.c_int8))
        cfg.dash_mem = k["dm"].ctypes.data_as(C.POINTER(C.c_int8))
        cfg.bias = None if k["bias"] is None else k["bias"].ctypes.data_as(C.POINTER(C.c_int16))
        cfg.weight_shift_in = int(net.weight_shift_in)
        cfg.weight_shift_rec = int(net.weight_shift_rec)
        cfg.max_spikes = int(net.max_spikes)
        h = C.c_void_p()
        N.check(self._lib.micloc_xylo_create(C.byref(cfg), device, C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self._lib.micloc_xylo_destroy(self._h)
            self._h = None

    __del__ = close

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def run(self, audio: torch.Tensor, exact: bool = True, want_spikes_in: bool = False, want_raster: bool = False,
            peak_win: int = 0) -> Dict[str, Optional[torch.Tensor]]:
        """audio [B,T,M] (float32 / int16, on this GPU) -> counts [B,N], doa [B], doa_peak [B]
        (+ input spikes [B,T,N_in] in {0,1}, hidden raster [B,T,N] on request)."""
        if audio.dim() == 2:
            audio = audio.unsqueeze(0)
        if audio.dim() != 3 or audio.shape[2] != self.M:
            raise ValueError(f"number of channels in the input siganl {audio.shape[-1]} should be the same as the "
                             f"number of microphones {self.M}!")
        if audio.dtype == torch.float32:
            dt = N.F32
        elif audio.dtype == torch.int16:
            dt = N.I16
        else:
            raise ValueError(f"audio must be float32 or int16, got {audio.dtype}")
        if audio.device != self.device:
            raise ValueError(f"audio lives on {audio.device}, engine on {self.device}")
        audio = audio.contiguous()
        B, T, _ = audio.shape
        dev = self.device
        counts = torch.empty((B, self.N), dtype=torch.int32, device=dev)
        doa = torch.empty(B, dtype=torch.int32, device=dev)
        flags = torch.empty(B, dtype=torch.int32, device=dev)
        doa_peak = torch.empty(B, dtype=torch.int32, device=dev) if peak_win else None
        spikes_in = torch.empty((B, T, self.N_in), dtype=torch.int8, device=dev) if want_spikes_in else None
        raster = torch.empty((B, T, self.N), dtype=torch.uint8, device=dev) if want_raster else None
        N.check(self._lib.micloc_xylo_run(self._h, _ptr(audio), dt, B, T, int(bool(exact)), _ptr(spikes_in), _ptr(raster),
                                          _ptr(counts), _ptr(doa), _ptr(doa_peak), int(peak_win), _ptr(flags),
                                          self._stream()))
        return {"counts": counts, "doa": doa, "doa_peak": doa_peak, "spikes_in": spikes_in, "raster": raster,
                "flags": flags}

    def process(self, spikes_in: torch.Tensor, want_raster: bool = True, peak_win: int = 0):
        """Integer network only: spikes_in [B,T,N_in] int8 {0,1} on this GPU."""
        if spikes_in.dim() == 2:
            spikes_in = spikes_in.unsqueeze(0)
        if spikes_in.dim() != 3 or spikes_in.shape[2] != self.N_in or spikes_in.dtype != torch.int8:
            raise ValueError(f"spikes_in should be an int8 tensor of shape [B, T, {self.N_in}]")
        spikes_in = spikes_in.contiguous()
        B, T, _ = spikes_in.shape
        dev = self.device
        counts = torch.empty((B, self.N), dtype=torch.int32, device=dev)
        doa = torch.empty(B, dtype=torch.int32, device=dev)
        doa_peak = torch.empty(B, dtype=torch.int32, device=dev) if peak_win else None
        raster = torch.empty((B, T, self.N), dtype=torch.uint8, device=dev) if want_raster else None
        N.check(self._lib.micloc_xylo_process(self._h, _ptr(spikes_in), B, T, _ptr(raster), _ptr(counts), _ptr(doa),
                                              _ptr(doa_peak), int(peak_win), self._stream()))
        return {"counts": counts, "doa": doa, "doa_peak": doa_peak, "raster": raster}


class XyloStreamBatch(_SlotBatch):
    """`num_streams` independent recordings ("slots") through the exact (float64) front end and the integer network
    with their state carried across pushes (micloc_xylo_streams_*).  N pushed frames plus a flush give, for every slot,
    bit for bit what `XyloEngine.run(exact=True)` gives on one clip of their concatenation (in-phase branch: the causal
    delay x[t - K/2]); results lag the input by `latency` samples.  Slot lists, positions, flushed slots and unwritten
    rows as in `MultibandStreamBatch`.  Frames are [num_streams, n, channels] device tensors, int32 / int16 / float32
    (channels beyond the microphones are dropped).

    `fs` and `doa_list` (the DoA grid, radians) serve the per-call estimators: rate [S, G] as `Demo.extract_rate` over
    each slot's final samples, periodic_ml / trimmed_periodic_ml [S] as `Demo.estimate_doa_from_rate` (through
    micloc_power_fuse: the angle is scale-free, so the band-summed counts go in as they are)."""

    def __init__(self, engine: XyloEngine, num_streams: int, max_frame_len: int, fs: float = 48_000.0,
                 doa_list: Optional[np.ndarray] = None):
        self.engine = engine
        self.fs = float(fs)
        self.M, self.F, self.G, self.N, self.N_in = engine.M, engine.F, engine.G, engine.N, engine.N_in
        lib = N.lib()
        h = C.c_void_p()
        rc = lib.micloc_xylo_streams_create(engine._h, int(num_streams), int(max_frame_len), C.byref(h))
        if rc in (N.ERR_CONFIG, N.ERR_UNSUPPORTED):
            raise N.MiclocError(rc, lib.micloc_last_error().decode("utf-8", "replace"))
        N.check(rc)
        self._attach(lib, h, "micloc_xylo_streams", int(num_streams), int(max_frame_len), engine.device)
        self._doa_dev = None
        if doa_list is not None:
            doa_list = np.ascontiguousarray(doa_list, dtype=np.float64)
            if doa_list.shape != (self.G,):
                raise ValueError(f"doa_list should hold {self.G} angles")
            self._doa_dev = torch.from_numpy(doa_list).to(self.device)

    def _outputs(self, rows, want_spikes_in, want_raster, peak_win):
        S, dev = self.num_streams, self.device
        return {"spikes_in": torch.empty((S, rows, self.N_in), dtype=torch.int8, device=dev) if want_spikes_in else None,
                "raster": torch.empty((S, rows, self.N), dtype=torch.uint8, device=dev) if want_raster else None,
                "counts": torch.zeros((S, self.N), dtype=torch.int32, device=dev),
                "doa": torch.full((S,), -1, dtype=torch.int32, device=dev),          # -1: not written (n_out == 0)
                "doa_peak": torch.full((S,), -1, dtype=torch.int32, device=dev) if peak_win else None,
                "flags": torch.empty(S, dtype=torch.int32, device=dev)}

    def _estimators(self, out, n_out):
        """rate [S, G] (Demo.extract_rate over the final samples) and the periodic-ML estimators; NaN where n_out == 0."""
        S, F, G = self.num_streams, self.F, self.G
        cnt = out["counts"].view(S, F, G)
        n = torch.from_numpy(n_out).to(self.device)
        live = n > 0
        rate = cnt.sum(1, dtype=torch.int64).double() * self.fs / (F * n.clamp(min=1).double()).unsqueeze(1)
        out["rate"] = torch.where(live.unsqueeze(1), rate, torch.full_like(rate, float("nan")))
        fflags = torch.zeros(S, dtype=torch.int32, device=self.device)
        if self._doa_dev is not None:
            power = cnt.permute(1, 0, 2).float().contiguous()                       # [F][S][G]
            ml = torch.empty(S, dtype=torch.float64, device=self.device)
            trimmed = torch.empty(S, dtype=torch.float64, device=self.device)
            N.check(self._lib.micloc_power_fuse(_ptr(power), F, S, G, _ptr(self._doa_dev), None, None, _ptr(ml),
                                                _ptr(trimmed), _ptr(fflags), self.device.index or 0,
                                                _stream_ptr(self.device)))
            nan = torch.full_like(ml, float("nan"))
            out["periodic_ml"] = torch.where(live, ml, nan)
            out["trimmed_periodic_ml"] = torch.where(live, trimmed, nan)
            fflags = torch.where(live, fflags & 2, torch.zeros_like(fflags))
        return fflags

    def push(self, frames: torch.Tensor, want_spikes_in: bool = False, want_raster: bool = False,
             peak_win: int = 0) -> Dict[str, object]:
        """One frame per slot in, the samples that became final out: n_out (numpy int64 [S]), counts [S, N] (zero
        where n_out == 0), doa / doa_peak [S] (-1 where n_out == 0), rate [S, G], periodic_ml / trimmed_periodic_ml
        [S] (with a doa_list; NaN where n_out == 0), flags [S] (bit 0: the slot's results are not guaranteed to be the
        clip's bits since its reset; bit 1: the trimmed estimator's IndexError, estimate NaN), spikes_in [S, n + D,
        N_in] / raster [S, n + D, N] on request (slot s fills its first n_out[s] rows).  No host synchronisation
        beyond the row counts."""
        frames, dt = _check_frames(frames, self.M, self.device, self.num_streams)
        S, n, ch = frames.shape
        out = self._outputs(n + self.latency, want_spikes_in, want_raster, peak_win)
        n_out = np.zeros(S, dtype=np.int64)
        N.check(self._lib.micloc_xylo_streams_push(
            self._h, _ptr(frames), dt, n, ch, _ptr(out["spikes_in"]), _ptr(out["raster"]), _ptr(out["counts"]),
            _ptr(out["doa"]), _ptr(out["doa_peak"]), int(peak_win), _ptr(out["flags"]), n_out.ctypes.data_as(C.c_void_p),
            _stream_ptr(self.device)))
        out["flags"] = out["flags"] | self._estimators(out, n_out)
        out["n_out"] = n_out
        return out

    def flush(self, slots=None, want_spikes_in: bool = False, want_raster: bool = False,
              peak_win: int = 0) -> Dict[str, object]:
        """End of the listed recordings (None: all): their remaining samples as in `push` (rows: max_frame_len +
        latency).  'flags' is numpy int32 [S] on the host: bit 0 as in push, bit 1 the trimmed estimator's IndexError
        on the flushed samples."""
        arr, p, ns = self._slots(slots)
        out = self._outputs(self.max_frame_len + self.latency, want_spikes_in, want_raster, peak_win)
        n_out = np.zeros(self.num_streams, dtype=np.int64)
        flags = np.zeros(self.num_streams, dtype=np.int32)
        N.check(self._lib.micloc_xylo_streams_flush(
            self._h, p, ns, _ptr(out["spikes_in"]), _ptr(out["raster"]), _ptr(out["counts"]), _ptr(out["doa"]),
            _ptr(out["doa_peak"]), int(peak_win), _ptr(out["flags"]), n_out.ctypes.data_as(C.c_void_p),
            flags.ctypes.data_as(C.c_void_p), _stream_ptr(self.device)))
        fflags = self._estimators(out, n_out).cpu().numpy()
        out.update({"n_out": n_out, "flags": flags | fflags})
        return out


class Demo:
    """Same constructor and processing methods as the reference's `Demo`
    (micloc/xylo_snn_localization.py:74-444); `localize` is the batched call."""

    def __init__(self, geometry: ArrayGeometry, freq_bands: np.ndarray, doa_list: np.ndarray,
                 recording_duration: float = 0.25, kernel_duration: float = 10e-3, bipolar_spikes: bool = True,
                 xylosim_version: bool = True, fs: float = 48_000, device: int = 0, bf_mats=None,
                 exact: bool = True, filter_order: int = 1):
        self.freq_bands = np.asarray(freq_bands, dtype=np.float64)
        if self.freq_bands.ndim == 1:
            self.freq_bands = self.freq_bands.reshape(1, -1)
        self.beamfs: List[SNNBeamformer] = []
        self.bf_mats = []
        self.tau_vecs = []
        for i, freq_range in enumerate(self.freq_bands):
            freq_mid = np.mean(freq_range)
            tau_mem = 1 / (2 * np.pi * freq_mid)
            tau_vec = [tau_mem, tau_mem]
            self.tau_vecs.append(tau_vec)
            beamf = SNNBeamformer(geometry=geometry, kernel_duration=kernel_duration, freq_range=freq_range,
                                  tau_vec=tau_vec, bipolar_spikes=bipolar_spikes, fs=fs, device=device)
            self.beamfs.append(beamf)
            if bf_mats is not None:
                self.bf_mats.append(np.asarray(bf_mats[i], dtype=np.float64))
            else:
                time_temp = np.arange(0, recording_duration, step=1 / fs)
                sig_temp = np.sin(2 * np.pi * freq_mid * time_temp)
                self.bf_mats.append(beamf.design_from_template(template=(time_temp, sig_temp), doa_list=doa_list))
        self.tau_vecs = np.asarray(self.tau_vecs)
        self.filterbank = ButterworthFilterbank(freq_bands=self.freq_bands, order=filter_order, fs=fs)
        self.doa_list = np.asarray(doa_list)
        self.recording_duration = recording_duration
        self.kernel_duration = kernel_duration
        self.bipolar_spikes = bipolar_spikes
        self.xylosim_version = xylosim_version
        self.fs = fs
        self.dt = 1.0 / fs
        self.exact = exact
        self.geometry = geometry
        self._device = device
        self._initialize_snn_module(target_dt=1e-3)

    def _initialize_snn_module(self, target_dt: float):
        self.net = quantize_network(self.bf_mats, self.tau_vecs, self.fs, self.bipolar_spikes, target_dt)
        enc = self.beamfs[0].spk_encoder
        self.engine = XyloEngine(num_mic=len(self.geometry), stht_kernel=self.beamfs[0].kernel,
                                 sos_list=self.filterbank.sos_list, ba_list=self.filterbank.ba_list,
                                 robust_width=max(int(np.ceil(enc.robust_width)), 1), bipolar=self.bipolar_spikes,
                                 net=self.net, num_doa=len(self.doa_list), device=self._device)

    # ------------------------------------------------------------------
    def _audio_tensor(self, sig_in: np.ndarray) -> torch.Tensor:
        sig = np.asarray(sig_in)
        if sig.dtype == np.int16:
            t = torch.from_numpy(np.ascontiguousarray(sig))
        else:
            s32 = np.ascontiguousarray(sig, dtype=np.float32)
            if self.exact and sig.dtype == np.float64 and not np.array_equal(s32.astype(np.float64), sig):
                raise ValueError("exact mode takes float32-representable (or int16) audio: the device input is float32")
            t = torch.from_numpy(s32)
        return t.to(self.engine.device)

    def spike_encoding(self, sig_in: np.ndarray) -> np.ndarray:
        """`T x N_in` int64 spikes in {0,1} (micloc/xylo_snn_localization.py:315-356)."""
        out = self.engine.run(self._audio_tensor(sig_in), exact=self.exact, want_spikes_in=True)
        return out["spikes_in"][0].cpu().numpy().astype(np.int64)

    def xylo_process(self, spikes_in: np.ndarray) -> np.ndarray:
        """`T x N` hidden-layer spike raster = rec["Spikes"] (micloc/xylo_snn_localization.py:358-377)."""
        s = torch.from_numpy(np.ascontiguousarray(spikes_in, dtype=np.int8)).to(self.engine.device)
        out = self.engine.process(s, want_raster=True)
        return out["raster"][0].cpu().numpy().astype(np.int64)

    def extract_rate(self, spikes_in: np.ndarray) -> np.ndarray:
        """micloc/xylo_snn_localization.py:379-398."""
        rate_channels = np.mean(spikes_in, axis=0) * self.fs
        return rate_channels.reshape(-1, len(self.doa_list)).mean(0)

    def estimate_doa_from_rate(self, spike_rate: np.ndarray, method: str) -> float:
        """micloc/xylo_snn_localization.py:400-444."""
        method_list = ["peak", "periodic_ml", "trimmed_periodic_ml"]
        if method not in method_list:
            raise ValueError(f"only the following estimation methods are supported:\n{method_list}")
        if method == "peak":
            return self.doa_list[np.argmax(spike_rate)]
        if method == "periodic_ml":
            return np.angle(np.mean(spike_rate * np.exp(1j * self.doa_list)))
        DoA_index = np.argmax(spike_rate)
        num_DoA = len(self.doa_list) // 2
        DoA_range = np.arange(-num_DoA // 2, num_DoA // 2 + 1) - DoA_index
        return np.angle(np.mean(spike_rate[DoA_range] * np.exp(1j * self.doa_list[DoA_range])))

    def stream_batch(self, num_streams: int, max_frame_len: int) -> XyloStreamBatch:
        """`num_streams` continuous recordings through this network's exact chain, one push per frame tick."""
        return XyloStreamBatch(self.engine, num_streams, max_frame_len, fs=self.fs, doa_list=self.doa_list)

    def localize(self, audio: torch.Tensor, peak_win: int = 0, exact: Optional[bool] = None):
        """Batched chain: audio [B,T,M] CUDA tensor -> dict(counts, doa, doa_peak, flags)."""
        return self.engine.run(audio, exact=self.exact if exact is None else exact, peak_win=peak_win)
