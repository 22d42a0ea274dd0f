"""Multi-band SNN localiser: the arithmetic of micloc/localization_demo_snn.py's `Demo` on the GPU.

Same constructor as the reference class (micloc/localization_demo_snn.py:22-98).  The reference's `run()` is an endless
record -> process -> plot loop around a `sox` recorder and a matplotlib visualiser (both out of scope); `process_frame`
is the body of that loop (localization_demo_snn.py:134-193): int32 `T x 8` wav frame in, DoA in degrees (or NaN when
the activity detector finds no signal) out.  `localize` is the batched form: frames [B, T, channels] in one go.

Per frame: filterbank on the raw integers (micloc_filterbank), one fused SNN chain per band (micloc_snn_run on that
band's rows), power summed over the bands + argmax + the periodic-ML estimators (micloc_power_fuse).

`stream_batch` makes the same localiser continuous over many arrays at once: a `MultibandStreamBatch` carries the
filterbank, band chains and power fusion of S recordings across pushes (micloc_snn_mb_streams_*).
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence

import numpy as np
import torch

from . import _native as N
from .array_geometry import ArrayGeometry
from .engine import SnnEngine, _SlotBatch, _activity, _check_frames, _ptr, _stream_ptr
from .filterbank import ButterworthFilterbank
from .snn_beamformer import SNNBeamformer


class Demo:
    def __init__(self, geometry: ArrayGeometry, freq_bands: np.ndarray, doa_list: np.ndarray, recording_duration: float,
                 kernel_duration: float, bipolar_spikes: bool, fs: float, device: int = 0,
                 bf_mats: Optional[Sequence[np.ndarray]] = None):
        """`bf_mats` (optional) skips the design step with matrices designed earlier (e.g. by the reference)."""
        freq_bands = np.asarray(freq_bands, dtype=np.float64)
        if freq_bands.ndim == 1:
            freq_bands = freq_bands.reshape(1, -1)
        self.beamfs, self.bf_mats = [], []
        time_temp = np.arange(0, recording_duration, step=1 / fs)
        for i, freq_range in enumerate(freq_bands):
            freq_mid = np.mean(freq_range)
            tau_mem = 1 / (2 * np.pi * freq_mid)                   # localization_demo_snn.py:62-65
            beamf = SNNBeamformer(geometry=geometry, kernel_duration=kernel_duration, freq_range=freq_range,
                                  tau_vec=[tau_mem, tau_mem], bipolar_spikes=bipolar_spikes, fs=fs, device=device)
            beamf.verbose = False
            self.beamfs.append(beamf)
            if bf_mats is not None:
                self.bf_mats.append(np.asarray(bf_mats[i], dtype=np.float64))
            else:
                sig_temp = np.sin(2 * np.pi * freq_mid * time_temp)
                self.bf_mats.append(beamf.design_from_template(template=(time_temp, sig_temp), doa_list=doa_list))
        self.filterbank = ButterworthFilterbank(freq_bands=freq_bands, order=1, fs=fs)
        self.doa_list = np.asarray(doa_list, dtype=np.float64)
        self.recording_duration = recording_duration
        self.kernel_duration = kernel_duration
        self.fs = fs
        self.device = torch.device("cuda", device)
        self.num_mic = len(geometry)
        self._doa_dev = None

    # ------------------------------------------------------------------
    def localize(self, frames: torch.Tensor, rel_threshold: float = 0.0001, full_scale: Optional[float] = None,
                 want_spikes: bool = False) -> Dict[str, torch.Tensor]:
        """frames [B, T, channels >= num_mic] (CUDA, int32 / int16 / float32; extra channels are dropped like the
        reference's `data[:, :-1]`) -> dict(power_grid [B, G], doa [B] index of the peak, doa_deg [B] (NaN = no
        activity), periodic_ml / trimmed_periodic_ml [B] radians, active [B] bool, power [F, B, G], flags [B])."""
        if frames.dim() == 2:
            frames = frames.unsqueeze(0)
        frames, dt = _check_frames(frames, self.num_mic, self.device, frames.shape[0])
        B, T, ch = frames.shape
        F, M, G = len(self.beamfs), self.num_mic, len(self.doa_list)
        lib = N.lib()
        dev = self.device
        st = _stream_ptr(dev)
        sos = np.ascontiguousarray(self.filterbank.sos_list, dtype=np.float64)          # [F][nsec][6]
        banded = torch.empty((F, B, T, M), dtype=torch.float32, device=dev)
        sumsq = torch.empty(B, dtype=torch.float64, device=dev)
        N.check(lib.micloc_filterbank(_ptr(frames), dt, B, T, ch, M, F, sos.shape[1], sos.ctypes.data_as(N._dp),
                                      _ptr(banded), _ptr(sumsq), dev.index or 0, st))
        time_vec = np.arange(0, T) / self.fs
        power = torch.empty((F, B, G), dtype=torch.float32, device=dev)
        flags = torch.zeros(B, dtype=torch.int32, device=dev)
        spikes = []
        for f, (beamf, bf) in enumerate(zip(self.beamfs, self.bf_mats)):
            eng = beamf.engine(bf, time_vec)
            out = eng.run(banded[f], want_spikes=want_spikes, want_power=True, fused=True)
            spikes.append(out["spikes"])
            power[f].copy_(out["power"])
            flags |= out["flags"]
        if self._doa_dev is None:
            self._doa_dev = torch.from_numpy(self.doa_list).to(dev)
        power_grid = torch.empty((B, G), dtype=torch.float32, device=dev)
        doa = torch.empty(B, dtype=torch.int32, device=dev)
        ml = torch.empty(B, dtype=torch.float64, device=dev)
        trimmed = torch.empty(B, dtype=torch.float64, device=dev)
        fflags = torch.empty(B, dtype=torch.int32, device=dev)
        N.check(lib.micloc_power_fuse(_ptr(power), F, B, G, _ptr(self._doa_dev), _ptr(power_grid), _ptr(doa), _ptr(ml),
                                      _ptr(trimmed), _ptr(fflags), dev.index or 0, st))
        active, doa_deg = _activity(sumsq, T, M, frames.dtype, rel_threshold, full_scale, doa, self._doa_dev)
        return {"power_grid": power_grid, "doa": doa, "doa_deg": doa_deg, "periodic_ml": ml, "trimmed_periodic_ml": trimmed,
                "active": active, "power": power, "flags": flags | fflags, "spikes": spikes if want_spikes else None,
                "banded": banded}

    def stream_batch(self, num_streams: int, max_frame_len: int) -> "MultibandStreamBatch":
        """`num_streams` continuous recordings through this localiser, one push per frame tick."""
        return MultibandStreamBatch(self, num_streams, max_frame_len)

    def process_frame(self, data: np.ndarray) -> float:
        """One recording as the reference's loop handles it: `T x 8` integer wav frame -> DoA in degrees, NaN when no
        activity was detected (what the loop pushes to its visualiser)."""
        data = np.asarray(data)
        out = self.localize(torch.from_numpy(np.ascontiguousarray(data)).to(self.device))
        return float(out["doa_deg"][0])

    def run(self, frames=None):
        """The reference records from the devkit forever; here `frames` is any iterable of wav frames."""
        if frames is None:
            raise NotImplementedError("the recorder / visualiser loop is out of scope: pass an iterable of wav frames")
        for data in frames:
            yield self.process_frame(data)


class MultibandStreamBatch(_SlotBatch):
    """`num_streams` independent recordings ("slots") through the multi-band localiser with its state carried across
    pushes (micloc_snn_mb_streams_*).  N pushed frames give, for every band, what the filterbank of their
    concatenation followed by that band's stream gives (see engine.SnnStreamBatch); every band finalises the same
    samples, `latency` = max over the bands of their RZCC lag behind the input.  reset / flush take slot lists as in
    SnnStreamBatch.  Frames are [num_streams, n, channels] device tensors, int32 / int16 / float32 (channels beyond the
    microphones are dropped).

    The batch owns its band engines (neuron normalisation of a `recording_duration` frame, as `Demo.localize` uses for
    a frame of that length): engines of SNNBeamformer's cache may be closed by its eviction while the batch lives."""

    def __init__(self, demo: Demo, num_streams: int, max_frame_len: int):
        self.demo = demo
        self.time_vec = np.arange(int(round(demo.recording_duration * demo.fs))) / demo.fs
        self.engines = [SnnEngine(beamf.chain_spec(self.time_vec), bf, device=demo.device.index or 0)
                        for beamf, bf in zip(demo.beamfs, demo.bf_mats)]
        self.F, self.M, self.G = len(self.engines), demo.num_mic, len(demo.doa_list)
        self.C2 = 2 * self.M
        lib = N.lib()
        sos = np.ascontiguousarray(demo.filterbank.sos_list, dtype=np.float64)           # [F][nsec][6]
        ctxs = (C.c_void_p * self.F)(*[e._h.value for e in self.engines])
        h = C.c_void_p()
        N.check(lib.micloc_snn_mb_streams_create(ctxs, self.F, sos.shape[1], sos.ctypes.data_as(N._dp),
                                                 demo.doa_list.ctypes.data_as(N._dp), int(num_streams),
                                                 int(max_frame_len), C.byref(h)))
        self._attach(lib, h, "micloc_snn_mb_streams", int(num_streams), int(max_frame_len), demo.device)
        self._doa_dev = torch.from_numpy(demo.doa_list).to(self.device)

    def _outputs(self, rows, want_spikes):
        S, dev = self.num_streams, self.device
        return {"spikes": torch.empty((self.F, S, rows, self.C2), dtype=torch.int8, device=dev) if want_spikes else None,
                "power": torch.empty((self.F, S, self.G), dtype=torch.float32, device=dev),
                "power_grid": torch.empty((S, self.G), dtype=torch.float32, device=dev),
                "doa": torch.full((S,), -1, dtype=torch.int32, device=dev),     # -1: not written (n_out == 0)
                "periodic_ml": torch.empty(S, dtype=torch.float64, device=dev),
                "trimmed_periodic_ml": torch.empty(S, dtype=torch.float64, device=dev),
                "flags": torch.empty(S, dtype=torch.int32, device=dev)}

    def push(self, frames: torch.Tensor, want_spikes: bool = False, rel_threshold: float = 0.0001,
             full_scale: Optional[float] = None) -> Dict[str, object]:
        """One frame per slot in, the samples that became final out, with `Demo.localize`'s keys: n_out (numpy int64
        [S]), power [F, S, G] and power_grid [S, G] over each slot's final samples, doa [S], periodic_ml /
        trimmed_periodic_ml [S], flags [S] (bit 0 RZCC overflow so far, bit 1 the trimmed estimator's IndexError),
        spikes [F, S, n + D, 2M] when `want_spikes`; these are NOT written for a slot with n_out == 0 (its doa stays
        -1).  active [S] and doa_deg [S] as in `localize`, the gate on the rms of the frame just pushed (D samples
        ahead of the power window); doa_deg is NaN where inactive or where n_out == 0.  sumsq [S] float64 of the
        frame.  No host synchronisation."""
        frames, dt = _check_frames(frames, self.M, self.device, self.num_streams)
        S, n, ch = frames.shape
        out = self._outputs(n + self.latency, want_spikes)
        sumsq = torch.empty(S, dtype=torch.float64, device=self.device)
        n_out = np.zeros(S, dtype=np.int64)
        N.check(self._lib.micloc_snn_mb_streams_push(
            self._h, _ptr(frames), dt, n, ch, _ptr(out["spikes"]), _ptr(out["power"]), _ptr(out["power_grid"]),
            _ptr(out["doa"]), _ptr(out["periodic_ml"]), _ptr(out["trimmed_periodic_ml"]), _ptr(sumsq), _ptr(out["flags"]),
            n_out.ctypes.data_as(C.c_void_p), _stream_ptr(self.device)))
        active, doa_deg = _activity(sumsq, n, self.M, frames.dtype, rel_threshold, full_scale, out["doa"], self._doa_dev,
                                    written=out["doa"] >= 0)         # (n_out > 0 without a host-to-device copy)
        out.update({"n_out": n_out, "active": active, "sumsq": sumsq, "doa_deg": doa_deg})
        if not want_spikes:
            del out["spikes"]
        return out

    def flush(self, slots=None, want_spikes: bool = False) -> Dict[str, object]:
        """End of the listed recordings (None: all): their remaining samples as in `push` (rows: max_frame_len +
        latency), without the activity gate (no new frame).  'flags' is numpy int32 [S] on the host: bit 0 = RZCC
        overflow anywhere in that slot's recording, any band; bit 1 = the trimmed estimator's IndexError on the
        flushed samples."""
        arr, p, ns = self._slots(slots)
        out = self._outputs(self.max_frame_len + self.latency, want_spikes)
        n_out = np.zeros(self.num_streams, dtype=np.int64)
        flags = np.zeros(self.num_streams, dtype=np.int32)
        N.check(self._lib.micloc_snn_mb_streams_flush(
            self._h, p, ns, _ptr(out["spikes"]), _ptr(out["power"]), _ptr(out["power_grid"]), _ptr(out["doa"]),
            _ptr(out["periodic_ml"]), _ptr(out["trimmed_periodic_ml"]), _ptr(out["flags"]),
            n_out.ctypes.data_as(C.c_void_p), flags.ctypes.data_as(C.c_void_p), _stream_ptr(self.device)))
        fused = out["flags"].cpu().numpy()
        flags |= np.where(n_out > 0, fused & 2, 0).astype(np.int32)
        out.update({"n_out": n_out, "flags": flags})
        if not want_spikes:
            del out["spikes"]
        return out
