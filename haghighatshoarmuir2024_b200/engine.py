"""Batched device engine over the C-ABI: the call a Monte-Carlo driver makes.

`SnnEngine` owns one `micloc_snn` context on one GPU.  torch is used only for
device memory and streams; all arithmetic happens in libmicloc_b200.so.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, Optional, Sequence

import numpy as np
import torch

from . import _native as N


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream_ptr(device: torch.device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _check_frames(frames: torch.Tensor, M: int, device: torch.device, num_streams: Optional[int] = None):
    """The frames of a stream push: [n, channels] (num_streams None) or [num_streams, n, channels], channels >= M, on
    `device`, float32 / int16 / int32 -> (contiguous frames, dtype code)."""
    if frames.dim() != (2 if num_streams is None else 3) or frames.shape[-1] < M:
        raise ValueError(
            f"number of channels in the input siganl {frames.shape[-1]} should be the same as the number of microphones {M}!")
    if num_streams is not None and frames.shape[0] != num_streams:
        raise ValueError(f"frames hold {frames.shape[0]} slots, the batch has {num_streams}")
    if frames.device != device:
        raise ValueError(f"frames live on {frames.device}, not on {device}")
    dt = {torch.float32: N.F32, torch.int16: N.I16, torch.int32: N.I32}.get(frames.dtype)
    if dt is None:
        raise ValueError(f"frames must be float32, int16 or int32, got {frames.dtype}")
    return frames.contiguous(), dt


def _activity(sumsq: torch.Tensor, rows: int, M: int, dtype: torch.dtype, rel_threshold: float,
              full_scale: Optional[float], doa=None, doa_list=None, written=None):
    """The activity gate of micloc/localization_demo_snn.py:136-163 -> (active, doa_deg): active = the frame's rms (sumsq
    over `rows` samples of M microphones) >= rel_threshold * full_scale (None: an integer `dtype`'s largest value, 1.0
    for float32); doa_deg = doa_list[doa] in degrees, NaN where inactive or not `written`; None without doa_list."""
    if full_scale is None:
        full_scale = float(torch.iinfo(dtype).max) if not dtype.is_floating_point else 1.0
    active = torch.sqrt(sumsq / (rows * M)) >= rel_threshold * full_scale
    if doa is None or doa_list is None:
        return active, None
    keep, doa = (active, doa) if written is None else (written & active, torch.where(written, doa, 0))
    deg = doa_list[doa.long()] * 180 / np.pi
    return active, torch.where(keep, deg, torch.full_like(deg, float("nan")))


def _design_template(geometry, time: np.ndarray, sig: np.ndarray, device: torch.device):
    """micloc_design_template of (geometry, template on the fs grid) -> (struct, the arrays it points at)."""
    r = np.ascontiguousarray(geometry.r_vec, dtype=np.float64)
    th = np.ascontiguousarray(geometry.theta_vec, dtype=np.float64)
    t_d, s_d = _dev64(time, device), _dev64(sig, device)
    if t_d.dim() != 1 or s_d.shape != t_d.shape:
        raise ValueError(f"template time and signal must be 1-D of one length; got {tuple(t_d.shape)}, {tuple(s_d.shape)}")
    tp = N.DesignTemplate()
    tp.num_mic = len(r)
    tp.r_vec = r.ctypes.data_as(N._dp)
    tp.theta_vec = th.ctypes.data_as(N._dp)
    tp.speed = float(geometry.speed)
    tp.T = len(t_d)
    tp.time_dev = _ptr(t_d)
    tp.sig_dev = _ptr(s_d)
    return tp, (r, th, t_d, s_d)


def _dev64(x, device: torch.device) -> torch.Tensor:
    """float64 contiguous on `device`; a tensor already there is not copied."""
    if not isinstance(x, torch.Tensor):
        x = torch.as_tensor(np.asarray(x, dtype=np.float64))
    return x.to(device=device, dtype=torch.float64).contiguous()


def _doa_tensor(doa, device: torch.device) -> torch.Tensor:
    return _dev64(doa, device).reshape(-1)


def design_vectors(mode: int, cov: torch.Tensor, want_value: bool = False):
    """The batched float64 design solver alone (micloc_design_vectors) on device covariances: cov [G, 2M, 2M] float64
    (modes 0 SNN unipolar, 1 SNN bipolar) or [G, M, M] complex128 (modes 2 Hilbert, 3 Hilbert with interference
    removal) -> bf ([2M, G] float64 for modes 0 / 1, [M, G] complex128 for 2 / 3) and, with want_value, value [G]."""
    cov = cov.contiguous()
    G = cov.shape[0]
    if cov.is_complex():
        M = cov.shape[1]
        raw = torch.view_as_real(cov)
    else:
        M = cov.shape[1] // 2
        raw = cov
    dev = cov.device
    complex_out = mode in (2, 3)
    bf = torch.empty((M, G, 2) if complex_out else (2 * M, G), dtype=torch.float64, device=dev)
    value = torch.empty(G, dtype=torch.float64, device=dev) if want_value else None
    N.check(N.lib().micloc_design_vectors(int(mode), _ptr(raw), M, G, _ptr(bf), _ptr(value), dev.index,
                                          _stream_ptr(dev)))
    if complex_out:
        bf = torch.view_as_complex(bf)
    return (bf, value) if want_value else bf


class _SlotBatch:
    """What the stream batches share: the native batch `_h` of `num_streams` slots on `device`, whose C functions are
    named `<api>_reset`, `<api>_latency` and `<api>_destroy`, and its slot lists.  A subclass creates the handle and
    hands it to `_attach`."""

    def _attach(self, lib, h, api: str, num_streams: int, max_frame_len: int, device: torch.device):
        self._lib, self._h, self._api = lib, h, api
        self.num_streams, self.max_frame_len, self.device = num_streams, max_frame_len, device
        self.latency = int(getattr(lib, api + "_latency")(h))

    def close(self):
        if getattr(self, "_h", None):
            getattr(self._lib, self._api + "_destroy")(self._h)
            self._h = None

    __del__ = close

    @staticmethod
    def _slots(slots):
        if slots is None:
            return None, None, 0
        arr = np.ascontiguousarray(np.atleast_1d(np.asarray(slots)), dtype=np.int32)
        return arr, arr.ctypes.data_as(C.c_void_p), len(arr)

    def reset(self, slots=None):
        """Fresh state for the listed slots (None: all); they restart at sample 0."""
        arr, p, n = self._slots(slots)
        N.check(getattr(self._lib, self._api + "_reset")(self._h, p, n, _stream_ptr(self.device)))


@dataclass
class ChainSpec:
    """Host constants of one SNN chain (what SNNBeamformer derives, snn_beamformer.py:45-80,342-361)."""
    num_mic: int
    stht_kernel: np.ndarray      # [K] float64
    sos: np.ndarray              # [n_sections, 6]
    robust_width: int
    bipolar: bool
    neuron_decay: float
    neuron_scale: float
    neuron_len: int


def neuron_alpha_params(time_vec: np.ndarray, tau_vec: Sequence[float]):
    """Truncated, normalised alpha kernel of snn_beamformer.py:342-361 as (taps, a, c, L).

    h[n] = (t_n/tau) exp(-t_n/tau) / sum_T(...), cut where the cumulative mass reaches
    0.999.  Returned closed form: h[n] = c * n * a^n for n < L."""
    tau_syn, tau_mem = float(tau_vec[0]), float(tau_vec[1])
    tn = np.asarray(time_vec, dtype=np.float64) - time_vec[0]
    if tau_mem != tau_syn:
        # The reference's kernel for unequal time constants, (exp(-t/tau_syn) - exp(+t/tau_mem)) / (1/tau_mem - 1/tau_syn)
        # (snn_beamformer.py:349-353), grows without bound and trips its own `assert np.all(h >= 0)`; the device
        # recurrence implements the alpha kernel c n a^n of the tau_syn == tau_mem branch only.
        raise ValueError("tau_syn != tau_mem is not supported: the device neuron filter is the alpha kernel of "
                         "tau_syn == tau_mem (the reference's unequal-tau kernel fails its own assertion)")
    h = (tn / tau_syn) * np.exp(-tn / tau_syn)
    total = np.sum(h)
    h = h / total
    L = int(np.sum(np.cumsum(h) < 0.999))
    dt = float(tn[1] - tn[0]) if len(tn) > 1 else 1.0
    a = float(np.exp(-dt / tau_syn))
    c = float((dt / tau_syn) / total)
    return h[:L], a, c, max(L, 1)


class SnnEngine:
    def __init__(self, spec: ChainSpec, bf_mat: np.ndarray, device: int = 0):
        if not torch.cuda.is_available():
            raise RuntimeError("SnnEngine needs a CUDA device (B200); there is no CPU fallback")
        self.spec = spec
        self.device = torch.device("cuda", device)
        self._lib = N.lib()
        bf = np.ascontiguousarray(bf_mat, dtype=np.float64)
        if bf.ndim != 2 or bf.shape[0] != 2 * spec.num_mic:
            raise ValueError(f"bf_mat should have shape (2*num_mic, num_DoA); got {bf.shape}")
        self._kernel = np.ascontiguousarray(spec.stht_kernel, dtype=np.float64)
        self._sos = np.ascontiguousarray(spec.sos, dtype=np.float64).reshape(-1, 6)
        cfg = N.SnnConfig()
        cfg.num_mic = spec.num_mic
        cfg.kernel_len = len(self._kernel)
        cfg.stht_kernel = self._kernel.ctypes.data_as(N._dp)
        cfg.n_sections = self._sos.shape[0]
        cfg.sos = self._sos.ctypes.data_as(N._dp)
        cfg.robust_width = int(spec.robust_width)
        cfg.bipolar = int(bool(spec.bipolar))
        cfg.neuron_decay = float(spec.neuron_decay)
        cfg.neuron_scale = float(spec.neuron_scale)
        cfg.neuron_len = int(spec.neuron_len)
        cfg.num_doa = bf.shape[1]
        cfg.bf_mat = bf.ctypes.data_as(N._dp)
        h = C.c_void_p()
        N.check(self._lib.micloc_snn_create(C.byref(cfg), device, C.byref(h)))
        self._h = h
        self.M, self.C2, self.G = spec.num_mic, 2 * spec.num_mic, bf.shape[1]
        self._fused_unsupported = False

    def close(self):
        if getattr(self, "_h", None):
            self._lib.micloc_snn_destroy(self._h)
            self._h = None

    __del__ = close

    def set_bf(self, bf_mat: np.ndarray):
        bf = np.ascontiguousarray(bf_mat, dtype=np.float64)
        if bf.ndim != 2 or bf.shape[0] != self.C2:
            raise ValueError(f"bf_mat should have shape (2*num_mic, num_DoA); got {bf.shape}")
        N.check(self._lib.micloc_snn_set_bf(self._h, bf.ctypes.data_as(N._dp), bf.shape[1]))
        self.G = bf.shape[1]

    # ------------------------------------------------------------------
    def _check_audio(self, audio: torch.Tensor, check_device: bool = True):
        if audio.dim() == 2:
            audio = audio.unsqueeze(0)
        if audio.dim() != 3 or audio.shape[2] != self.M:
            raise ValueError(
                f"number of channels in the input siganl {audio.shape[-1]} should be the same as the number of microphones {self.M}!")
        if audio.dtype == torch.float32:
            dt = N.F32
        elif audio.dtype == torch.int16:
            dt = N.I16
        else:
            raise ValueError(f"audio must be float32 or int16, got {audio.dtype}")
        if check_device and audio.device != self.device:
            raise ValueError(f"audio lives on {audio.device}, engine on {self.device}")
        return audio.contiguous(), dt

    def run(self, audio: torch.Tensor, want_spikes: bool = False, want_power: bool = True,
            fused: bool = True, refine: bool = True) -> Dict[str, torch.Tensor]:
        """audio [B,T,M] on this engine's GPU -> {'doa','power','spikes','flags'} (device tensors).

        The fused kernel reports clips whose RZCC clusters overflowed its bounded streaming encoder in `flags` bit 0;
        with `refine` (default) they are redone by the library with the unbounded encoder before this returns, which
        synchronises the stream.  Pipelined callers pass refine=False and call `refine(audio, out)` once per step."""
        audio, dt = self._check_audio(audio)
        B, T, _ = audio.shape
        dev = self.device
        doa = torch.empty(B, dtype=torch.int32, device=dev)
        flags = torch.empty(B, dtype=torch.int32, device=dev)
        power = torch.empty((B, self.G), dtype=torch.float32, device=dev) if want_power else None
        spikes = torch.empty((B, T, self.C2), dtype=torch.int8, device=dev) if want_spikes else None
        fused = bool(fused) and not self._fused_unsupported
        rc = self._lib.micloc_snn_run(self._h, _ptr(audio), dt, B, T, _ptr(spikes), _ptr(power), _ptr(doa),
                                      _ptr(flags), int(fused), _stream_ptr(dev))
        if rc == N.ERR_UNSUPPORTED and fused:
            # geometries the fused kernels do not cover (more than 8 microphones, dense STHT kernels, ...) take the
            # tiled / staged kernels; remembered per engine
            self._fused_unsupported = True
            rc = self._lib.micloc_snn_run(self._h, _ptr(audio), dt, B, T, _ptr(spikes), _ptr(power), _ptr(doa),
                                          _ptr(flags), 0, _stream_ptr(dev))
        N.check(rc)
        out = {"doa": doa, "power": power, "spikes": spikes, "flags": flags}
        if refine and fused:
            self.refine(audio, out)
        return out

    def refine(self, audio: torch.Tensor, out: Dict[str, torch.Tensor]) -> int:
        """micloc_snn_refine on the outputs of a fused `run`: number of clips redone (0 almost always)."""
        audio, dt = self._check_audio(audio)
        B, T, _ = audio.shape
        n = C.c_int64()
        N.check(self._lib.micloc_snn_refine(self._h, _ptr(audio), dt, B, T, _ptr(out.get("spikes")), _ptr(out.get("power")),
                                            _ptr(out.get("doa")), _ptr(out["flags"]), C.byref(n), _stream_ptr(self.device)))
        return n.value

    @property
    def refined_count(self) -> int:
        return int(self._lib.micloc_snn_refined_count(self._h))

    def run_taps(self, audio: torch.Tensor, want: Sequence[str] = ("q", "z", "spikes", "vmem", "y", "power", "doa")):
        """Staged path with per-stage taps (device tensors)."""
        audio, dt = self._check_audio(audio)
        B, T, _ = audio.shape
        dev = self.device
        mk = lambda name, shape, dtype: torch.empty(shape, dtype=dtype, device=dev) if name in want else None
        out = {
            "q": mk("q", (B, T, self.M), torch.float32),
            "z": mk("z", (B, T, self.C2), torch.float32),
            "spikes": mk("spikes", (B, T, self.C2), torch.int8),
            "vmem": mk("vmem", (B, T, self.C2), torch.float32),
            "y": mk("y", (B, T, self.G), torch.float32),
            "power": mk("power", (B, self.G), torch.float32),
            "doa": mk("doa", (B,), torch.int32),
            "flags": torch.empty(B, dtype=torch.int32, device=dev),
        }
        N.check(self._lib.micloc_snn_run_taps(
            self._h, _ptr(audio), dt, B, T, _ptr(out["q"]), _ptr(out["z"]), _ptr(out["spikes"]), _ptr(out["vmem"]),
            _ptr(out["y"]), _ptr(out["power"]), _ptr(out["doa"]), _ptr(out["flags"]), _stream_ptr(dev)))
        return out

    def gram(self, audio: torch.Tensor, t_start: int) -> torch.Tensor:
        """sum_{t>=t_start} v v^T per clip, float64 [B,2M,2M] (design-time covariance)."""
        audio, dt = self._check_audio(audio)
        B, T, _ = audio.shape
        g = torch.empty((B, self.C2, self.C2), dtype=torch.float64, device=self.device)
        N.check(self._lib.micloc_snn_gram(self._h, _ptr(audio), dt, B, T, int(t_start), _ptr(g), _stream_ptr(self.device)))
        return g

    def set_hilbert_bf(self, bf_complex: np.ndarray):
        """Steering matrix [M, G] complex of the Hilbert beamformer (`hilbert`); the SNN bf_mat is left as it is."""
        bf = np.asarray(bf_complex)
        if bf.ndim != 2 or bf.shape[0] != self.M:
            raise ValueError(f"bf_mat should have shape (num_mic, num_DoA); got {bf.shape}")
        re = np.ascontiguousarray(bf.real, dtype=np.float64)
        im = np.ascontiguousarray(bf.imag, dtype=np.float64) if np.iscomplexobj(bf) else np.zeros_like(re)
        N.check(self._lib.micloc_hilbert_set_bf(self._h, re.ctypes.data_as(N._dp), im.ctypes.data_as(N._dp),
                                                bf.shape[1]))
        self.hilbert_G = bf.shape[1]

    def hilbert(self, audio: torch.Tensor, t_start: int = 0, bandpass: bool = True,
                want: Sequence[str] = ("doa", "power")) -> Dict[str, torch.Tensor]:
        """Hilbert beamformer on audio [B,T,M] (micloc_hilbert_localize): the analytic signal s_t (band-passed, or
        roll + STHT without `bandpass`) over rows t >= t_start gives any of 'doa' [B] int32, 'power' [B,G] float32
        (mean |s_t . conj(bf_g)|^2), 'cov' [B,M,M] complex128 (sum conj(s_t) s_t^T) and 'z' [B,T,2M] float32 (real |
        imag of s_t), as device tensors; stream-ordered."""
        audio, dt = self._check_audio(audio)
        B, T, _ = audio.shape
        dev = self.device
        G = getattr(self, "hilbert_G", 0)
        mk = lambda name, shape, dtype: torch.empty(shape, dtype=dtype, device=dev) if name in want else None
        out = {"doa": mk("doa", (B,), torch.int32), "power": mk("power", (B, G), torch.float32),
               "cov": mk("cov", (B, self.M, self.M, 2), torch.float64), "z": mk("z", (B, T, self.C2), torch.float32)}
        N.check(self._lib.micloc_hilbert_localize(self._h, _ptr(audio), dt, B, T, int(t_start), int(bool(bandpass)),
                                                  _ptr(out["z"]), _ptr(out["cov"]), _ptr(out["power"]),
                                                  _ptr(out["doa"]), _stream_ptr(dev)))
        if out["cov"] is not None:
            out["cov"] = torch.view_as_complex(out["cov"])
        return {k: v for k, v in out.items() if v is not None}

    # ------------------------------------------------------------------
    def design_templates(self, geometry, time: np.ndarray, sig: np.ndarray, doa) -> torch.Tensor:
        """The template (time, sig) on the fs grid delayed for every DoA: clips [G, T, M] float32 on this GPU
        (micloc_design_templates)."""
        tp, keep = _design_template(geometry, time, sig, self.device)
        doa_d = _doa_tensor(doa, self.device)
        clips = torch.empty((len(doa_d), tp.T, tp.num_mic), dtype=torch.float32, device=self.device)
        N.check(self._lib.micloc_design_templates(C.byref(tp), _ptr(doa_d), len(doa_d), _ptr(clips), self.device.index,
                                                  _stream_ptr(self.device)))
        return clips

    def snn_design(self, geometry, time: np.ndarray, sig: np.ndarray, doa, want_cov: bool = False):
        """SNN design on the device (micloc_snn_design; unipolar or bipolar from this chain): (bf [2M, G] float64,
        cov [G, 2M, 2M] float64 or None), device tensors; this engine's chain must be the one of `time`."""
        tp, keep = _design_template(geometry, time, sig, self.device)
        doa_d = _doa_tensor(doa, self.device)
        G = len(doa_d)
        bf = torch.empty((self.C2, G), dtype=torch.float64, device=self.device)
        cov = torch.empty((G, self.C2, self.C2), dtype=torch.float64, device=self.device) if want_cov else None
        N.check(self._lib.micloc_snn_design(self._h, C.byref(tp), _ptr(doa_d), G, _ptr(bf), _ptr(cov),
                                            _stream_ptr(self.device)))
        return bf, cov

    def hilbert_design(self, geometry, time: np.ndarray, sig: np.ndarray, doa, interference_removal: bool = False):
        """Hilbert design on the device (micloc_hilbert_design): (bf [M, G] complex128, cov [G, M, M] complex128),
        device tensors."""
        tp, keep = _design_template(geometry, time, sig, self.device)
        doa_d = _doa_tensor(doa, self.device)
        G = len(doa_d)
        bf = torch.empty((self.M, G, 2), dtype=torch.float64, device=self.device)
        cov = torch.empty((G, self.M, self.M, 2), dtype=torch.float64, device=self.device)
        N.check(self._lib.micloc_hilbert_design(self._h, C.byref(tp), _ptr(doa_d), G, int(bool(interference_removal)),
                                                _ptr(bf), _ptr(cov), _stream_ptr(self.device)))
        return torch.view_as_complex(bf), torch.view_as_complex(cov)

    def run_host(self, audio, want_spikes: bool = False, want_power: bool = True, fused: bool = True):
        """End-to-end with HOST buffers (numpy or CPU torch tensors, ideally pinned):
        H2D copy, hot path, D2H copy all inside the C call."""
        t = torch.as_tensor(audio)
        if t.is_cuda:
            raise ValueError("run_host takes host memory; use run() for device tensors")
        t, dt = self._check_audio(t, check_device=False)
        B, T, _ = t.shape
        pin = t.is_pinned()
        mk = lambda shape, dtype: torch.empty(shape, dtype=dtype, pin_memory=pin)
        doa = mk((B,), torch.int32)
        flags = mk((B,), torch.int32)
        power = mk((B, self.G), torch.float32) if want_power else None
        spikes = mk((B, T, self.C2), torch.int8) if want_spikes else None
        N.check(self._lib.micloc_snn_run_host(self._h, _ptr(t), dt, B, T, _ptr(spikes), _ptr(power), _ptr(doa),
                                              _ptr(flags), int(fused)))
        return {"doa": doa, "power": power, "spikes": spikes, "flags": flags}

    def enable_timing(self, on: bool = True):
        N.check(self._lib.micloc_snn_enable_timing(self._h, int(on)))

    def last_kernel_ms(self):
        ms = C.c_float()
        n = C.c_int32()
        N.check(self._lib.micloc_snn_last_kernel_ms(self._h, C.byref(ms), C.byref(n)))
        return ms.value, n.value


class SnnStream:
    """Stateful frames of one continuous recording (micloc_snn_stream_*): N pushed frames give what one clip of their
    concatenation gives (STHT history, band-pass, RZCC and neuron state carry over), with the results lagging the
    input by `latency` samples.  The live loop of micloc/localization_demo_snn.py:125-193 restarts from zero state at
    every frame instead.  Frames are [n, channels] device tensors, float32 / int16 / int32 (the recorder's `T x 8`
    wav frames: channels beyond the microphones are dropped, localization_demo_snn.py:145)."""

    def __init__(self, engine: SnnEngine, max_frame_len: int, fs: float = 48_000.0, rise_time: float = 10e-3,
                 fall_time: float = 100e-3):
        self.engine = engine
        self._lib = engine._lib
        self.max_frame_len = int(max_frame_len)
        h = C.c_void_p()
        N.check(self._lib.micloc_snn_stream_create(engine._h, self.max_frame_len, float(fs), float(rise_time),
                                                   float(fall_time), C.byref(h)))
        self._h = h
        self.latency = int(self._lib.micloc_snn_stream_latency(h))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.micloc_snn_stream_destroy(self._h)
            self._h = None

    __del__ = close

    def reset(self):
        N.check(self._lib.micloc_snn_stream_reset(self._h, _stream_ptr(self.engine.device)))

    def _outputs(self, rows, want_env):
        e = self.engine
        dev = e.device
        return {"spikes": torch.empty((rows, e.C2), dtype=torch.int8, device=dev),
                "power": torch.empty(e.G, dtype=torch.float32, device=dev),
                "doa": torch.empty(1, dtype=torch.int32, device=dev),
                "env": torch.empty((rows, e.G), dtype=torch.float32, device=dev) if want_env else None,
                "doa_t": torch.empty(rows, dtype=torch.int32, device=dev) if want_env else None}

    def _trim(self, out, n):
        res = {"n_out": n, "spikes": out["spikes"][:n], "power": out["power"] if n else None,
               "doa": out["doa"] if n else None}
        if out["env"] is not None:
            res["env"], res["doa_t"] = out["env"][:n], out["doa_t"][:n]
        return res

    def push(self, frame: torch.Tensor, want_env: bool = False) -> Dict[str, torch.Tensor]:
        """One frame in, the samples that became final out: dict(n_out, spikes [n_out, 2M], power [G] and doa [1]
        over those samples, env [n_out, G] + doa_t [n_out] when `want_env`)."""
        e = self.engine
        frame, dt = _check_frames(frame, e.M, e.device)
        n = frame.shape[0]
        out = self._outputs(n + self.latency, want_env)
        n_out = C.c_int64()
        N.check(self._lib.micloc_snn_stream_push(self._h, _ptr(frame), dt, n, frame.shape[1], _ptr(out["spikes"]),
                                                 _ptr(out["power"]), _ptr(out["doa"]), _ptr(out["env"]), _ptr(out["doa_t"]),
                                                 C.byref(n_out), _stream_ptr(e.device)))
        return self._trim(out, n_out.value)

    def flush(self, want_env: bool = False) -> Dict[str, torch.Tensor]:
        """End of the recording: the remaining `latency` samples (+ 'flags': RZCC overflow bit of the whole stream)."""
        out = self._outputs(self.max_frame_len + self.latency, want_env)
        n_out, flags = C.c_int64(), C.c_int32()
        N.check(self._lib.micloc_snn_stream_flush(self._h, _ptr(out["spikes"]), _ptr(out["power"]), _ptr(out["doa"]),
                                                  _ptr(out["env"]), _ptr(out["doa_t"]), C.byref(n_out), C.byref(flags),
                                                  _stream_ptr(self.engine.device)))
        res = self._trim(out, n_out.value)
        res["flags"] = flags.value
        return res


class SnnStreamBatch(_SlotBatch):
    """`num_streams` independent recordings ("slots") advanced together (micloc_snn_streams_*): one push hands every
    slot one frame of the same length and runs a fixed number of kernels whatever the number of slots.  Each slot
    behaves as an `SnnStream`; `reset` and `flush` act on a list of slots only, and a flushed slot ignores its rows of
    later pushes (n_out = 0) until it is reset.  Frames are [num_streams, n, channels] device tensors, float32 / int16 /
    int32 (channels beyond the microphones are dropped)."""

    def __init__(self, engine: SnnEngine, num_streams: int, max_frame_len: int, fs: float = 48_000.0,
                 rise_time: float = 10e-3, fall_time: float = 100e-3):
        self.engine = engine
        h = C.c_void_p()
        N.check(engine._lib.micloc_snn_streams_create(engine._h, int(num_streams), int(max_frame_len), float(fs),
                                                      float(rise_time), float(fall_time), C.byref(h)))
        self._attach(engine._lib, h, "micloc_snn_streams", int(num_streams), int(max_frame_len), engine.device)

    def _outputs(self, rows, want_env):
        e, S = self.engine, self.num_streams
        dev = e.device
        return {"spikes": torch.empty((S, rows, e.C2), dtype=torch.int8, device=dev),
                "power": torch.empty((S, e.G), dtype=torch.float32, device=dev),
                "doa": torch.empty(S, dtype=torch.int32, device=dev),
                "env": torch.empty((S, rows, e.G), dtype=torch.float32, device=dev) if want_env else None,
                "doa_t": torch.empty((S, rows), dtype=torch.int32, device=dev) if want_env else None}

    def push(self, frames: torch.Tensor, want_env: bool = False) -> Dict[str, object]:
        """One frame per slot in, the samples that became final out: dict(n_out numpy int64 [S], spikes [S, n + D, 2M],
        power [S, G], doa [S], + env [S, n + D, G] and doa_t [S, n + D] when `want_env`).  Slot s fills its first
        n_out[s] rows; the other rows, and power / doa of a slot with n_out[s] == 0, are left as allocated."""
        frames, dt = _check_frames(frames, self.engine.M, self.device, self.num_streams)
        n = frames.shape[1]
        out = self._outputs(n + self.latency, want_env)
        n_out = np.zeros(self.num_streams, dtype=np.int64)
        N.check(self._lib.micloc_snn_streams_push(self._h, _ptr(frames), dt, n, frames.shape[2], _ptr(out["spikes"]),
                                                  _ptr(out["power"]), _ptr(out["doa"]), _ptr(out["env"]),
                                                  _ptr(out["doa_t"]), n_out.ctypes.data_as(C.c_void_p),
                                                  _stream_ptr(self.device)))
        out["n_out"] = n_out
        if not want_env:
            del out["env"], out["doa_t"]
        return out

    def flush(self, slots=None, want_env: bool = False) -> Dict[str, object]:
        """End of the listed recordings (None: all): their remaining samples as in `push` (rows: max_frame_len +
        latency) + 'flags' numpy int32 [S], bit 0 = RZCC overflow anywhere in that slot's recording."""
        arr, p, ns = self._slots(slots)
        out = self._outputs(self.max_frame_len + self.latency, want_env)
        n_out = np.zeros(self.num_streams, dtype=np.int64)
        flags = np.zeros(self.num_streams, dtype=np.int32)
        N.check(self._lib.micloc_snn_streams_flush(self._h, p, ns, _ptr(out["spikes"]), _ptr(out["power"]),
                                                   _ptr(out["doa"]), _ptr(out["env"]), _ptr(out["doa_t"]),
                                                   n_out.ctypes.data_as(C.c_void_p), flags.ctypes.data_as(C.c_void_p),
                                                   _stream_ptr(self.device)))
        out["n_out"], out["flags"] = n_out, flags
        if not want_env:
            del out["env"], out["doa_t"]
        return out


def envelope(x: torch.Tensor, fs: float, rise_time: float, fall_time: float, want_argmax: bool = False):
    """Envelope(rise_time, fall_time, fs).evolve on a device array [T, C] float32 (micloc/utils.py:15-81);
    with `want_argmax` also the per-row argmax (tests/test_snn_hilbert_localization.py:284-293)."""
    if x.dtype != torch.float32 or not x.is_cuda or x.dim() != 2:
        raise ValueError("x must be a CUDA float32 tensor of shape [T, C]")
    x = x.contiguous()
    T, Cc = x.shape
    env = torch.empty_like(x)
    idx = torch.empty(T, dtype=torch.int32, device=x.device) if want_argmax else None
    N.check(N.lib().micloc_envelope(_ptr(x), T, Cc, float(fs), float(rise_time), float(fall_time), _ptr(env), _ptr(idx),
                                    x.device.index or 0, _stream_ptr(x.device)))
    return (env, idx) if want_argmax else env


def rzcc_encode(sig: torch.Tensor, robust_width: int, bipolar: bool) -> torch.Tensor:
    """Exact ZeroCrossingSpikeEncoder.evolve on float64 device input [B,T,C] -> int8 spikes."""
    if sig.dtype != torch.float64 or not sig.is_cuda or sig.dim() != 3:
        raise ValueError("sig must be a CUDA float64 tensor of shape [B, T, C]")
    sig = sig.contiguous()
    B, T, Cc = sig.shape
    out = torch.empty((B, T, Cc), dtype=torch.int8, device=sig.device)
    N.check(N.lib().micloc_rzcc_encode_f64(_ptr(sig), B, T, Cc, int(robust_width), int(bool(bipolar)), _ptr(out),
                                           sig.device.index or 0, _stream_ptr(sig.device)))
    return out
