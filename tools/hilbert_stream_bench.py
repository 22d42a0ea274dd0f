"""Live Hilbert beamformer throughput: S recordings advanced by one HilbertStreamBatch push per frame tick, against the
one-shot path on the same S frames as independent clips (micloc_filterbank + micloc_hilbert_localize per band +
micloc_power_fuse with a filterbank; Beamformer.localize's micloc_hilbert_localize without one).

Cases (frames of n = 4800 samples, 100 ms at 48 kHz):
  c2_bank    BASELINE config 2's three bands (7-mic circular array, 10 ms STHT kernel, G = 449) behind the Butterworth
             filterbank, int32 `4800 x 8` wav frames; outputs power_grid, doa, both estimators, sumsq / activity gate.
             Steering matrices: the config-2 matrices of tests/golden/bench_c2_bf.npz read as complex ([Re; Im] rows).
             S in {1, 256, 1024, 4096}.
  c2_raw     band 1 of config 2 alone, no filterbank, the same frames; outputs power and doa.  Same S.
  linear64   the 64-microphone linear array (2 cm pitch, 400-2000 Hz band, random complex steering, G = 181), float32
             frames, no filterbank; outputs power and doa.  S in {1, 64}.
Every slot holds a seeded tone + noise recording; the same frame is pushed again and again (state carries on).  After
5 warm-up pushes, --pushes pushes (at least 50) are timed with CUDA events on the pushing stream, and the one-shot
path likewise.  One JSON document: per case push_ms, launches_per_push, slot_samples_per_s, realtime_factor (seconds of
audio each recording advances per second of push), oneshot_ms and ratio, plus one torch.profiler pass of c2_bank at
S = 4096 (per-kernel device time per push, its own run) and the card name and power limit read in the same run.
Usage: python tools/hilbert_stream_bench.py [--out FILE] [--pushes K]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FS = 48_000
N_FRAME = 4800


def card_info(dev_index):
    import torch
    name = torch.cuda.get_device_name(dev_index)
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(dev_index), "--query-gpu=power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        out = f"unavailable ({type(e).__name__})"
    return name, out


def timed(torch, fn, pushes, warmup=5):
    """device ms per call over `pushes` calls after `warmup` calls, and the launch-count delta per call"""
    from haghighatshoarmuir2024_b200 import _native as N
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    c0 = N.lib().micloc_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(pushes):
        fn()
    ev1.record()
    ev1.synchronize()
    return ev0.elapsed_time(ev1) / pushes, (N.lib().micloc_launch_count() - c0) / pushes


def frames_for(torch, geo_r, geo_th, S, M, dtype, seed):
    """one frame per slot [S, 4800, M + 1]: a tone from a random direction (plane wave delays) + noise; last channel junk"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    t = torch.arange(N_FRAME, device="cuda", dtype=torch.float64) / FS
    doa = torch.rand(S, 1, 1, generator=g, device="cuda", dtype=torch.float64) * 2 * np.pi
    r = torch.as_tensor(geo_r, device="cuda")[None, None]
    th = torch.as_tensor(geo_th, device="cuda")[None, None]
    delay = -r * torch.cos(th - doa) / 340.0
    x = torch.sin(2 * np.pi * 1800.0 * (t[None, :, None] - delay))
    x = x + 0.3 * torch.randn(x.shape, generator=g, device="cuda", dtype=torch.float64)
    x = x / x.abs().amax(dim=(1, 2), keepdim=True) * 0.9
    x = torch.cat([x, torch.full_like(x[..., :1], 0.001)], dim=2)
    if dtype == torch.int32:
        return (x * 2.0 ** 31).round().to(torch.int32).contiguous()
    return x.to(torch.float32).contiguous()


def c2_setup(d):
    from haghighatshoarmuir2024_b200.array_geometry import ArrayGeometry
    from haghighatshoarmuir2024_b200.beamformer import Beamformer
    geo = ArrayGeometry(d["r_vec"], d["theta_vec"])
    M = len(d["r_vec"])
    bands = []
    for f, band in enumerate(d["bands"]):
        bf = Beamformer(geo, float(d["kernel_duration"]), list(band), fs=FS)
        bf.verbose = False
        w = np.asarray(d[f"bf_{f}"], np.float64)
        bands.append((bf, w[:M] + 1j * w[M:]))
    return geo, bands


def run_case(torch, name, bands, bank, doa_list, S, frames, want, pushes):
    from haghighatshoarmuir2024_b200 import _native as N
    from haghighatshoarmuir2024_b200.beamformer import HilbertStreamBatch
    from haghighatshoarmuir2024_b200.engine import _ptr
    hb = HilbertStreamBatch(bands, S, N_FRAME, filterbank=bank, doa_list=doa_list)
    push_ms, lpp = timed(torch, lambda: hb.push(frames, want=want), pushes)
    M, G, F = hb.M, hb.G, hb.F
    L = N.lib()
    engs = hb.engines
    if bank is not None:
        sos = np.ascontiguousarray(bank.sos_list, dtype=np.float64)
        rows = torch.empty((F, S, N_FRAME, M), dtype=torch.float32, device="cuda")
        ss = torch.empty(S, dtype=torch.float64, device="cuda")
        power = torch.empty((F, S, G), dtype=torch.float32, device="cuda")
        grid = torch.empty((S, G), dtype=torch.float32, device="cuda")
        doa = torch.empty(S, dtype=torch.int32, device="cuda")
        ml = torch.empty(S, dtype=torch.float64, device="cuda")
        tr = torch.empty(S, dtype=torch.float64, device="cuda")
        fl = torch.empty(S, dtype=torch.int32, device="cuda")
        dl = torch.from_numpy(np.ascontiguousarray(doa_list, dtype=np.float64)).cuda()
        code = N.I32 if frames.dtype == torch.int32 else N.F32

        def oneshot():
            N.check(L.micloc_filterbank(_ptr(frames), code, S, N_FRAME, frames.shape[2], M, F, sos.shape[1],
                                        sos.ctypes.data_as(N._dp), _ptr(rows), _ptr(ss), 0, None))
            for f, e in enumerate(engs):
                N.check(L.micloc_hilbert_localize(e._h, _ptr(rows[f]), N.F32, S, N_FRAME, 0, 1, None, None,
                                                  _ptr(power[f]), None, None))
            N.check(L.micloc_power_fuse(_ptr(power), F, S, G, _ptr(dl), _ptr(grid), _ptr(doa), _ptr(ml), _ptr(tr),
                                        _ptr(fl), 0, None))
    else:
        clips = frames[..., :M].to(torch.float32).contiguous()     # Beamformer.localize takes [B, T, M] f32 / i16
        bf, bf_mat = bands[0]
        oneshot = lambda: bf.localize(bf_mat, clips)
    one_ms, one_lpp = timed(torch, oneshot, pushes)
    hb.close()
    rec = {"case": name, "S": S, "frame": N_FRAME, "bands": F, "mics": M, "G": G, "dtype": str(frames.dtype),
           "want": list(want), "pushes": pushes, "push_ms": round(push_ms, 4), "launches_per_push": lpp,
           "slot_samples_per_s": S * N_FRAME / (push_ms * 1e-3),
           "realtime_factor": (N_FRAME / FS) / (push_ms * 1e-3),
           "oneshot_ms": round(one_ms, 4), "oneshot_launches": one_lpp, "ratio_to_oneshot": round(push_ms / one_ms, 3)}
    print(json.dumps(rec), flush=True)
    return rec


def profile(torch, bands, bank, doa_list, S, frames, want):
    from torch.profiler import ProfilerActivity, profile as tprofile
    from haghighatshoarmuir2024_b200.beamformer import HilbertStreamBatch
    hb = HilbertStreamBatch(bands, S, N_FRAME, filterbank=bank, doa_list=doa_list)
    for _ in range(3):
        hb.push(frames, want=want)
    torch.cuda.synchronize()
    k = 5
    with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(k):
            hb.push(frames, want=want)
        torch.cuda.synchronize()
    hb.close()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
        if t > 0:
            out[e.key[:120]] = {"ms_per_push": round(t / 1e3 / k, 4), "calls_per_push": e.count / k}
    return dict(sorted(out.items(), key=lambda kv: -kv[1]["ms_per_push"]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--pushes", type=int, default=50)
    a = ap.parse_args()
    if a.pushes < 50:
        ap.error("--pushes must be at least 50")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("hilbert_stream_bench needs a CUDA device")
    from haghighatshoarmuir2024_b200.array_geometry import ArrayGeometry
    from haghighatshoarmuir2024_b200.beamformer import Beamformer
    from haghighatshoarmuir2024_b200.filterbank import ButterworthFilterbank
    name, plimit = card_info(0)
    d = np.load(os.path.join(ROOT, "tests", "golden", "bench_c2_bf.npz"))
    geo, bands = c2_setup(d)
    bank = ButterworthFilterbank(d["bands"], order=2, fs=FS)
    doa_list = np.asarray(d["doa_list"], np.float64)
    bank_want = ("power_grid", "doa", "periodic_ml", "trimmed_periodic_ml")
    results = []
    for S in (1, 256, 1024, 4096):
        fr = frames_for(torch, geo.r_vec, geo.theta_vec, S, len(geo.r_vec), torch.int32, seed=S)
        results.append(run_case(torch, "c2_bank", bands, bank, doa_list, S, fr, bank_want, a.pushes))
        results.append(run_case(torch, "c2_raw", bands[1:2], None, None, S, fr, ("power", "doa"), a.pushes))
        del fr
    M64 = 64
    r64, th64 = np.abs(np.arange(M64) - (M64 - 1) / 2) * 0.02, np.where(np.arange(M64) < M64 / 2, np.pi, 0.0)
    geo64 = ArrayGeometry(r64, th64)
    bf64 = Beamformer(geo64, 10e-3, [400.0, 2000.0], fs=FS)
    bf64.verbose = False
    rng = np.random.default_rng(64)
    W64 = rng.standard_normal((M64, 181)) + 1j * rng.standard_normal((M64, 181))
    for S in (1, 64):
        fr = frames_for(torch, r64, th64, S, M64, torch.float32, seed=64 + S)
        results.append(run_case(torch, "linear64", [(bf64, W64)], None, None, S, fr, ("power", "doa"), a.pushes))
    fr = frames_for(torch, geo.r_vec, geo.theta_vec, 4096, len(geo.r_vec), torch.int32, seed=4096)
    kernels = profile(torch, bands, bank, doa_list, 4096, fr, bank_want)
    doc = {"card": name, "power_limit": plimit, "torch": torch.__version__, "results": results,
           "profile_c2_bank_S4096": kernels}
    text = json.dumps(doc, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    print(json.dumps({"card": name, "power_limit": plimit, "profile": kernels}))


if __name__ == "__main__":
    main()
