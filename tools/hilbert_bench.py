"""Hilbert beamformer at batch scale (micloc_hilbert_localize) on the Monte-Carlo workload of BASELINE configs[1].

Workload: 7-mic centre-circular array (r = 4.5 cm), fs = 48 kHz, one-second clips, 10 ms STHT kernel, the three bands
1600-2000 / 2000-2300 / 2300-2600 Hz, G = 449 DoAs in [-pi, pi]; --clips-per-band noisy single-target clips per band
synthesised on the device (SnrSweep.synthesize: sine at the band's upper edge, uniform DoA, the 11 SNRs of
target_snn_localization.py:435 in turn).  The steering matrix of each band is designed by Beamformer.design_from_template
(one batched device call per chunk of DoAs + host SVDs) from a one-second linear chirp across the band.

Measured, in one run, with the card name and power limit read in the same run:
  design_s             design_from_template for G = 449, per band (host template synthesis + device covariance + SVDs)
  clips_per_s          micloc_hilbert_localize on all bands' clips (CUDA events around --reps passes, after a warm-up)
  kernels_ms           per-kernel device time of one pass, from a separate torch.profiler run
  roofline             FLOP per mic sample F = K + 40 + (2M)(2M+1)/M (FMA = 2: K/2 kept STHT taps, 2 channels x 2
                       biquads, the upper triangle of the float64 Gram matrix; the power epilogue is per clip and left
                       out) x mic samples/s, over the measured FP32 FFMA peak (micloc_fp32_peak variant 0)
  same_clips           --dense-clips clips of band 0 through micloc_hilbert_beamform (dense y [B][T][G][2], power,
                       DoA), micloc_hilbert_localize and the fused SNN chain (micloc_snn_run): ms each, DoA agreement
  doa_error_by_snr     mean arcsin|sin(est - true)| (target_snn_localization.py:466) per SNR, both arms, same clips
Usage: python tools/hilbert_bench.py --out DIR   (writes DIR/hilbert_bench.json)
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FS = 48_000
T_CLIP = 48_000
SNR_GRID = np.linspace(-10, 20, 11)          # target_snn_localization.py:435


def card_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        out = f"unavailable ({type(e).__name__})"
    return name, out


def flops_per_mic_sample(K, M):
    return K + 40 + (2 * M) * (2 * M + 1) / M


def events_ms(fn, reps):
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="output directory")
    ap.add_argument("--clips-per-band", type=int, default=7104)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--dense-clips", type=int, default=64)
    args = ap.parse_args()

    import torch
    from haghighatshoarmuir2024_b200 import _native as N
    from haghighatshoarmuir2024_b200.array_geometry import ArrayGeometry
    from haghighatshoarmuir2024_b200.beamformer import Beamformer
    from haghighatshoarmuir2024_b200.engine import _ptr, _stream_ptr
    from haghighatshoarmuir2024_b200.montecarlo import BandSetup, SnrSweep

    if not torch.cuda.is_available():
        raise SystemExit("hilbert_bench needs a CUDA device")
    card, power_limit = card_info()
    d = np.load(os.path.join(ROOT, "tests", "golden", "bench_c2_bf.npz"))
    bands = [list(map(float, b)) for b in d["bands"]]
    doa_list = np.asarray(d["doa_list"])
    kd = float(d["kernel_duration"])
    geo = ArrayGeometry(d["r_vec"], d["theta_vec"])
    M, G, Bb = len(d["r_vec"]), len(doa_list), args.clips_per_band

    # ---- design (G = 449 per band) from a one-second chirp across the band ----
    t = np.arange(T_CLIP) / FS
    bf_h, design_s = [], []
    for band in bands:
        bf = Beamformer(geo, kd, band, fs=FS)
        bf.verbose = False
        chirp = np.sin(2 * np.pi * (band[0] * t + (band[1] - band[0]) * t ** 2 / (2 * t[-1])))
        if not bf_h:
            bf.design_from_template((t[:4800], chirp[:4800]), doa_list[:8])        # warm-up: context, kernels
        t0 = time.perf_counter()
        w, _ = bf.design_from_template((t, chirp), doa_list)
        torch.cuda.synchronize()
        design_s.append(time.perf_counter() - t0)
        bf_h.append(w)
    setups = [BandSetup(band=bands[i], tau=float(d[f"tau_{i}"]), bf_mat=d[f"bf_{i}"], bf_hilbert=bf_h[i])
              for i in range(len(bands))]
    sweep = SnrSweep(setups, d["r_vec"], d["theta_vec"], FS, kd, T_CLIP)
    audio, doa_true, snr_idx = [], [], []
    for i in range(len(bands)):
        a, dt_, si = sweep.synthesize(i, Bb, seed=20_000 + i, snr_db_grid=SNR_GRID)
        audio.append(a); doa_true.append(dt_); snr_idx.append(si)
    torch.cuda.synchronize()

    # ---- throughput ----
    def pass_all():
        return [sweep.run_band_hilbert(i, audio[i]) for i in range(len(bands))]
    outs = pass_all()
    torch.cuda.synchronize()
    n0 = N.lib().micloc_launch_count()
    ms = events_ms(pass_all, args.reps)
    launches = (N.lib().micloc_launch_count() - n0) / args.reps
    clips = Bb * len(bands)
    clips_per_s = clips / (ms / 1e3)
    mic_samples_per_s = clips_per_s * T_CLIP * M

    # ---- per-kernel split (separate run) ----
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        pass_all()
        torch.cuda.synchronize()
    kernels = {}
    for e in prof.key_averages():
        if e.device_type.name == "CUDA" and e.device_time_total > 0:
            kernels[e.key] = {"ms": e.device_time_total / 1e3, "calls": e.count}

    # ---- roofline ----
    peak = ctypes.c_double()
    N.check(N.lib().micloc_fp32_peak(0, 0, ctypes.byref(peak)))
    F = flops_per_mic_sample(len(d["kernel"]), M)
    achieved = F * mic_samples_per_s / 1e12

    # ---- the same clips through the dense path, the new path and the fused SNN chain ----
    Bd = min(args.dense_clips, Bb)
    x = audio[0][:Bd].contiguous()
    eng = sweep.engines[0]
    y = torch.empty((Bd, T_CLIP, G, 2), dtype=torch.float32, device="cuda")
    pd = torch.empty((Bd, G), dtype=torch.float32, device="cuda")
    dd = torch.empty(Bd, dtype=torch.int32, device="cuda")
    re, im = np.ascontiguousarray(bf_h[0].real), np.ascontiguousarray(bf_h[0].imag)

    def dense():
        N.check(N.lib().micloc_hilbert_beamform(eng._h, _ptr(x), N.F32, Bd, T_CLIP, re.ctypes.data_as(N._dp),
                                                im.ctypes.data_as(N._dp), G, _ptr(y), _ptr(pd), _ptr(dd),
                                                _stream_ptr(eng.device)))
    dense(); torch.cuda.synchronize()
    dense_ms = events_ms(dense, 3)
    new_out = sweep.run_band_hilbert(0, x)
    new_ms = events_ms(lambda: sweep.run_band_hilbert(0, x), 10)
    sweep.run_band(0, x, want_power=False)
    snn_ms = events_ms(lambda: sweep.run_band(0, x, want_power=False, refine=False), 10)
    torch.cuda.synchronize()
    agree = float((new_out["doa"] == dd).float().mean())
    p_rel = float(((new_out["power"] - pd).abs().max(dim=1).values / pd.abs().max(dim=1).values).max())

    # ---- DoA error by SNR, both arms on the same clips ----
    err_h = np.zeros(len(SNR_GRID)); err_s = np.zeros(len(SNR_GRID)); cnt = np.zeros(len(SNR_GRID))
    for i in range(len(bands)):
        eh = sweep.doa_error(outs[i]["doa"].cpu().numpy(), doa_true[i], doa_list)
        es = sweep.doa_error(sweep.run_band(i, audio[i], want_power=False)["doa"].cpu().numpy(), doa_true[i], doa_list)
        for k in range(len(SNR_GRID)):
            sel = snr_idx[i] == k
            err_h[k] += eh[sel].sum(); err_s[k] += es[sel].sum(); cnt[k] += sel.sum()

    res = {
        "card": card, "power_limit": power_limit,
        "workload": f"configs[1]: {len(bands)} bands x {Bb} one-second 7-mic clips, G = {G}, 11 SNRs in [-10, 20] dB",
        "design_s_per_band_G449": design_s,
        "localize": {"ms_per_pass": ms, "clips_per_pass": clips, "clips_per_s": clips_per_s,
                     "mic_samples_per_s": mic_samples_per_s, "launches_per_pass": launches},
        "kernels_ms_one_pass": kernels,
        "roofline": {"flop_per_mic_sample": F, "formula": "K + 40 + (2M)(2M+1)/M, K = 480",
                     "achieved_tflops": achieved, "fp32_peak_tflops": peak.value, "frac": achieved / peak.value},
        "same_clips": {"clips": Bd, "band": 0, "hilbert_beamform_dense_ms": dense_ms, "hilbert_localize_ms": new_ms,
                       "snn_fused_run_ms": snn_ms, "doa_agreement_localize_vs_dense": agree,
                       "power_max_rel_diff_localize_vs_dense": p_rel},
        "doa_error_by_snr": {"snr_db": SNR_GRID.tolist(), "hilbert_rad": (err_h / cnt).tolist(),
                             "snn_rad": (err_s / cnt).tolist(), "clips_per_snr": cnt.tolist()},
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "hilbert_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("card", "power_limit", "localize", "roofline", "same_clips")}))


if __name__ == "__main__":
    main()
