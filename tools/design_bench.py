"""design_from_template on the host path against design_on_device, end to end, with the results compared.

Cases (fs = 48 kHz, 10 ms STHT kernel):
  c2_band0_snn_bipolar / c2_band0_hilbert   BASELINE config 2 band 0 (1600-2000 Hz): 7-mic centre-circular array
                                            (r = 4.5 cm), G = 449 DoAs in [-pi, pi], a 1 s linear chirp across the band
  c5_linear64_bipolar_{0.25,1}s             config 5: the 64-mic linear array of the snn_c5_linear64 golden (its band,
                                            tau, bipolar SNN), G = 512, a chirp template of 0.25 s and 1 s
  c5_random64_unipolar_{0.25,1}s            the same for the 64-mic random array of snn_c5_random64 (unipolar)
Per case: host_s (design_from_template: host np.interp of the templates, device covariance, host SVDs / bisection),
device_s (design_on_device until the device is idle), and the agreement of the two matrices: unipolar inf-norm,
otherwise min_g |<u_dev, u_host>| (phase-invariant).  Each timed once after a warm-up call on a small DoA grid.
Also, from separate runs:
  kernels_ms   per-kernel device time of one c5_linear64_bipolar_0.25s device design (torch.profiler)
  solver       micloc_design_vectors alone on 512 random PSD matrices of 128 x 128 (mode 0, and mode 2 on their
               64 x 64 complex counterparts), against torch.linalg.eigh on the same batches on the GPU (CUDA events,
               best of 3)
The card name and power limit are read in the same run.
Usage: python tools/design_bench.py [--out profiles/r07_design_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

FS = 48_000


def card_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        out = f"unavailable ({type(e).__name__})"
    return name, out


def chirp(seconds, f0, f1):
    t = np.arange(int(seconds * FS)) / FS
    return t, np.sin(2 * np.pi * (f0 + (f1 - f0) * t / t[-1] / 2) * t)


def cases():
    import helpers as H
    from haghighatshoarmuir2024_b200.array_geometry import ArrayGeometry, CenterCircularArray
    from haghighatshoarmuir2024_b200.beamformer import Beamformer
    from haghighatshoarmuir2024_b200.snn_beamformer import SNNBeamformer
    out = []
    c1 = H.load("snn_c1_bipolar")
    tau = float(c1["tau"])
    band = [1600.0, 2000.0]
    doa449 = np.linspace(-np.pi, np.pi, 449)
    geo7 = CenterCircularArray(4.5e-2, 7)
    out.append(("c2_band0_snn_bipolar", SNNBeamformer(geo7, 10e-3, band, np.array([tau, tau]), bipolar_spikes=True,
                                                      fs=FS), chirp(1.0, *band), doa449, "snn"))
    out.append(("c2_band0_hilbert", Beamformer(geo7, 10e-3, band, fs=FS), chirp(1.0, *band), doa449, "hilbert"))
    for name, label in (("snn_c5_linear64", "c5_linear64_bipolar"), ("snn_c5_random64", "c5_random64_unipolar")):
        g = H.load(name)
        geo = ArrayGeometry(g["r_vec"], g["theta_vec"])
        tg = float(g["tau"])
        for sec in (0.25, 1.0):
            bf = SNNBeamformer(geo, float(g["kernel_duration"]), list(g["band"]), np.array([tg, tg]),
                               bipolar_spikes=bool(g["bipolar"]), fs=FS)
            out.append((f"{label}_{sec:g}s", bf, chirp(sec, *g["band"]), np.asarray(g["doa_list"]), "snn"))
    return out


def compare(kind, bipolar, dev, host):
    if kind == "hilbert":
        return {"min_phase_inner": float(np.abs(np.sum(np.conj(dev) * host, axis=0)).min())}
    if not bipolar:
        return {"inf_norm": float(np.abs(dev - host).max())}
    M = dev.shape[0] // 2
    u, h = dev[:M] + 1j * dev[M:], host[:M] + 1j * host[M:]
    return {"min_phase_inner": float(np.abs(np.sum(np.conj(u) * h, axis=0)).min())}


def run_case(name, beamf, template, doa, kind):
    import torch
    beamf.verbose = False
    design_dev = (lambda d: beamf.design_on_device(template, d)[0]) if kind == "hilbert" else \
        (lambda d: beamf.design_on_device(template, d))
    design_host = (lambda d: beamf.design_from_template(template, d)[0]) if kind == "hilbert" else \
        (lambda d: beamf.design_from_template(template, d))
    design_dev(doa[:8]); design_host(doa[:8])                 # contexts, scratch, module loads
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    dev = design_dev(doa)
    torch.cuda.synchronize()
    dev_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    host = design_host(doa)
    host_s = time.perf_counter() - t0
    bipolar = kind == "snn" and bool(beamf.spk_encoder.bipolar)
    r = {"case": name, "num_mic": len(beamf.geometry), "G": len(doa), "T": len(template[0]), "host_s": host_s,
         "device_s": dev_s, "speedup": host_s / dev_s}
    r.update(compare(kind, bipolar, dev.cpu().numpy(), host))
    print(json.dumps(r), flush=True)
    return r


def kernel_split(beamf, template, doa):
    import torch
    from torch.profiler import ProfilerActivity, profile
    beamf.design_on_device(template, doa)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        beamf.design_on_device(template, doa)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if e.device_type.name == "CUDA" and getattr(e, "device_time_total", 0) > 0:
            out[e.key[:80]] = {"ms": e.device_time_total / 1e3, "calls": e.count}
    return dict(sorted(out.items(), key=lambda kv: -kv[1]["ms"]))


def events_best_ms(fn, reps=3):
    import torch
    best = float("inf")
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        best = min(best, a.elapsed_time(b))
    return best


def solver_vs_eigh():
    import torch
    from haghighatshoarmuir2024_b200.engine import design_vectors
    rng = np.random.default_rng(0)
    X = rng.standard_normal((512, 128, 131))
    C = torch.from_numpy(X @ X.transpose(0, 2, 1)).cuda()
    Z = rng.standard_normal((512, 64, 67)) + 1j * rng.standard_normal((512, 64, 67))
    Hc = torch.from_numpy(Z @ np.conj(Z.transpose(0, 2, 1))).cuda()
    design_vectors(0, C); design_vectors(2, Hc); torch.linalg.eigh(C); torch.linalg.eigh(Hc)
    torch.cuda.synchronize()
    r = {"batch": 512,
         "mode0_n128_ms": events_best_ms(lambda: design_vectors(0, C)),
         "eigh_real_n128_ms": events_best_ms(lambda: torch.linalg.eigh(C)),
         "mode2_M64_ms": events_best_ms(lambda: design_vectors(2, Hc)),
         "eigh_complex_M64_ms": events_best_ms(lambda: torch.linalg.eigh(Hc))}
    v = design_vectors(2, Hc).cpu().numpy()
    w = torch.linalg.eigh(Hc)[1][:, :, -1].cpu().numpy().T
    r["mode2_vs_eigh_min_phase_inner"] = float(np.abs(np.sum(np.conj(v) * w, axis=0)).min())
    print(json.dumps(r), flush=True)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_design_bench.json"))
    a = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "design_bench needs a GPU"
    card, power_limit = card_info()
    res = {"card": card, "power_limit": power_limit, "cases": []}
    cs = cases()
    for name, beamf, template, doa, kind in cs:
        res["cases"].append(run_case(name, beamf, template, doa, kind))
    _, beamf, template, doa, _ = next(c for c in cs if c[0] == "c5_linear64_bipolar_0.25s")
    res["kernels_ms_c5_linear64_bipolar_0.25s"] = kernel_split(beamf, template, doa)
    res["solver"] = solver_vs_eigh()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
