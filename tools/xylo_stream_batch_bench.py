"""Live-path throughput of the Xylo integer chain: S recordings advanced by one XyloStreamBatch push per frame tick,
against micloc_xylo_run(exact = 1) on the same frames as independent clips (the reference's per-frame behaviour: every
frame restarts from zero state).

Workload: the Xylo demo's frames (paper_plots/snn_localization_benchmark.py: 0.4 s frames) -- int32 `19 200 x 8` wav
frames, 7 microphones + 1 channel that is dropped, 16-bit samples in the upper half of the int32 word -- synthesised on
the device (micloc_synth_clips, seeded: a sine at the band's upper edge, random DoA, SNR cycling over -10..20 dB).
Two networks:
  c3       BASELINE config 3 bipolar (tests/golden/xylo_c3_bipolar.npz): one band, G = 449, tensor-core LIF
  3band    the three bands of config 2 with order-2 filters and the steering matrices of tests/golden/bench_c2_bf.npz:
           N = 1347, N_in = 84, event-loop LIF
Per push: counts + DoA + rate (XyloStreamBatch.push).  After warm-up, pushes are timed for at least --seconds with CUDA
events on the pushing stream.  One JSON line per (network, S):
  push_ms            device time per push
  launches_per_push  micloc_launch_count() delta / pushes
  realtime_factor    S * 0.4 s / push time
  slot_samples_per_s
  oneshot_ms         micloc_xylo_run(exact = 1) on the same S frames as float32 clips (the same sample values)
plus the card name and power limit read in the same run.
  --profile FILE     instead: a torch.profiler run of a few pushes per network at the largest S, per-kernel device time.
Usage: python tools/xylo_stream_batch_bench.py [--slots 1 256 1024 4096] [--out FILE] [--profile FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FS = 48_000
N_FRAME = 19_200               # 0.4 s
N_DISTINCT = 3                 # distinct frames per slot, pushed in turn


def card_info(dev_index):
    import torch
    name = torch.cuda.get_device_name(dev_index)
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(dev_index), "--query-gpu=power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        out = f"unavailable ({type(e).__name__})"
    return name, out


def timed(torch, fn, seconds, warmup=3):
    """(device ms per call, calls) over a run of >= `seconds` of calls, after `warmup` calls."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    calls, total_ms = 0, 0.0
    while total_ms < seconds * 1e3:
        k = max(1, calls)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(k):
            fn()
        ev1.record()
        ev1.synchronize()
        total_ms += ev0.elapsed_time(ev1)
        calls += k
    return total_ms / calls, calls


def networks():
    """(name, XyloEngine, r_vec, theta_vec, synthesis frequency) of the two measured networks."""
    from scipy.signal import butter
    from haghighatshoarmuir2024_b200.xylo_snn_localization import XyloEngine, quantize_network
    out = []
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "xylo_c3_bipolar.npz")))
    fs, order = float(g["fs"]), int(g["order"])
    net = quantize_network(list(g["bf_mats"]), g["taus"], fs, bool(g["bipolar"]))
    eng = XyloEngine(num_mic=7, stht_kernel=g["kernel"],
                     sos_list=[butter(order, b, btype="bandpass", output="sos", fs=fs) for b in g["bands"]],
                     ba_list=list(zip(g["ba_b"], g["ba_a"])), robust_width=int(np.ceil(float(g["robust_width"]))),
                     bipolar=True, net=net, num_doa=len(g["doa_list"]))
    out.append(("c3", eng, g["r_vec"], g["theta_vec"], float(g["bands"][0][1])))
    d = dict(np.load(os.path.join(ROOT, "tests", "golden", "bench_c2_bf.npz")))
    bands = d["bands"]
    taus = np.array([[float(d[f"tau_{f}"])] * 2 for f in range(3)])
    net = quantize_network([d[f"bf_{f}"] for f in range(3)], taus, FS, True)
    eng = XyloEngine(num_mic=7, stht_kernel=d["kernel"],
                     sos_list=[butter(2, b, btype="bandpass", output="sos", fs=FS) for b in bands],
                     ba_list=[butter(2, b, btype="bandpass", output="ba", fs=FS) for b in bands],
                     robust_width=int(np.ceil(float(d["robust_width_0"]))), bipolar=True, net=net, num_doa=449)
    out.append(("3band", eng, d["r_vec"], d["theta_vec"], float(bands[1][1])))
    return out


def frames_for(torch, r_vec, theta_vec, freq, S, seed):
    """N_DISTINCT int32 [S, N_FRAME, 8] wav frames and their float32 [S, N_FRAME, 7] twins (same sample values)."""
    from haghighatshoarmuir2024_b200.montecarlo import synthesize_clips
    rng = np.random.default_rng(seed)
    snr_db = np.linspace(-10, 20, 11)[np.arange(S) % 11]
    snr = 10 ** (snr_db / 10)
    a16 = synthesize_clips(r_vec, theta_vec, FS, N_FRAME * N_DISTINCT, rng.uniform(0, 2 * np.pi, S), snr_lin=snr,
                           sine_freq=freq, seed=seed, dtype=torch.int16)
    a32 = a16.to(torch.int32) * 65536
    del a16
    junk = torch.full((S, N_FRAME, 1), 12345, dtype=torch.int32, device=a32.device)
    wav = [torch.cat([a32[:, i * N_FRAME:(i + 1) * N_FRAME], junk], dim=2).contiguous() for i in range(N_DISTINCT)]
    f32 = a32[:, :N_FRAME].float().contiguous()
    del a32
    return wav, f32


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--slots", type=int, nargs="+", default=[1, 256, 1024, 4096])
    ap.add_argument("--seconds", type=float, default=2.0, help="least timed device time per stream figure")
    ap.add_argument("--out", default=None, help="also write the lines as a JSON list to this file")
    ap.add_argument("--profile", default=None, help="per-kernel torch.profiler split at the largest S to this file")
    args = ap.parse_args()

    import torch
    from haghighatshoarmuir2024_b200 import _native as N
    from haghighatshoarmuir2024_b200.xylo_snn_localization import XyloStreamBatch

    if not torch.cuda.is_available():
        raise SystemExit("xylo_stream_batch_bench.py needs a CUDA device")
    lib = N.lib()
    card, power_limit = card_info(0)
    lines, prof_lines = [], []
    for name, eng, r_vec, theta_vec, freq in networks():
        for S in (args.slots if not args.profile else [max(args.slots)]):
            wav, f32 = frames_for(torch, r_vec, theta_vec, freq, S, seed=1000 + S)
            xsb = XyloStreamBatch(eng, S, N_FRAME, fs=FS)
            tick = [0]

            def push():
                xsb.push(wav[tick[0] % N_DISTINCT])
                tick[0] += 1

            if args.profile:
                from torch.profiler import ProfilerActivity, profile
                for _ in range(3):
                    push()
                torch.cuda.synchronize()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    for _ in range(5):
                        push()
                    torch.cuda.synchronize()
                kern = {}
                for e in prof.key_averages():
                    t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
                    if t > 0:
                        kern[e.key] = {"ms_per_push": t / 1e3 / 5, "calls_per_push": e.count / 5}
                prof_lines.append({"network": name, "slots": S, "n": N_FRAME, "kernels": kern, "card": card,
                                   "power_limit": power_limit,
                                   "timing": "torch.profiler (CUDA activities), 5 pushes after 3 warm-up pushes"})
                print(json.dumps(prof_lines[-1]), flush=True)
            else:
                c0 = lib.micloc_launch_count()
                ms, calls = timed(torch, push, args.seconds)
                launches = (lib.micloc_launch_count() - c0) / (calls + 3)
                ms_one, calls_one = timed(torch, lambda: eng.run(f32, exact=True), args.seconds / 2, warmup=1)
                line = {"network": name, "N": eng.N, "N_in": eng.N_in,
                        "workload": "int32 19200 x 8 wav frames (0.4 s at 48 kHz, 7 mics + 1 dropped), counts + DoA "
                                    "+ rate per push",
                        "slots": S, "n": N_FRAME, "push_ms": ms, "pushes_timed": calls, "launches_per_push": launches,
                        "realtime_factor": S * N_FRAME / FS / (ms * 1e-3),
                        "slot_samples_per_s": S * N_FRAME / (ms * 1e-3), "latency_samples": xsb.latency,
                        "oneshot_ms": ms_one, "oneshot_calls_timed": calls_one, "push_over_oneshot": ms / ms_one,
                        "card": card, "power_limit": power_limit,
                        "timing": "CUDA events around runs of back-to-back calls on the current stream, "
                                  f">= {args.seconds} s of pushes after 3 warm-up pushes, >= {args.seconds / 2} s "
                                  "of one-shot calls after 1 warm-up"}
                print(json.dumps(line), flush=True)
                lines.append(line)
            xsb.close()
            del xsb, wav, f32
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
        eng.close()
    dest, data = (args.profile, prof_lines) if args.profile else (args.out, lines)
    if dest:
        os.makedirs(os.path.dirname(os.path.abspath(dest)), exist_ok=True)
        with open(dest, "w") as f:
            json.dump(data, f, indent=1)
            f.write("\n")


if __name__ == "__main__":
    main()
