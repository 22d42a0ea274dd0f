"""Live multi-band localiser throughput: S recordings advanced by one MultibandStreamBatch push per frame tick, against
`Demo.localize` on the same S frames as independent clips (what the project offered before for the multi-band path).

Workload: the live demo's frames (micloc/localization_demo_snn.py:125-193) -- int32 `n x 8` wav frames, 7 microphones
+ 1 channel that is dropped -- of n = 4800 samples (100 ms at 48 kHz), through the three bands of BASELINE config 2
(7-mic circular array, 10 ms STHT kernel, bipolar RZCC, G = 449; the steering matrices of tests/golden/bench_c2_bf.npz):
filterbank, three chains, power summed over the bands, argmax + both periodic-ML estimators, activity gate.  Every
slot gets its own noisy one-second recording (on-device synthesis, seeded: a 2 kHz tone, inside the middle band, at
an SNR cycling over -10..20 dB), pushed as ten frames and then again from the start.  After a warm-up, pushes are
timed for at least --seconds with CUDA events on the pushing stream.  One JSON line per S:
  push_ms            device time per push (events around a run of pushes / pushes)
  launches_per_push  micloc_launch_count() delta / pushes
  realtime_factor    S * n / fs / push time
  localize_ms        (S <= --max-localize) Demo.localize on the same S frames per tick, each frame an independent clip
plus the card name and power limit read in the same run.  --profile DIR adds one torch.profiler run of a few pushes at
the largest S, per-kernel device times written to DIR/multiband_stream_kernels.json (its own run: tracing slows the
host).  Usage: python tools/multiband_stream_bench.py [--out FILE] [--profile DIR]
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
N_FRAME = 4800
T_REC = 48_000                 # one second per slot, pushed as 10 frames and repeated


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
        k = max(1, calls)                          # doubling runs: few synchronisations
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(k):
            fn()
        ev1.record()
        ev1.synchronize()
        total_ms += ev0.elapsed_time(ev1)
        calls += k
    return total_ms / calls, calls


def make_demo():
    from haghighatshoarmuir2024_b200.array_geometry import ArrayGeometry
    from haghighatshoarmuir2024_b200.localization_demo_snn import Demo
    d = np.load(os.path.join(ROOT, "tests", "golden", "bench_c2_bf.npz"))
    return Demo(geometry=ArrayGeometry(d["r_vec"], d["theta_vec"]), freq_bands=d["bands"], doa_list=d["doa_list"],
                recording_duration=N_FRAME / FS, kernel_duration=float(d["kernel_duration"]), bipolar_spikes=True,
                fs=FS, bf_mats=[d[f"bf_{f}"] for f in range(3)]), d


def frames_for(torch, d, S, dev):
    """S seeded one-second recordings as ten int32 [S, 4800, 8] frames (8th channel junk)."""
    from haghighatshoarmuir2024_b200.montecarlo import synthesize_clips
    rng = np.random.default_rng(1000 + S)
    snr_db = np.linspace(-10, 20, 11)[np.arange(S) % 11]
    audio = synthesize_clips(d["r_vec"], d["theta_vec"], FS, T_REC, rng.uniform(0, 2 * np.pi, S),
                             snr_lin=10 ** (snr_db / 10), sine_freq=2000.0, mode=0, seed=1000 + S, dtype=torch.int16,
                             device=dev.index or 0)
    frames = torch.cat([audio.to(torch.int32) * 65536,
                        torch.full((S, T_REC, 1), 12345, dtype=torch.int32, device=dev)], dim=2)
    del audio
    return [frames[:, i * N_FRAME:(i + 1) * N_FRAME].contiguous() for i in range(T_REC // N_FRAME)]


def profile(torch, demo, frame_list, S, out_dir):
    from torch.profiler import ProfilerActivity, profile as tprofile
    mb = demo.stream_batch(S, max_frame_len=N_FRAME)
    for i in range(3):
        mb.push(frame_list[i])
    torch.cuda.synchronize()
    pushes = 5
    with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(pushes):
            mb.push(frame_list[(3 + i) % len(frame_list)])
        torch.cuda.synchronize()
    rows = []
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = getattr(e, "cuda_time_total", 0.0)
        if t > 0:
            rows.append({"name": e.key, "calls": e.count, "ms_per_push": t / 1e3 / pushes})
    rows.sort(key=lambda r: -r["ms_per_push"])
    mb.close()
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "multiband_stream_kernels.json"), "w") as f:
        json.dump({"slots": S, "pushes": pushes, "kernels": rows}, f, indent=1)
        f.write("\n")
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--slots", type=int, nargs="+", default=[1, 64, 256, 1024, 4096])
    ap.add_argument("--seconds", type=float, default=2.0, help="least timed device time per measurement")
    ap.add_argument("--max-localize", type=int, default=4096, help="largest S also run through Demo.localize")
    ap.add_argument("--out", default=None, help="also write the lines as a JSON list to this file")
    ap.add_argument("--profile", default=None, help="directory for the per-kernel profile at the largest S")
    args = ap.parse_args()

    import torch
    from haghighatshoarmuir2024_b200 import _native as N

    if not torch.cuda.is_available():
        raise SystemExit("multiband_stream_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    demo, d = make_demo()
    lib = N.lib()
    card, power_limit = card_info(0)
    lines = []
    for S in args.slots:
        frame_list = frames_for(torch, d, S, dev)
        tick = [0]
        mb = demo.stream_batch(S, max_frame_len=N_FRAME)

        def push():
            mb.push(frame_list[tick[0] % len(frame_list)])
            tick[0] += 1

        c0 = lib.micloc_launch_count()
        ms, calls = timed(torch, push, args.seconds)
        launches = (lib.micloc_launch_count() - c0) / (calls + 3)
        line = {"workload": "live frames: int32 n x 8 (7 mics + 1 dropped), n = 4800 (100 ms at 48 kHz), the three "
                            "bands of BASELINE config 2 (G = 449): filterbank, chains, power fusion, estimators, "
                            "activity gate per push",
                "slots": S, "n": N_FRAME, "bands": len(demo.beamfs), "push_ms": ms, "pushes_timed": calls,
                "launches_per_push": launches, "realtime_factor": S * N_FRAME / FS / (ms * 1e-3),
                "slot_samples_per_s": S * N_FRAME / (ms * 1e-3), "latency_samples": mb.latency}
        mb.close()
        del mb
        if S <= args.max_localize:
            tick[0] = 0

            def localize():
                demo.localize(frame_list[tick[0] % len(frame_list)])
                tick[0] += 1

            ms_loc, calls_loc = timed(torch, localize, args.seconds)
            line.update({"localize_ms": ms_loc, "localize_ticks_timed": calls_loc,
                         "localize_over_push": ms_loc / ms})
        if args.profile and S == max(args.slots):
            line["profile"] = "multiband_stream_kernels.json"
            profile(torch, demo, frame_list, S, args.profile)
        del frame_list
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        line.update({"card": card, "power_limit": power_limit,
                     "timing": "CUDA events around runs of back-to-back calls on the current stream, "
                               f">= {args.seconds} s per figure after 3 warm-up calls"})
        print(json.dumps(line), flush=True)
        lines.append(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(lines, f, indent=1)
            f.write("\n")


if __name__ == "__main__":
    main()
