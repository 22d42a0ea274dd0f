"""Live-path throughput: S recordings advanced by one SnnStreamBatch push per frame tick, against S separate SnnStreams.

Workload: the live demo's frames (micloc/localization_demo_snn.py:125-193) -- int32 `n x 8` wav frames, 7 microphones
+ 1 channel that is dropped -- of n = 4800 samples (100 ms at 48 kHz), on band 0 of BASELINE config 2 (7-mic circular
array, 10 ms STHT kernel, bipolar RZCC, G = 449; the steering matrix of tests/golden/bench_c2_bf.npz).  Every slot
gets its own noisy one-second recording (on-device synthesis, seeded), pushed as ten frames and then again from the
start, with power + DoA per push (no envelope).  After a warm-up, pushes are timed for at least --seconds with CUDA
events on the pushing stream.  One JSON line per S:
  push_ms          device time per push (events around a run of pushes / pushes)
  launches_per_push  micloc_launch_count() delta / pushes
  realtime_factor  S * n / fs / push time
  slot_samples_per_s
  separate_push_ms  (S <= --max-separate) the same frames through S SnnStream objects, one push each per tick
plus the card name and power limit read in the same run.  Usage: python tools/stream_batch_bench.py [--out FILE]
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


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--slots", type=int, nargs="+", default=[1, 16, 256, 4096])
    ap.add_argument("--seconds", type=float, default=1.0, help="least timed device time per measurement")
    ap.add_argument("--max-separate", type=int, default=256, help="largest S also run as S separate SnnStreams")
    ap.add_argument("--out", default=None, help="also write the lines as a JSON list to this file")
    args = ap.parse_args()

    import torch
    from haghighatshoarmuir2024_b200 import _native as N
    from haghighatshoarmuir2024_b200.engine import SnnStream, SnnStreamBatch
    from haghighatshoarmuir2024_b200.montecarlo import BandSetup, SnrSweep

    if not torch.cuda.is_available():
        raise SystemExit("stream_batch_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    d = np.load(os.path.join(ROOT, "tests", "golden", "bench_c2_bf.npz"))
    band = [float(v) for v in d["bands"][0]]
    sweep = SnrSweep([BandSetup(band=band, tau=float(d["tau_0"]), bf_mat=d["bf_0"])], d["r_vec"], d["theta_vec"], FS,
                     float(d["kernel_duration"]), T_REC, device=0)
    eng = sweep.engines[0]
    lib = N.lib()
    card, power_limit = card_info(0)
    lines = []
    for S in args.slots:
        audio, _, _ = sweep.synthesize(0, S, seed=1000 + S, snr_db_grid=np.linspace(-10, 20, 11), dtype=torch.int16)
        frames = torch.cat([audio.to(torch.int32), torch.full((S, T_REC, 1), 12345, dtype=torch.int32, device=dev)], dim=2)
        del audio
        frame_list = [frames[:, i * N_FRAME:(i + 1) * N_FRAME].contiguous() for i in range(T_REC // N_FRAME)]
        del frames
        tick = [0]

        sb = SnnStreamBatch(eng, S, max_frame_len=N_FRAME)

        def push_batch():
            sb.push(frame_list[tick[0] % len(frame_list)])
            tick[0] += 1

        c0 = lib.micloc_launch_count()
        ms, calls = timed(torch, push_batch, args.seconds)
        launches = (lib.micloc_launch_count() - c0) / (calls + 3)
        line = {"workload": "live frames: int32 n x 8 (7 mics + 1 dropped), n = 4800 (100 ms at 48 kHz), band 0 of "
                            "BASELINE config 2 (G = 449), power + DoA per push",
                "slots": S, "n": N_FRAME, "push_ms": ms, "pushes_timed": calls, "launches_per_push": launches,
                "realtime_factor": S * N_FRAME / FS / (ms * 1e-3),
                "slot_samples_per_s": S * N_FRAME / (ms * 1e-3), "latency_samples": sb.latency}
        sb.close()
        del sb
        if S <= args.max_separate:
            streams = [SnnStream(eng, max_frame_len=N_FRAME) for _ in range(S)]
            per_slot = [[f[s] for f in frame_list] for s in range(S)]

            def push_separate():
                k = tick[0] % len(frame_list)
                for s, st in enumerate(streams):
                    st.push(per_slot[s][k])
                tick[0] += 1

            tick[0] = 0
            c0 = lib.micloc_launch_count()
            ms_sep, calls_sep = timed(torch, push_separate, args.seconds)
            line.update({"separate_push_ms": ms_sep, "separate_ticks_timed": calls_sep,
                         "separate_launches_per_tick": (lib.micloc_launch_count() - c0) / (calls_sep + 3),
                         "speedup_vs_separate": ms_sep / ms})
            for st in streams:
                st.close()
            del streams, per_slot
        del frame_list
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        line.update({"card": card, "power_limit": power_limit,
                     "timing": "CUDA events around runs of back-to-back pushes on the current stream, "
                               f">= {args.seconds} s per figure after 3 warm-up pushes"})
        print(json.dumps(line), flush=True)
        lines.append(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(lines, f, indent=1)
            f.write("\n")


if __name__ == "__main__":
    main()
