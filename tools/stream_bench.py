"""Streaming HiFi-GAN benchmark: S concurrent 10-s sessions fed in fixed-size mel chunks, stepped together.

For each (S, chunk) it reports the step time (mean, p95; host clock around a device synchronise), the aggregate seconds
of audio per second, the time to first audio of every session, and the device time of the whole stream relative to one
batched forward of the same S utterances.  The same schedule is then run with every request widened to its whole window
(all samples of each window computed, the requested ones kept), which shows what the per-launch row cropping buys.
The card name and power limit are read with nvidia-smi in the same run.  Aborts if the streamed audio differs from the
whole-utterance audio by more than 1e-5 (the whole call may take the two-sub-tile variant of the 128-channel stage,
which rounds differently in the last bits; see DESIGN.md section 5).

    python tools/stream_bench.py --out profiles/r3_stream_bench.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import hifigan_ref as H  # noqa: E402
import tts_cube_b200 as cube  # noqa: E402

SR = 24000
FRAMES_10S = 10 * SR // 240


def load_generator():
    cfg = dict(H.CONFIG_NEB)
    p = os.path.join(ROOT, "oracle", "_ref", "weights", "g_00600000")
    if os.path.exists(p):
        sd = torch.load(p, map_location="cpu", weights_only=False)
        sd, trained = (sd["generator"] if isinstance(sd, dict) and "generator" in sd else sd), True
    else:
        sd, trained = H.random_state_dict(cfg, seed=21, std=0.3, g_scale=0.125), False
    g = cube.CubeGenerator(cfg).to("cuda:0")
    g.load_state_dict(sd)
    return g.eval(), trained


def widened(g):
    """vocode_range that computes every sample of each window and keeps the requested ones"""
    def vr(mel, nf, begin, end):
        full = g.forward_range(mel, nf, [0] * len(nf), [g.out_len(f) for f in nf])
        return [full[b][begin[b]:end[b]] for b in range(len(nf))]
    return vr


def run_streams(g, mels, chunk, start, vocode_range=None):
    S = len(mels)
    streams = [None] * S
    pos = [0] * S
    pieces = [[] for _ in range(S)]
    t_open = [None] * S
    ttfa = [None] * S
    steps = []
    r = 0
    t_begin = time.perf_counter()
    while True:
        live = []
        for i in range(S):
            if r < start[i]:
                continue
            if streams[i] is None:
                streams[i] = g.open_stream()
                t_open[i] = time.perf_counter()
            s = streams[i]
            if s.done:
                continue
            if pos[i] < mels[i].shape[1]:
                s.feed(mels[i][:, pos[i]:pos[i] + chunk])
                pos[i] += chunk
            else:
                s.close_input()
            live.append(i)
        if not live and r >= max(start):
            break
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if vocode_range is None:
            out = g.step_streams([streams[i] for i in live])
        else:
            out = cube.step_streams([streams[i] for i in live], vocode_range, device=g.device)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        steps.append(t1 - t0)
        for i, p in zip(live, out):
            pieces[i].append(p)
            if ttfa[i] is None and p.numel():
                ttfa[i] = t1 - t_open[i]
        r += 1
    wall = time.perf_counter() - t_begin
    return [torch.cat(p) for p in pieces], steps, ttfa, wall


def whole_time(g, mb, reps=5):
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        y = g(mb)
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return sorted(ts)[len(ts) // 2], y


def stats(steps):
    s = sorted(steps)
    return {"mean_ms": 1e3 * sum(s) / len(s), "p95_ms": 1e3 * s[min(len(s) - 1, int(0.95 * len(s)))], "n": len(s)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--sessions", default="1,16,64")
    ap.add_argument("--chunks", default="11,23,46,92")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("stream_bench needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    g, trained = load_generator()
    res = {"gpu": smi[0] if smi else "unknown", "weights": "trained" if trained else "seeded", "utterance_s": 10,
           "frames": FRAMES_10S, "hop": g.hop, "runs": []}
    with torch.no_grad():
        for S in [int(v) for v in a.sessions.split(",")]:
            mb = torch.cat([H.synthetic_mel(1, FRAMES_10S, seed=100 + i) for i in range(S)]).to("cuda:0")
            mels = [mb[i] for i in range(S)]
            t_whole, y = whole_time(g, mb)
            for chunk in [int(v) for v in a.chunks.split(",")]:
                start = [(i * 3) % 8 for i in range(S)]                # staggered starts
                run_streams(g, [m[:, :200] for m in mels[:2]], chunk, start[:2])   # warm-up of the step shapes
                row = {"sessions": S, "chunk_frames": chunk, "whole_forward_ms": 1e3 * t_whole}
                for tag, vr in (("cropped", None), ("widened", widened(g))):
                    got, steps, ttfa, wall = run_streams(g, mels, chunk, start, vr)
                    diff = max(float((got[i] - y[i, 0]).abs().max()) for i in range(S))
                    exact = all(torch.equal(got[i], y[i, 0]) for i in range(S))
                    if diff > 1e-5 or any(got[i].numel() != y.shape[-1] for i in range(S)):
                        sys.exit(f"streamed audio differs from the whole-utterance audio: S={S} chunk={chunk} {tag} max|d|={diff}")
                    st = stats(steps)
                    row[tag] = {**st, "device_s": sum(steps), "vs_whole_forward": sum(steps) / t_whole,
                                "audio_s_per_s": S * 10.0 / wall, "ttfa_ms": [round(1e3 * t, 3) for t in ttfa],
                                "ttfa_mean_ms": 1e3 * sum(ttfa) / S, "bit_exact_vs_whole": exact, "max_abs_diff": diff}
                row["cropping_speedup"] = row["widened"]["device_s"] / row["cropped"]["device_s"]
                res["runs"].append(row)
                print(json.dumps({k: (v if not isinstance(v, dict) else {kk: vv for kk, vv in v.items() if kk != "ttfa_ms"})
                                  for k, v in row.items()}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
