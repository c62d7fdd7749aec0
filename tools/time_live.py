"""Time TableTennisPipeline.live against predict: S simulated cameras push synthetic 1080p frames (numpy, pageable memory) on a host
clock at a given fps, and each camera's 50-frame rallies end on schedule.

  latency : one camera at --fps; per rally, the time from the end_rally call to its result on the host (spin synchronised, positions
            already there), then predict on the same 50 frames at rally end, timed the same way; results compared bit for bit.
  k       : frames/s of one camera pushing as fast as it can (no clock), one frame per push, for several k (ready stacks per pass).
  max_fps : for S = 1, 2, 4 the largest per-camera fps of a ladder at which the pushes keep to the camera clock: the 95th percentile
            of (push returns - frame due) stays below one frame interval.  Rally ends are staggered over the cameras; the end_rally
            calls run on the same host thread, so their latency counts against the clock too.
Pipeline: WASB main + aux at 1280x704, HRNet main + aux (tf32), uplift (tf32x3) -- bench.py's pipeline leg.  Writes one JSON file.

    python tools/time_live.py --out profiles/r06_live_timing.json
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))
from time_clips import write_checkpoints      # noqa: E402  (tools/ is the script's directory)

RALLY = 50


def wait_until(t):
    d = t - time.perf_counter()
    if d > 0:
        time.sleep(d)


def latency(pipe, pool, fps, rallies):
    """One camera at fps: end_rally -> host result, and predict on the same rally at its end."""
    live_ms, predict_ms, same = [], [], True
    with pipe.live(fps) as live:
        for r in range(rallies + 1):                            # rally 0 warms up
            frames = [pool[(r * RALLY + j) % len(pool)] for j in range(RALLY)]
            t0 = time.perf_counter()
            for j, f in enumerate(frames):
                wait_until(t0 + j / fps)
                live.push(0, f)
            wait_until(t0 + RALLY / fps)
            t = time.perf_counter()
            got = live.end_rally(0)
            torch.cuda.synchronize()
            t_live = time.perf_counter() - t
            torch.cuda.synchronize()
            t = time.perf_counter()
            want = pipe.predict(frames, fps)
            torch.cuda.synchronize()
            t_pred = time.perf_counter() - t
            same &= bool(torch.equal(got[0], want[0]) and np.array_equal(got[1], want[1]))
            if r:
                live_ms.append(t_live * 1e3)
                predict_ms.append(t_pred * 1e3)
    stat = lambda v: {'median': float(np.median(v)), 'p99': float(np.percentile(v, 99)), 'all': v}
    return {'fps': fps, 'rallies': rallies, 'frames_per_rally': RALLY, 'end_rally_ms': stat(live_ms), 'predict_ms': stat(predict_ms),
            'identical_to_predict': same}


def throughput(pipe, pool, k, rallies):
    with pipe.live(50.0, k=k) as live:
        def run(n):
            for r in range(n):
                for j in range(RALLY):
                    live.push(0, pool[(r * RALLY + j) % len(pool)])
                live.end_rally(0)
            torch.cuda.synchronize()
        run(1)
        t = time.perf_counter()
        run(rallies)
        dt = time.perf_counter() - t
    return {'k': k, 'frames': rallies * RALLY, 'frames_per_s': rallies * RALLY / dt}


def paced(pipe, pool, streams, fps, rallies):
    """S cameras at fps, one frame each per tick, rally ends staggered; returns the push lags (s) and the push durations (s)."""
    lags, durs, refused = [], [], [0]
    ticks = rallies * RALLY
    offset = [s * RALLY // streams for s in range(streams)]
    with pipe.live(fps, streams=streams) as live:
        t0 = time.perf_counter() + 0.05
        for t in range(ticks):
            due = t0 + t / fps
            wait_until(due)
            for s in range(streams):
                a = time.perf_counter()
                live.push(s, pool[(t * streams + s) % len(pool)])
                b = time.perf_counter()
                lags.append(b - due)
                durs.append(b - a)
                if (t + offset[s]) % RALLY == RALLY - 1 or t == ticks - 1:
                    try:
                        live.end_rally(s)
                    except ValueError:      # a rally predict would refuse: timed like any other
                        refused[0] += 1
        torch.cuda.synchronize()
    return np.array(lags), np.array(durs), refused[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--fps', type=float, default=60.0)
    ap.add_argument('--rallies', type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('time_live.py measures on a GPU; none is visible')
    from upliftingtabletennis_b200 import synthetic
    from upliftingtabletennis_b200.interface import TableTennisPipeline
    from upliftingtabletennis_b200.live import DEFAULT_K, DEFAULT_SLOTS
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True).stdout
    hub = tempfile.mkdtemp(prefix='ttk_live_hub_')
    torch.hub.set_dir(hub)
    write_checkpoints(hub)
    pipe = TableTennisPipeline(ball_model='wasb', ball_model_aux='wasb', table_model='hrnet', table_model_aux='hrnet')
    pool = list(synthetic.frames_1080p(128, seed=11))
    result = {'gpus': [l.strip() for l in q.strip().splitlines()], 'default_k': DEFAULT_K, 'default_slots': DEFAULT_SLOTS,
              'pipeline': 'WASB main + aux at 1280x704 (tf32), HRNet main + aux (tf32), uplift (tf32x3); 1080p numpy frames'}
    result['latency'] = latency(pipe, pool, args.fps, args.rallies)
    print('latency', json.dumps({k: v for k, v in result['latency'].items()}), flush=True)
    result['k'] = [throughput(pipe, pool, k, 4) for k in (4, 8, 16, 32)]
    print('k', json.dumps(result['k']), flush=True)
    ladder = (30, 60, 90, 120, 150, 180, 240)
    result['max_fps'] = {}
    for streams in (1, 2, 4):
        best, trials = None, []
        for fps in ladder:
            lags, durs, refused = paced(pipe, pool, streams, fps, 3)
            ok = bool(np.percentile(lags, 95) < 1.0 / fps)
            trials.append({'fps': fps, 'sustained': ok, 'lag_ms_p50': float(np.median(lags) * 1e3),
                           'lag_ms_p95': float(np.percentile(lags, 95) * 1e3), 'lag_ms_max': float(lags.max() * 1e3),
                           'push_ms_p50': float(np.median(durs) * 1e3), 'push_ms_p99': float(np.percentile(durs, 99) * 1e3),
                           'refused_rallies': refused})
            print('streams', streams, json.dumps(trials[-1]), flush=True)
            if not ok:
                break
            best = fps
        result['max_fps'][str(streams)] = {'per_camera_fps': best, 'ladder': list(ladder), 'trials': trials}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(result, f, indent=1)


if __name__ == '__main__':
    main()
