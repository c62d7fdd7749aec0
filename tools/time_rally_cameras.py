"""Time the rally cameras: TableTennisPipeline.predict_clips(..., cameras=True) against the workflow a user of the reference runs to
draw the predicted trajectory onto the video, in one process on one GPU, arms alternating, medians reported.

  cameras  : pipe.predict_clips(clips, fps, cameras=True)
  workflow : per clip pipe.predict, pipe.table_detector.predict and pipe.table_detector_aux.predict (the two table passes predict
             already ran), pipe.table_detector.filter_trajectory, pipe.calibrate_camera and pipe.reproject
  plain    : pipe.predict_clips(clips, fps), for the cost the cameras add

Workload: 64 clips of 50 synthetic 1080p numpy frames (BASELINE configs[4]), every clip its own frames.  Pipeline: the default
composition's main detectors, ViTPose at 1152x640 (tf32x3), for the ball and the table, and the uplifting transformer.  Each auxiliary
detector is a second ViTPose with the main one's weights: with synthetic weights the default WASB / HRNet auxiliaries never agree with
ViTPose, and a rally without agreeing detections has neither a trajectory nor visible table keypoints, so there would be nothing to
calibrate or draw.  The records of the cameras arm are compared field by field with the workflow's results.  Writes one JSON file with
the GPU's name, power limit and SM clocks read in the same run.

    python tools/time_rally_cameras.py --out profiles/r08_rally_cameras_timing.json [--reps 3] [--clips 64]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, '..'))
sys.path.insert(0, HERE)

from time_clips import make_clips, timed, write_checkpoints     # noqa: E402
from time_live import VIT_RES, write_vitpose_checkpoints       # noqa: E402

FPS = 50.0


def workflow(pipe, clips):
    out = []
    for c in clips:
        spin, pos = pipe.predict(c, FPS)
        tk, _ = pipe.table_detector.predict(c, return_heatmaps=False)
        tk_aux, _ = pipe.table_detector_aux.predict(c, return_heatmaps=False)
        kp = pipe.table_detector.filter_trajectory(tk, tk_aux)
        try:
            mint, mext = pipe.calibrate_camera(kp)
        except (AssertionError, ValueError) as e:
            out.append((spin, pos, kp, None, None, None, str(e)))
            continue
        out.append((spin, pos, kp, mint, mext, pipe.reproject(pos, mint, mext), None))
    return out


def bits(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def same(cams, ref):
    """The cameras arm's records against the workflow's results, bit for bit."""
    if len(cams) != len(ref):
        return False
    for (spin, pos, cam), (rspin, rpos, kp, mint, mext, ball_2d, error) in zip(cams, ref):
        if not (torch.equal(spin.cpu(), rspin.cpu()) and np.array_equal(pos, rpos) and cam.error == error):
            return False
        for a, b in ((cam.keypoints, kp), (cam.Mint, mint), (cam.Mext, mext), (cam.ball_2d, ball_2d)):
            if (a is None) != (b is None) or (a is not None and not np.array_equal(bits(a), bits(b))):
                return False
    return True


def gpu_state():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.sm,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout
    return [line.strip() for line in q.strip().splitlines()]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--clips', type=int, default=64)
    ap.add_argument('--frames', type=int, default=50)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('time_rally_cameras.py measures on a GPU; none is visible')
    from upliftingtabletennis_b200 import synthetic
    from upliftingtabletennis_b200.interface import TableTennisPipeline
    hub = tempfile.mkdtemp(prefix='ttk_cameras_hub_')
    torch.hub.set_dir(hub)
    write_checkpoints(hub)
    write_vitpose_checkpoints(hub)
    pipe = TableTennisPipeline(ball_model='vitpose', ball_model_aux='vitpose', table_model='vitpose', table_model_aux='vitpose')
    clips = make_clips([args.frames] * args.clips, synthetic.frames_1080p(64, seed=11))
    arms = {'cameras': lambda: pipe.predict_clips(clips, FPS, cameras=True),
            'workflow': lambda: workflow(pipe, clips),
            'plain': lambda: pipe.predict_clips(clips, FPS)}
    results = {name: timed(fn)[1] for name, fn in arms.items()}           # warm-up of every arm
    times = {name: [] for name in arms}
    states = [gpu_state()]
    for _ in range(args.reps):                                              # arms alternate
        for name, fn in arms.items():
            times[name].append(timed(fn)[0])
        states.append(gpu_state())
    med = {name: float(np.median(ts)) for name, ts in times.items()}
    cams = results['cameras']
    errors = {}
    for _, _, cam in cams:
        errors[cam.error or 'calibrated'] = errors.get(cam.error or 'calibrated', 0) + 1
    result = {
        'gpu_state': states,         # name, power limit, SM clock, max SM clock: before the timed reps and after each
        'device_count': torch.cuda.device_count(), 'reps': args.reps, 'clips': args.clips, 'frames_per_clip': args.frames,
        'pipeline': 'ViTPose main + aux (same weights) for ball and table at %dx%d (tf32x3), uplift (tf32x3); 1080p numpy frames' % VIT_RES,
        'identical_to_workflow': same(cams, results['workflow']),
        'plain_equals_cameras': all(torch.equal(a[0], b[0]) and np.array_equal(a[1], b[1]) for a, b in zip(results['plain'], cams)),
        'calibration_outcomes': errors,
        'median_ms': med, 'all_ms': times,
        'workflow_over_cameras': med['workflow'] / med['cameras'],
        'cameras_added_ms': med['cameras'] - med['plain'],
        'cameras_added_ms_per_clip': (med['cameras'] - med['plain']) / args.clips,
    }
    print(json.dumps({k: v for k, v in result.items() if k != 'all_ms'}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(result, f, indent=1)


if __name__ == '__main__':
    main()
