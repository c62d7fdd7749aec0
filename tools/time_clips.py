"""Time TableTennisPipeline.predict_clips against the per-clip predict loop, in one process, arms alternating, medians reported.

Workloads (1080p numpy frames in pageable memory, every clip its own frames, WASB main + aux at 1280x704, HRNet main + aux, the
uplifting transformer; main and auxiliary detectors share their weights so that every ball stack agrees):
  rally : BASELINE configs[4], 64 clips of 50 frames
  short : 64 clips of 12 to 49 frames
On one GPU: [pipe.predict(c, fps) for c in clips] against pipe.predict_clips(clips, fps); then predict_clips over 1, 2, 4 and 8 devices
(those that exist) and over two replicas on GPU 0 (devices=[0, 0]).  Results of the two arms are compared bit for bit.  Writes one JSON file.
--timestamps: instead, the rally workload on one GPU through predict_clips with fps against predict_clips with per-frame capture
timestamps (fps=None, stamps (k - 1) / fps, so that both arms must return the same bits).
--known-table: instead, the rally workload on one GPU through predict_clips with the table detected against predict_clips with each
clip's own filtered keypoints given as table_keypoints (so that both arms must return the same bits).  --pipeline wasb-hrnet is the
pipeline above; vitpose is ViTPose at 1152x640 (tf32x3) for all four detectors, each auxiliary sharing its main detector's weights
(as tools/time_rally_cameras.py runs it).

    python tools/time_clips.py --out profiles/r05_clips_timing.json [--reps 5]
    python tools/time_clips.py --timestamps --out profiles/r09_timestamps_timing.json [--reps 9]
    python tools/time_clips.py --known-table --pipeline vitpose --out known_table_vitpose.json [--reps 5]
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

RES = (1280, 704)


def write_checkpoints(hub):
    from upliftingtabletennis_b200 import synthetic
    from upliftingtabletennis_b200.detector import HRNetEngine
    from upliftingtabletennis_b200.uplift import get_model
    w = os.path.join(hub, 'checkpoints', 'tt_uplifting_extracted', 'weights')
    up = get_model('connectstage', 'large', 'dynamic', 'new')
    for sub, sd, info in (
            ('inference_balldetection/wasb', synthetic.hrnet_blob_state_dict(HRNetEngine(9, 3, 1, 1).state_dict_layout(), seed=1),
             {'model_name': 'wasb', 'image_resolution': RES, 'in_frames': 3, 'lr': 0.0}),
            ('inference_tabledetection/hrnet', synthetic.hrnet_state_dict(HRNetEngine(3, 13, 0, 13).state_dict_layout(), seed=2),
             {'model_name': 'hrnet', 'image_resolution': RES}),
            ('inference_uplifting/ours', synthetic.uplift_state_dict(up, seed=3),
             {'name': 'connectstage', 'size': 'large', 'tabletoken_mode': 'dynamic', 'time_rotation': 'new', 'transform_mode': 'global',
              'randdet_prob': 0.0, 'randmiss_prob': 0.0, 'tablemiss_prob': 0.0})):
        os.makedirs(os.path.join(w, sub), exist_ok=True)
        torch.save({'model_state_dict': sd, 'identifier': 'synthetic', 'additional_info': info}, os.path.join(w, sub, 'model.pt'))


def make_clips(lengths, pool):
    """Clips of distinct frames (copies of a pool of synthetic frames): every frame is its own host memory, as in a decoded video."""
    out, k = [], 0
    for n in lengths:
        out.append([pool[(k + j) % len(pool)].copy() for j in range(n)])
        k += n
    return out


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3, r


def same(a, b):
    return len(a) == len(b) and all(torch.equal(s.cpu(), s2.cpu()) and np.array_equal(p, p2) for (s, p), (s2, p2) in zip(a, b))


def time_timestamps(pipe, clips, reps):
    """predict_clips(clips, fps) against predict_clips(clips, None, timestamps=...) on one GPU, arms alternating."""
    fps = 50.0
    stamps = [(np.arange(len(c), dtype=np.float64) - 1) / fps for c in clips]
    plain = lambda: pipe.predict_clips(clips, fps)
    stamped = lambda: pipe.predict_clips(clips, None, timestamps=stamps)
    _, want = timed(plain)                                        # warm-up of both arms
    _, got = timed(stamped)
    t_fps, t_stamps = [], []
    for _ in range(reps):
        t_fps.append(timed(plain)[0])
        t_stamps.append(timed(stamped)[0])
    return {'clips': len(clips), 'frames': sum(len(c) for c in clips), 'identical': same(got, want),
            'fps_ms': float(np.median(t_fps)), 'timestamps_ms': float(np.median(t_stamps)),
            'fps_ms_spread': [float(min(t_fps)), float(max(t_fps))], 'timestamps_ms_spread': [float(min(t_stamps)), float(max(t_stamps))],
            'fps_ms_all': t_fps, 'timestamps_ms_all': t_stamps}


def time_known_table(pipe, clips, reps):
    """predict_clips(clips, fps) against predict_clips(clips, fps, table_keypoints=each clip's own keypoints) on one GPU, arms
    alternating."""
    fps = 50.0
    tables = [cam.keypoints for _, _, cam in pipe.predict_clips(clips, fps, cameras=True)]
    detected = lambda: pipe.predict_clips(clips, fps)
    known = lambda: pipe.predict_clips(clips, fps, table_keypoints=tables)
    _, want = timed(detected)                                     # warm-up of both arms
    _, got = timed(known)
    t_detected, t_known = [], []
    for _ in range(reps):
        t_detected.append(timed(detected)[0])
        t_known.append(timed(known)[0])
    med_d, med_k = float(np.median(t_detected)), float(np.median(t_known))
    return {'clips': len(clips), 'frames': sum(len(c) for c in clips), 'identical': same(got, want),
            'visible_keypoints_per_clip': sorted({int(k[:, 2].sum()) for k in tables}),
            'detected_ms': med_d, 'known_table_ms': med_k, 'detected_over_known': med_d / med_k,
            'detected_ms_spread': [float(min(t_detected)), float(max(t_detected))],
            'known_table_ms_spread': [float(min(t_known)), float(max(t_known))],
            'detected_ms_all': t_detected, 'known_table_ms_all': t_known}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--timestamps', action='store_true', help='time predict_clips with per-frame stamps against fps (rally workload)')
    ap.add_argument('--known-table', action='store_true', help='time predict_clips with known tables against detected ones (rally workload)')
    ap.add_argument('--pipeline', choices=('wasb-hrnet', 'vitpose'), default='wasb-hrnet', help='the pipeline of --known-table')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('time_clips.py measures on a GPU; none is visible')
    from upliftingtabletennis_b200 import synthetic
    from upliftingtabletennis_b200.interface import TableTennisPipeline
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True).stdout
    hub = tempfile.mkdtemp(prefix='ttk_clips_hub_')
    torch.hub.set_dir(hub)
    write_checkpoints(hub)
    pipe = TableTennisPipeline(ball_model='wasb', ball_model_aux='wasb', table_model='hrnet', table_model_aux='hrnet')
    pool = synthetic.frames_1080p(64, seed=11)
    rng = np.random.default_rng(5)
    workloads = {'rally': [50] * 64, 'short': [int(n) for n in rng.integers(12, 50, 64)]}
    result = {'gpus': [l.strip() for l in q.strip().splitlines()], 'device_count': torch.cuda.device_count(), 'reps': args.reps,
              'pipeline': 'WASB main + aux at %dx%d (tf32), HRNet main + aux (tf32), uplift (tf32x3); 1080p numpy frames' % RES,
              'workloads': {}}
    if args.known_table:
        if args.pipeline == 'vitpose':
            from time_live import VIT_RES, write_vitpose_checkpoints
            write_vitpose_checkpoints(hub)
            pipe = TableTennisPipeline(ball_model='vitpose', ball_model_aux='vitpose', table_model='vitpose', table_model_aux='vitpose')
            result['pipeline'] = 'ViTPose main + aux (same weights) for ball and table at %dx%d (tf32x3), uplift (tf32x3); 1080p numpy frames' % VIT_RES
        result['known_table'] = time_known_table(pipe, make_clips(workloads['rally'], pool), args.reps)
        print('known_table', json.dumps({k: v for k, v in result['known_table'].items() if not k.endswith('_all')}), flush=True)
        result['gpus_after'] = [l.strip() for l in subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                                                                  capture_output=True, text=True).stdout.strip().splitlines()]
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(result, f, indent=1)
        return
    if args.timestamps:
        result['timestamps'] = time_timestamps(pipe, make_clips(workloads['rally'], pool), args.reps)
        print('timestamps', json.dumps({k: v for k, v in result['timestamps'].items() if not k.endswith('_all')}), flush=True)
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(result, f, indent=1)
        return
    for name, lengths in workloads.items():
        clips = make_clips(lengths, pool)
        frames = sum(lengths)
        loop = lambda: [pipe.predict(c, 50.0) for c in clips]
        batched = lambda: pipe.predict_clips(clips, 50.0)
        _, want = timed(loop)                                     # warm-up of both arms
        _, got = timed(batched)
        t_loop, t_clips = [], []
        for _ in range(args.reps):                                # arms alternate
            t_loop.append(timed(loop)[0])
            t_clips.append(timed(batched)[0])
        entry = {'clips': len(lengths), 'frames': frames, 'identical': same(got, want),
                 'predict_loop_ms': float(np.median(t_loop)), 'predict_clips_ms': float(np.median(t_clips)),
                 'predict_loop_ms_all': t_loop, 'predict_clips_ms_all': t_clips}
        entry['speedup'] = entry['predict_loop_ms'] / entry['predict_clips_ms']
        entry['predict_clips_frames_per_s'] = frames / (entry['predict_clips_ms'] * 1e-3)
        devs = {}
        # 1, 2, 4, 8 GPUs (those that exist), and two replicas on GPU 0: two launcher threads sharing one device
        for name_k, ds in [(str(k), list(range(k))) for k in (1, 2, 4, 8) if k <= torch.cuda.device_count()] + [('0,0', [0, 0])]:
            fn = lambda: pipe.predict_clips(clips, 50.0, devices=ds)
            _, r = timed(fn)
            ts = [timed(fn)[0] for _ in range(args.reps)]
            devs[name_k] = {'ms': float(np.median(ts)), 'ms_all': ts, 'frames_per_s': frames / (float(np.median(ts)) * 1e-3),
                            'identical': same(r, want)}
        entry['devices'] = devs
        result['workloads'][name] = entry
        print(name, json.dumps({k: v for k, v in entry.items() if not k.endswith('_all')}), flush=True)
        del clips
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(result, f, indent=1)


if __name__ == '__main__':
    main()
