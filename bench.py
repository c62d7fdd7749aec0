"""Benchmark of the hot path (BASELINE.json: frames/sec end-to-end + uplift trajectories/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dtype tf32|bf16|fp32] [--legs ...] [--dump-outputs DIR]

A step = one pass of ball-detect + decode over one batch of 32 synthetic 1920x1080 three-frame stacks
(BASELINE.json configs[1]): fused resize/normalise/stack -> WASB heatmap network -> argmax + sub-pixel decode.
The headline runs at the API's default arithmetic class, TF32 on the tcgen05 tensor cores with fp32 activations (the class of
the reference's cuDNN convolutions on a GPU); the bf16 path is reported separately under "bf16", and "parity" states how both
compare with the strict fp32 path on the very batch that is timed.
`value` counts frames (= stacks) per second with the uint8 frames already resident in HBM; `e2e` is the same metric through
the hub API (`hubconf.ball_detection('wasb').predict(triples)`) the way a user of the reference calls it: numpy frames in
pageable host memory, every triple made of copies, heatmaps and positions returned as numpy (other input styles as sub-keys).
Same run: "uplift" (configs[3]: 50 000 trajectories sharded over the ranks), "pipeline" (configs[2]), "clips" (configs[4]:
64 clips sharded over the ranks, NCCL gather of the per-clip records), "vitpose", "calibration", "gpu_eager_baseline" (stock
PyTorch on the same GPU) and "cpu_baseline" (oracle port on the host cores).
Multi-GPU: clips are independent, every rank processes its own batch (weak scaling) and NCCL gathers the
per-stack results; time = max over ranks.  `--impl reference` times the CPU oracle port of the reference's
path on the host cores (the reference is Python and cannot travel to the GPU box; see DESIGN.md).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH = 32                 # stacks per step (BASELINE.json configs[1])
RES = (1280, 704)          # WASB input resolution (balldetection/config.py:84-85)
SRC = (1080, 1920)
WASB_GFLOP_PER_STACK = 344.07        # SURVEY.md section 8d (2*MAC, convs only)
UPLIFT_GFLOP_PER_TRAJ = 0.753
UPLIFT_TOTAL = 50000        # BASELINE.json configs[3]
UPLIFT_CHUNK = 4096         # trajectories per library call
N_CLIPS, N_BASE_CLIPS = 64, 4   # BASELINE.json configs[4]: 64 clips (4 distinct synthetic ones, repeated)
VIT_RES = (1152, 640)      # ViTPose input resolution (balldetection/config.py:82-83)
VIT_GFLOP_PER_STACK = 313.5          # SURVEY.md section 8d
VIT_BATCH = 16
CALIB_CLIPS = 64
CLIP_FRAMES = 300          # BASELINE.json configs[2]: full hub pipeline on a synthetic 300-frame clip
RALLY_FRAMES = 50          # ... processed as rallies of 50 frames (see the pipeline leg)
WORKLOAD = 'configs[1]: WASB ball-detect (1280x704 input, 344 GFLOP/stack) + heatmap decode on synthetic 1920x1080 3-frame stacks, batch %d per GPU' % BATCH


def dump_outputs(out_dir, pos, heat):
    """Write what the last timed step returned, so that two builds can be compared output for output on identical seeded
    inputs: the decoded (x, y, 1) of every stack (float64) and the heatmaps of every fourth stack (float32; all 32 would be
    115 MB), with the indices of those stacks."""
    os.makedirs(out_dir, exist_ok=True)
    stacks = np.arange(0, heat.shape[0], 4)
    np.save(os.path.join(out_dir, 'positions.npy'), pos.reshape(-1, 3).cpu().numpy().astype(np.float64))
    np.save(os.path.join(out_dir, 'heatmaps.npy'), heat[::4].cpu().numpy().astype(np.float32))
    np.save(os.path.join(out_dir, 'heatmap_stacks.npy'), stacks.astype(np.float64))


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return {'hbm_gbs': d['hbm_gbs'], 'bf16_tflops': d['bf16_tflops'], 'bf16_tflops_sustained': d.get('bf16_tflops_sustained', d['bf16_tflops']),
                'source': 'measured (MEASURED_PEAKS.json)'}
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0, 'source': 'fallback (B200_PROFILING.md)'}


def ncu_traffic(kernel_name, images_per_launch):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed ncu --set full
    capture (profiles/ncu_traffic.json, written by tools/ncu_summary.py); None if that kernel was not captured."""
    p = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    if not os.path.exists(p):
        return None
    rec = json.load(open(p)).get(kernel_name)
    if not rec:
        return None
    # the capture ran a smaller sub-batch per launch than the bench does: DRAM traffic of these streaming kernels scales with the images
    return rec['dram_bytes_per_launch'] * images_per_launch / rec.get('images_per_launch', images_per_launch)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = 'index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace('.', '').isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 8 and r[4 + i].lower().startswith('active') for r in self.rows)]
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': reasons,
                'samples': len(sm)}


def make_checkpoints(hub_dir):
    """Synthetic weights tree in the reference's checkpoint format so that the hub API can be used as a user would."""
    from upliftingtabletennis_b200 import synthetic
    from upliftingtabletennis_b200.detector import HRNetEngine
    from upliftingtabletennis_b200.uplift import get_model
    w = os.path.join(hub_dir, 'checkpoints', 'tt_uplifting_extracted', 'weights')
    wasb_sd = synthetic.hrnet_blob_state_dict(HRNetEngine(9, 3, 1, 1).state_dict_layout(), seed=1)
    up = get_model('connectstage', 'large', 'dynamic', 'new')
    up_sd = synthetic.uplift_state_dict(up, seed=3)
    for sub, sd, info in (('inference_balldetection/wasb', wasb_sd, {'model_name': 'wasb', 'image_resolution': RES, 'in_frames': 3, 'lr': 0.0}),
                          ('inference_uplifting/ours', up_sd, {'name': 'connectstage', 'size': 'large', 'tabletoken_mode': 'dynamic',
                                                               'time_rotation': 'new', 'transform_mode': 'global', 'randdet_prob': 0.0,
                                                               'randmiss_prob': 0.0, 'tablemiss_prob': 0.0})):
        d = os.path.join(w, sub)
        os.makedirs(d, exist_ok=True)
        torch.save({'model_state_dict': sd, 'identifier': 'synthetic', 'additional_info': info}, os.path.join(d, 'model.pt'))
    table_sd = synthetic.hrnet_state_dict(HRNetEngine(3, 13, 0, 13).state_dict_layout(), seed=2)
    d = os.path.join(w, 'inference_tabledetection', 'hrnet')
    os.makedirs(d, exist_ok=True)
    torch.save({'model_state_dict': table_sd, 'identifier': 'synthetic', 'additional_info': {'model_name': 'hrnet', 'image_resolution': RES}},
               os.path.join(d, 'model.pt'))
    from upliftingtabletennis_b200 import vitpose
    vit_sd = synthetic.vit_state_dict(vitpose.state_dict_layout(9, 2880, 1), seed=5)
    d = os.path.join(w, 'inference_balldetection', 'vitpose')
    os.makedirs(d, exist_ok=True)
    torch.save({'model_state_dict': vit_sd, 'identifier': 'synthetic',
                'additional_info': {'model_name': 'vitpose', 'image_resolution': VIT_RES, 'in_frames': 3, 'lr': 0.0}}, os.path.join(d, 'model.pt'))
    return wasb_sd, up_sd, table_sd


def cpu_reference_step(wasb_sd, frames, n_stacks):
    """The reference's path restated on the CPU (oracle port): transform -> WASB forward -> decode, B=1 per stack like
    interface.py:102-119.  Returns seconds."""
    from oracle import decode as odec, hrnet as ohr, preprocess as opre
    t0 = time.perf_counter()
    for s in range(n_stacks):
        x = opre.preprocess_stack([frames[s], frames[s + 1], frames[s + 2]], RES[0], RES[1])
        hm = ohr.wasb_forward(wasb_sd, torch.from_numpy(x)[None]).numpy()
        odec.decode_heatmaps(hm[:, 0], SRC[1], SRC[0], odec.TABLE)
    return time.perf_counter() - t0


def gpu_eager_baseline(dev, steps=3, warmup=2, wasb_sub=8, uplift_batch=4096):
    """SURVEY.md section 2a's bar: stock PyTorch eager on the SAME B200 for the two network stages, i.e. what the reference's
    code does on a GPU (cuDNN convolutions + ATen batch norm / ReLU / add kernels, cuBLAS + SDPA for the transformer).  The
    reference's modules cannot travel to the GPU box, so the functional restatement in oracle/ is moved to CUDA as it is --
    same F.conv2d / F.batch_norm / F.linear / F.scaled_dot_product_attention calls.  Modes: torch defaults (cuDNN TF32 on,
    matmul fp32), strict fp32 (TF32 off), and bf16 channels-last / bf16 autocast-free weights."""
    from oracle import hrnet as ohr, uplift as oup
    from upliftingtabletennis_b200 import synthetic
    out = {}

    def timed(fn, n_units):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return n_units * steps / (e0.elapsed_time(e1) * 1e-3)

    sd = {k: v.to(dev) for k, v in synthetic.hrnet_blob_state_dict(ohr.state_dict_layout(9, 3), seed=1).items()}
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.randn((wasb_sub, 9, RES[1], RES[0]), device=dev, generator=g)
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.benchmark = True
    try:
        wasb = {}
        torch.backends.cudnn.allow_tf32 = True
        wasb['tf32_default'] = timed(lambda: ohr.wasb_forward(sd, x), wasb_sub)
        xcl = x.contiguous(memory_format=torch.channels_last)
        wasb['tf32_channels_last'] = timed(lambda: ohr.wasb_forward(sd, xcl), wasb_sub)
        torch.backends.cudnn.allow_tf32 = False
        wasb['fp32_strict'] = timed(lambda: ohr.wasb_forward(sd, x), wasb_sub)
        torch.backends.cudnn.allow_tf32 = True
        sd16 = {k: (v.to(torch.bfloat16) if v.is_floating_point() else v) for k, v in sd.items()}
        x16 = x.to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
        wasb['bf16_channels_last'] = timed(lambda: ohr.wasb_forward(sd16, x16), wasb_sub)
        out['wasb_forward'] = {'unit': 'stacks/s', 'sub_batch': wasb_sub, **wasb,
                               'note': 'network only (no resize / decode), %dx%d input, cudnn.benchmark on' % RES}
        del sd16, x16, xcl, x
        usd = {k: v.to(dev) for k, v in oup.random_state_dict(3).items()}
        ua = [torch.from_numpy(a).to(dev) for a in synthetic.trajectories(uplift_batch, seed=7)]
        up = {}
        for b in (512, uplift_batch):
            ub = [a[:b] for a in ua]
            up['fp32_sdpa_b%d' % b] = timed(lambda: oup.uplift_forward(usd, *ub, sdpa=True), b)
        usd16 = {k: v.to(torch.bfloat16) for k, v in usd.items()}
        ub16 = [a.to(torch.bfloat16) for a in ua]
        try:
            up['bf16_sdpa_b%d' % uplift_batch] = timed(lambda: oup.uplift_forward(usd16, *ub16, sdpa=True), uplift_batch)
        except Exception as e:      # noqa: BLE001 - report, the leg is informative only
            up['bf16_sdpa_error'] = str(e)[:200]
        out['uplift_forward'] = {'unit': 'trajectories/s', **up, 'note': 'cuBLAS + SDPA + ATen elementwise, matmul TF32 off (torch default)'}
        del usd, usd16, ua, ub16
        from oracle import vitpose as ovp
        hp, wp = ovp.tokens_hw(VIT_RES[1], VIT_RES[0])
        vsd = {k: v.to(dev) for k, v in ovp.random_state_dict(5, 9, hp * wp, 1).items()}
        vx = torch.randn((4, 9, VIT_RES[1], VIT_RES[0]), device=dev, generator=g)
        vit = {'fp32_default': timed(lambda: ovp.vitpose_forward_native(vsd, vx), 4)}
        torch.backends.cuda.matmul.allow_tf32 = True
        vit['tf32_matmul_opt_in'] = timed(lambda: ovp.vitpose_forward_native(vsd, vx), 4)
        torch.backends.cuda.matmul.allow_tf32 = False
        vsd16 = {k: (v.to(torch.bfloat16) if v.is_floating_point() else v) for k, v in vsd.items()}
        vx16 = vx.to(torch.bfloat16)
        try:
            vit['bf16'] = timed(lambda: ovp.vitpose_forward_native(vsd16, vx16), 4)
        except Exception as e:      # noqa: BLE001 - informative leg
            vit['bf16_error'] = str(e)[:200]
        out['vitpose_forward'] = {'unit': 'stacks/s', 'sub_batch': 4, **vit,
                                  'note': 'network only, %dx%d input; torch defaults = fp32 cuBLAS Linear layers + TF32 cuDNN convolutions' % VIT_RES}
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = old
    torch.cuda.empty_cache()
    return out


def run_reference(args, rank, world):
    if rank != 0:
        return
    # this arm must not map the product library: weights layout from the oracle, synthetic inputs from the pure-numpy generators
    from oracle import hrnet as ohr
    from upliftingtabletennis_b200 import synthetic
    torch.set_num_threads(os.cpu_count())
    sd = synthetic.hrnet_blob_state_dict(ohr.state_dict_layout(9, 3), seed=1)
    per_step = 2
    frames = synthetic.frames_1080p(per_step + 2, seed=100)
    for _ in range(args.warmup):
        cpu_reference_step(sd, frames, 1)
    t = sum(cpu_reference_step(sd, frames, per_step) for _ in range(args.steps))
    v = per_step * args.steps / t
    line = {'impl': 'reference', 'metric': 'frames_per_sec_detect_decode', 'value': v, 'unit': 'frames/s', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * t / args.steps, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'sample': 'each step = %d stacks of that workload, B=1 per forward like interface.py:102-119' % per_step},
            'cpu_baseline': {'value': v, 'unit': 'frames/s', 'cores': torch.get_num_threads(), 'kind': 'port',
                             'sample': '%d steps x %d stacks through oracle/ (numpy resize + CPU torch fp32 WASB + SciPy L-BFGS-B decode)' % (args.steps, per_step)},
            'e2e': {'value': v, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line))


def cpu_uplift_baseline(up_sd):
    """BASELINE.md section 3: the uplifting transformer of the reference restated on the CPU (oracle port), B = 1 and B = 512."""
    from oracle import uplift as oup
    from upliftingtabletennis_b200 import synthetic
    a = [torch.from_numpy(x) for x in synthetic.trajectories(512, seed=7)]
    out = {}
    for b, reps in ((1, 20), (512, 1)):
        ab = [x[:b] for x in a]
        oup.uplift_forward(up_sd, *ab)
        t0 = time.perf_counter()
        for _ in range(reps):
            oup.uplift_forward(up_sd, *ab)
        out['b%d' % b] = b * reps / (time.perf_counter() - t0)
    return out


def cpu_pipeline_baseline(wasb_sd, table_sd, up_sd, frames):
    """BASELINE.md section 3: TableTennisPipeline.predict (interface.py:265-289) chained by hand through oracle/ on a short clip:
    main + auxiliary WASB on every stack, main + auxiliary HRNet on every frame (B = 1 per forward like the reference), both
    decodes, both filters, _uplifting_transform, uplift, spin rotation.  Returns (seconds, frames)."""
    from oracle import decode as odec, hrnet as ohr, preprocess as opre, tails as otl, uplift as oup
    n = len(frames)
    t0 = time.perf_counter()
    bpos = []
    for _model in range(2):
        p = []
        for i in range(1, n - 1):
            x = opre.preprocess_stack([frames[i - 1], frames[i], frames[i + 1]], RES[0], RES[1])
            hm = ohr.wasb_forward(wasb_sd, torch.from_numpy(x)[None]).numpy()
            p.append(odec.decode_heatmaps(hm[:, 0], SRC[1], SRC[0], odec.TABLE)[0][0])
        bpos.append(np.stack(p))
    fpos, _, ftimes = otl.filter_trajectory_ball(bpos[0], bpos[1], 50.0)
    tpos = []
    for _model in range(2):
        p = []
        for i in range(n):
            x = opre.preprocess_stack([frames[i]], RES[0], RES[1])
            hm = ohr.hrnet_forward(table_sd, torch.from_numpy(x)[None]).numpy()
            p.append(odec.decode_heatmaps(hm[0], SRC[1], SRC[0], odec.TABLE)[0])
        tpos.append(np.stack(p))
    table = otl.filter_trajectory_table(tpos[0], tpos[1]).astype(np.float64)
    b, t, ti, m = otl.uplifting_transform(fpos, table, ftimes)
    rot, pos = oup.uplift_forward(up_sd, *(torch.from_numpy(a) for a in (b, t, m, ti)))
    otl.transform_rotationaxes(rot.numpy(), pos.numpy())
    return time.perf_counter() - t0, n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--dtype', default='tf32', choices=['tf32', 'bf16', 'fp32'], help='arithmetic class of the headline (default: the API default)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-eager-baseline', action='store_true')
    ap.add_argument('--legs', default='all', help='comma list of the secondary legs to run: bf16,uplift,vitpose,pipeline,clips,calibration (default all)')
    ap.add_argument('--dump-profile', default='', help='write the per-kernel table of one profiled step to this JSON file')
    ap.add_argument('--dump-outputs', default='', metavar='DIR',
                    help='write what the last timed step returned (positions, a fixed sample of the heatmaps) to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the CUDA path; the reference arm keeps none')
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    if args.impl == 'reference':
        run_reference(args, rank, world)
        return
    legs = set('bf16,uplift,vitpose,pipeline,clips,calibration'.split(',')) if args.legs == 'all' else set(x for x in args.legs.split(',') if x)
    args.warmup = max(args.warmup, 3)
    sub_steps = max(1, min(args.steps, 3))          # secondary legs: fewer repetitions, the default run has to finish within minutes
    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)

    from upliftingtabletennis_b200 import _lib, ops, sharding, synthetic
    # several ranks on one host: waiting host threads sleep instead of spin, so that the cores go to the threads that stage frames
    # (2 cores per GPU on this pool's boxes; INTEGRATION.md).  TTK_HOST_SYNC=spin keeps CUDA's default.
    host_sync = 'spin'
    if int(os.environ.get('LOCAL_WORLD_SIZE', world) or 1) > 1 and os.environ.get('TTK_HOST_SYNC', 'blocking') == 'blocking':
        _lib.host_blocking_sync(local)
        host_sync = 'blocking'

    from upliftingtabletennis_b200._lib import lib
    from upliftingtabletennis_b200.precision import storage_dtype
    hub = tempfile.mkdtemp(prefix='ttk_bench_hub_')
    torch.hub.set_dir(hub)
    wasb_sd, up_sd, table_sd = make_checkpoints(hub)
    import hubconf
    det = hubconf.ball_detection('wasb')              # the API default: TF32 tensor-core path
    api_default = det.model.compute_dtype
    det.model.compute_dtype = args.dtype
    engine = det.model.engine
    W, H = RES

    frames_np = synthetic.frames_1080p(BATCH + 2, seed=100 + rank)
    frames_pinned = torch.from_numpy(frames_np).pin_memory()
    frames_dev = frames_pinned.to(dev)
    heat = torch.empty((BATCH, 1, H, W), dtype=torch.float32, device=dev)
    gathered = torch.empty((world * BATCH, 3), dtype=torch.float64, device=dev) if world > 1 else None
    stage_ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    xbuf = {}

    def step_device(prec, gather=True, mark=False):
        sdt = storage_dtype(prec)
        if sdt not in xbuf:
            xbuf[sdt] = torch.empty((BATCH, H, W, 16), dtype=sdt, device=dev)
        x = xbuf[sdt]
        if mark:
            stage_ev[0].record()
        ops.preprocess_stacks(frames_dev, 3, 1, BATCH, W, H, layout='nhwc16', dtype=sdt, out=x)
        if mark:
            stage_ev[1].record()
        det.model._sync()
        engine.forward_nhwc16(x, out=heat, precision=prec)
        if mark:
            stage_ev[2].record()
        pos = ops.decode_heatmaps(heat, SRC[1], SRC[0], 'table')
        if mark:
            stage_ev[3].record()
        if world > 1 and gather:
            dist.all_gather_into_tensor(gathered, pos.view(BATCH, 3))
        return pos

    # the three ways a caller can hand over 32 (prev, cur, next) triples
    triples_copy = [(frames_np[i].copy(), frames_np[i + 1].copy(), frames_np[i + 2].copy()) for i in range(BATCH)]   # interface.py:275 builds them like this
    triples_view = [(frames_np[i], frames_np[i + 1], frames_np[i + 2]) for i in range(BATCH)]                         # views of one clip array
    triples_pinned = [(frames_pinned[i], frames_pinned[i + 1], frames_pinned[i + 2]) for i in range(BATCH)]

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.barrier()
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    def fps(ms, steps, units=BATCH):
        return world * units * steps / (ms * 1e-3)

    def detector_leg(prec, steps, warmup, full):
        det.model.compute_dtype = prec
        r = {}
        ms = timed(lambda: step_device(prec), steps, warmup)
        r['ms_dev'] = ms
        r['launches'] = 1 + engine.last_launches() + 2
        r['ms_copy_hm'] = timed(lambda: det.predict(triples_copy), steps, warmup)                           # the reference's default call
        r['ms_pinned'] = timed(lambda: det.predict(triples_pinned, return_heatmaps=False), steps, warmup)
        if full:
            r['ms_view'] = timed(lambda: det.predict(triples_view, return_heatmaps=False), steps, warmup)
            r['ms_copy'] = timed(lambda: det.predict(triples_copy, return_heatmaps=False), steps, warmup)
        return r

    last_pos = [None]

    def head_step():
        last_pos[0] = step_device(args.dtype)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    head = {'ms_dev': timed(head_step, args.steps, args.warmup)}
    head['launches'] = 1 + engine.last_launches() + 2
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:           # before anything else overwrites `heat`
        dump_outputs(args.dump_outputs, gathered if world > 1 else last_pos[0], heat)
    head['ms_copy_hm'] = timed(lambda: det.predict(triples_copy), args.steps, args.warmup)
    head['ms_pinned'] = timed(lambda: det.predict(triples_pinned, return_heatmaps=False), args.steps, args.warmup)
    head['ms_view'] = timed(lambda: det.predict(triples_view, return_heatmaps=False), sub_steps, 2)
    head['ms_copy'] = timed(lambda: det.predict(triples_copy, return_heatmaps=False), sub_steps, 2)
    head['ms_view_hm'] = timed(lambda: det.predict(triples_view), sub_steps, 2)
    value = fps(head['ms_dev'], args.steps)

    other = {}
    if 'bf16' in legs:
        for prec in ('tf32', 'bf16'):
            if prec != args.dtype:
                other[prec] = detector_leg(prec, sub_steps, 3, False)
    # output-level parity of the tensor-core paths on this very batch: strict fp32 (SIMT) path as the reference heatmap
    parity = {}
    with torch.no_grad():
        det.model.compute_dtype = 'fp32'
        p32, i32, _ = ops.decode_heatmaps(engine.forward_nhwc16(ops.preprocess_stacks(frames_dev, 3, 1, BATCH, W, H, dtype=torch.float32), out=heat, precision='fp32'),
                                          SRC[1], SRC[0], 'table', return_debug=True)
        h32 = heat.clone()
        scale = float(h32.abs().max())
        top2 = torch.topk(h32.view(BATCH, -1), 2, dim=1).values
        margin = (top2[:, 0] - top2[:, 1]) / scale
        for prec in ('tf32', 'bf16'):
            x = ops.preprocess_stacks(frames_dev, 3, 1, BATCH, W, H, dtype=storage_dtype(prec))
            pp, ii, _ = ops.decode_heatmaps(engine.forward_nhwc16(x, out=heat, precision=prec), SRC[1], SRC[0], 'table', return_debug=True)
            err = float((heat - h32).abs().max()) / scale
            bound = {'tf32': 1e-2, 'bf16': 4e-2}[prec]
            sure = margin > 2 * bound
            d = (pp - p32).view(BATCH, 3)[:, :2].abs().max(dim=1).values
            same = (ii == i32).view(-1)
            parity[prec] = {'heatmap_max_abs_err_over_max': err, 'stated_bound': bound, 'index_match_frac': float(same.float().mean()),
                            'maps_under_margin_rule': int(sure.sum()), 'index_match_under_rule': bool(same[sure].all()) if bool(sure.any()) else None,
                            'max_coord_diff_px': float(d.max()), 'max_coord_diff_px_under_rule': float(d[sure].max()) if bool(sure.any()) else None}
        del h32, x
    det.model.compute_dtype = args.dtype

    # ---- uplift transformer, BASELINE configs[3]: 50 000 synthetic trajectories sharded over the ranks (strong scaling) ----
    up_line = None
    if 'uplift' in legs:
        from upliftingtabletennis_b200.uplift import get_model
        up = get_model('connectstage', 'large', 'dynamic', 'new').to(dev).eval()
        up.load_state_dict(up_sd)
        lo, hi = sharding.shard_range(UPLIFT_TOTAL, rank, world)
        ua = [torch.from_numpy(a[lo:hi]) for a in synthetic.trajectories(UPLIFT_TOTAL, seed=7)]
        ua_p = [a.pin_memory() for a in ua]
        ua_d = [a.to(dev) for a in ua]
        up._sync()
        nloc = hi - lo
        rec_all = torch.empty((world * ((UPLIFT_TOTAL + world - 1) // world), 153), dtype=torch.float32, device=dev) if world > 1 else None

        def up_chunks(args_d, dt):
            rots, poss = [], []
            for c0 in range(0, nloc, UPLIFT_CHUNK):
                rot, pos = up.engine.forward(*(a[c0:c0 + UPLIFT_CHUNK] for a in args_d), dt)
                rots.append(ops.rotation_local(rot, pos))
                poss.append(pos)
            rot, pos = torch.cat(rots), torch.cat(poss)
            if world > 1:           # the per-trajectory records (spin[3] + pos[50][3]) of every shard, on every rank
                pad = torch.zeros((rec_all.shape[0] // world, 153), dtype=torch.float32, device=dev)
                pad[:nloc] = torch.cat([rot, pos.reshape(nloc, 150)], dim=1)
                dist.all_gather_into_tensor(rec_all, pad)
            return rot, pos

        up_res = {}
        for key in ('tf32x3', 'bf16', 'fp32'):
            ms_a = timed(lambda: up_chunks(ua_d, key), sub_steps if key != 'fp32' else 1, 2 if key != 'fp32' else 1)
            n_launch = (up.engine.last_launches() + 1) * ((nloc + UPLIFT_CHUNK - 1) // UPLIFT_CHUNK)

            def e2e_fn():
                rot, pos = up_chunks([a.to(dev, non_blocking=True) for a in ua_p], key)
                return rot.cpu(), pos.cpu()
            n_a = sub_steps if key != 'fp32' else 1
            ms_b = timed(e2e_fn, n_a, 1)
            up_res[key] = (UPLIFT_TOTAL * n_a / (ms_a * 1e-3), UPLIFT_TOTAL * n_a / (ms_b * 1e-3), ms_a / n_a, n_launch)
        with torch.no_grad():
            sl = [a[:4096] for a in ua_d]
            r32, p32u = up.engine.forward(*sl, 'fp32')
            r16, p16u = up.engine.forward(*sl, 'bf16')
            r3, p3u = up.engine.forward(*sl, 'tf32x3')
            vm = sl[2].bool()
            bf16_rel = float(((p16u - p32u)[vm].norm() / p32u[vm].norm()).item())
            x3_abs = float((p3u - p32u)[vm].abs().max().item())
        up_line = {'value': up_res['tf32x3'][0], 'unit': 'trajectories/s', 'dtype': 'tf32x3', 'api_default_dtype': up.compute_dtype, 'scaling': 'strong',
                   'workload': 'configs[3]: %d synthetic trajectories (T = 50, 13 table keypoints) sharded over %d rank(s) by index range, chunks of %d, '
                               'spin rotated to local axes; at N > 1 one NCCL all_gather of the 612-byte result records per pass' % (UPLIFT_TOTAL, world, UPLIFT_CHUNK),
                   'ms_per_pass': up_res['tf32x3'][2], 'gpu_launches_per_pass': up_res['tf32x3'][3],
                   'tflops': UPLIFT_GFLOP_PER_TRAJ * up_res['tf32x3'][0] / 1e3,
                   'e2e': {'value': up_res['tf32x3'][1], 'unit': 'trajectories/s', 'h2d_bytes_per_pass': int(sum(a.numel() * 4 for a in ua)) * world,
                           'd2h_bytes_per_pass': UPLIFT_TOTAL * 153 * 4},
                   'max_abs_pos_diff_vs_fp32_simt': x3_abs,
                   'note': "tf32x3: every Linear layer as three TF32 tensor-core products of split operands (fp32-level results; the reference's Linear layers are "
                           "fp32 on a GPU, torch keeps TF32 off for matmul); the API default",
                   'fp32_simt': {'value': up_res['fp32'][0], 'e2e': up_res['fp32'][1], 'ms_per_pass': up_res['fp32'][2], 'gpu_launches_per_pass': up_res['fp32'][3],
                                 'tflops': UPLIFT_GFLOP_PER_TRAJ * up_res['fp32'][0] / 1e3, 'note': 'fused SIMT stacks, the strict parity path'},
                   'bf16': {'value': up_res['bf16'][0], 'e2e': up_res['bf16'][1], 'ms_per_pass': up_res['bf16'][2], 'gpu_launches_per_pass': up_res['bf16'][3],
                            'tflops': UPLIFT_GFLOP_PER_TRAJ * up_res['bf16'][0] / 1e3,
                            'tensor_frac': UPLIFT_GFLOP_PER_TRAJ * up_res['bf16'][0] / 1e3 / world / peaks()['bf16_tflops_sustained'],
                            'vs_fp32_rel_l2': bf16_rel}}
        del ua_d, ua_p, ua

    # ---- second detector family (ViTPose-small, SURVEY.md section 8 row a4') ----
    vit_line = None
    if 'vitpose' in legs:
        vit = hubconf.ball_detection('vitpose')          # API default: tf32x3 (float32-class results on the tensor cores)
        vit.model._sync()
        vit_x = torch.empty((VIT_BATCH, 9, VIT_RES[1], VIT_RES[0]), dtype=torch.float32, device=dev)
        vit_heat = torch.empty((VIT_BATCH, 1, 4 * vit.model.engine.hp, 4 * vit.model.engine.wp), dtype=torch.float32, device=dev)
        vit_res = {}
        for key in ('tf32x3', 'bf16', 'fp32'):
            def vit_step():
                ops.preprocess_stacks(frames_dev, 3, 1, VIT_BATCH, VIT_RES[0], VIT_RES[1], layout='nchw', out=vit_x)
                vit.model.engine.forward(vit_x, key, out=vit_heat)
                return ops.decode_heatmaps(vit_heat, SRC[1], SRC[0], 'table')
            vsteps = sub_steps if key != 'fp32' else 1
            vms = timed(vit_step, vsteps, 2 if key != 'fp32' else 1)
            vit_res[key] = (fps(vms, vsteps, VIT_BATCH), vms / vsteps, vit.model.engine.last_launches() + 3)
        vit_e2e_ms = timed(lambda: vit.predict(triples_pinned[:VIT_BATCH], return_heatmaps=False), sub_steps, 2)
        with torch.no_grad():
            ops.preprocess_stacks(frames_dev, 3, 1, VIT_BATCH, VIT_RES[0], VIT_RES[1], layout='nchw', out=vit_x)
            hv32 = vit.model.engine.forward(vit_x, 'fp32').clone()
            hv16 = vit.model.engine.forward(vit_x, 'bf16').clone()
            hvx3 = vit.model.engine.forward(vit_x, 'tf32x3')
            vit_rel = float(((hv16 - hv32).norm() / hv32.norm()).item())
            vit_x3_err = float((hvx3 - hv32).abs().max().item())
            vit_x3_bound = 1e-4 * float(hv32.abs().max().item()) + 1e-5
        vit16 = hubconf.ball_detection('vitpose', dtype='bf16')
        vit16_e2e_ms = timed(lambda: vit16.predict(triples_pinned[:VIT_BATCH], return_heatmaps=False), sub_steps, 2)
        del vit16
        vit_line = {'value': vit_res['tf32x3'][0], 'unit': 'frames/s', 'dtype': 'tf32x3', 'batch_per_gpu': VIT_BATCH, 'ms_per_step': vit_res['tf32x3'][1],
                    'workload': 'ViTPose-small ball-detect (1152x640 input, 313.5 GFLOP/stack) + decode on the same 1080p stacks',
                    'e2e': {'value': fps(vit_e2e_ms, sub_steps, VIT_BATCH), 'unit': 'frames/s',
                            'h2d_bytes_per_step': int(frames_pinned[:VIT_BATCH + 2].numel()), 'd2h_bytes_per_step': VIT_BATCH * 3 * 8,
                            'api': "hubconf.ball_detection('vitpose').predict(triples, return_heatmaps=False), pinned frames"},
                    # algorithmic flops; the tensor cores execute three TF32 products per term in this class
                    'tflops': VIT_GFLOP_PER_STACK * vit_res['tf32x3'][0] / 1e3,
                    'gpu_launches': vit_res['tf32x3'][2],
                    'parity': {'vs': 'fp32 SIMT path of the same weights and input (itself within 1e-4 max|h| + 1e-5 of the CPU oracle)',
                               'max_abs_err': vit_x3_err, 'bound_fp32_class': vit_x3_bound, 'within_bound': bool(vit_x3_err <= vit_x3_bound)},
                    'bf16': {'value': vit_res['bf16'][0], 'ms_per_step': vit_res['bf16'][1], 'tflops': VIT_GFLOP_PER_STACK * vit_res['bf16'][0] / 1e3,
                             'tensor_frac': VIT_GFLOP_PER_STACK * vit_res['bf16'][0] / 1e3 / world / peaks()['bf16_tflops_sustained'],
                             'e2e': fps(vit16_e2e_ms, sub_steps, VIT_BATCH), 'vs_f32_rel_l2': vit_rel},
                    'f32_simt': {'value': vit_res['fp32'][0], 'ms_per_step': vit_res['fp32'][1]}}
        del vit, vit_x, vit_heat, hv32, hv16, hvx3

    # ---- the full hub pipeline: configs[2] (one 300-frame clip) and configs[4] (64 clips sharded over the ranks + NCCL gather).
    # Main and auxiliary detectors are separate objects loaded from the same WASB / HRNet checkpoints: random-init detectors of different
    # architectures never agree within 20 px, and the agreement filters would reject every frame.  The reference's uplifting model (and
    # this drop-in) raise ValueError on 50 or more detections (uplifting/model.py:541-546), so a clip is one rally of 50 frames
    # (48 detections); the 300-frame clip is processed as six such rallies ----
    pipe_line = clips_line = None
    if 'pipeline' in legs or 'clips' in legs:
        pipe = hubconf.full_pipeline(ball_model='wasb', ball_model_aux='wasb', table_model='hrnet', table_model_aux='hrnet')
        pipe_dtypes = {'ball': pipe.ball_detector.model.compute_dtype, 'table': pipe.table_detector.model.compute_dtype,
                       'uplift': pipe.uplifting_model.model.compute_dtype}
    if 'pipeline' in legs:
        clip = synthetic.frames_1080p(CLIP_FRAMES, seed=200 + rank)          # pageable numpy frames, what cv2 delivers
        rallies = [[clip[i] for i in range(r0, r0 + RALLY_FRAMES)] for r0 in range(0, CLIP_FRAMES, RALLY_FRAMES)]
        pipe_ms = timed(lambda: [pipe.predict(r, 50.0) for r in rallies], 2, 1)
        res = [pipe.predict(r, 50.0) for r in rallies]
        pipe_line = {'value': fps(pipe_ms, 2, CLIP_FRAMES), 'unit': 'frames/s', 'ms_per_clip': pipe_ms / 2, 'frames_per_clip': CLIP_FRAMES, 'dtypes': pipe_dtypes,
                     'scaling': 'weak', 'finite_outputs': all(bool(torch.isfinite(sp).all().item()) and bool(np.isfinite(p3).all()) for sp, p3 in res),
                     'trajectory_lengths': [int(p3.shape[0]) for _, p3 in res],
                     'workload': 'configs[2]: hubconf.full_pipeline(...).predict on one 300-frame 1080p clip per rank (numpy frames in pageable host memory), as 6 rallies '
                                 'of 50 frames: WASB main + aux on 288 stacks, HRNet main + aux on 300 frames, 8376 heatmap decodes, both agreement filters, uplift; end to end',
                     'h2d_bytes_per_clip': CLIP_FRAMES * SRC[0] * SRC[1] * 3}
        del clip, rallies
    if 'clips' in legs:
        base = [synthetic.frames_1080p(RALLY_FRAMES, seed=300 + i) for i in range(N_BASE_CLIPS)]
        clips = [[base[i % N_BASE_CLIPS][j] for j in range(RALLY_FRAMES)] for i in range(N_CLIPS)]
        sharding.run_clips(lambda c: pipe.predict(c, 50.0), clips[:world], dev)          # warm-up: one clip per rank
        got = []
        clips_ms = timed(lambda: got.append(sharding.run_clips(lambda c: pipe.predict(c, 50.0), clips, dev)), 1, 0)
        table = got[0]
        ok = tuple(table.shape) == (N_CLIPS, sharding.RECORD_FLOATS) and bool(torch.isfinite(table).all().item()) and bool((table[:, 0] == RALLY_FRAMES - 2).all().item())
        same = bool(torch.equal(table[0], table[N_BASE_CLIPS]))          # clips i and i + N_BASE_CLIPS have the same frames (and land on different ranks at N > 1)
        clips_line = {'value': N_CLIPS * RALLY_FRAMES / (clips_ms * 1e-3), 'unit': 'frames/s', 'clips_per_sec': N_CLIPS / (clips_ms * 1e-3), 'ms_per_pass': clips_ms,
                      'scaling': 'strong', 'dtypes': pipe_dtypes, 'records_ok': ok, 'repeated_clip_identical_across_ranks': same,
                      'workload': 'configs[4]: %d clips of %d 1080p frames (%d distinct synthetic clips, repeated) through sharding.run_clips: clips sharded over %d rank(s) by index '
                                  'range, hubconf.full_pipeline(...).predict per clip from pageable numpy frames, one NCCL all_gather of the 616-byte per-clip records'
                                  % (N_CLIPS, RALLY_FRAMES, N_BASE_CLIPS, world)}
        del base, clips
    calib_line = None
    if 'calibration' in legs:
        kps = synthetic.table_keypoints(CALIB_CLIPS, seed=11 + rank)
        kps_d = torch.from_numpy(kps).to(dev)
        smp_d = torch.from_numpy(ops.ransac_sample_table(kps)).to(dev)
        calib_ms = timed(lambda: ops.calibrate_camera(kps_d, smp_d), sub_steps, 2)
        calib_info = ops.calibrate_camera(kps_d, smp_d)[2].cpu().numpy()
        calib_line = {'value': fps(calib_ms, sub_steps, CALIB_CLIPS), 'unit': 'clips/s', 'clips_per_gpu': CALIB_CLIPS,
                      'ms_per_step': calib_ms / sub_steps, 'gpu_launches': 3,
                      'workload': 'calibrate_camera: DLT + 100 RANSAC hypotheses of SciPy-BFGS fits + refit per clip (13 keypoints, 1 outlier, 1 hidden)',
                      'median_inliers': float(np.median(calib_info[:, 0])),
                      'cpu_reference_note': 'the reference needs ~24 s per clip on the host (SURVEY.md section 6; 100 sequential scipy.optimize.minimize calls)'}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel: per-launch CUDA events on the launching stream ----------
    pk = peaks()
    check = _lib.check
    tensor_peak = {'bf16': pk['bf16_tflops_sustained'], 'tf32': pk['bf16_tflops_sustained'] / 2, 'fp32': pk['bf16_tflops_sustained'] / 2}

    def roofline_of(prec, dump=None):
        step_device(prec, gather=False, mark=True)
        torch.cuda.synchronize()
        x = xbuf[storage_dtype(prec)]
        pre_ms, dec_ms = stage_ev[0].elapsed_time(stage_ev[1]), stage_ev[2].elapsed_time(stage_ev[3])
        pre_bytes = frames_dev.numel() + x.numel() * x.element_size()
        dec_bytes = heat.numel() * 4 + BATCH * 24
        stages = {'preprocess': {'ms': pre_ms, 'algorithmic_bytes': pre_bytes, 'gbs': pre_bytes / (pre_ms * 1e-3) / 1e9,
                                 'hbm_frac': pre_bytes / (pre_ms * 1e-3) / 1e9 / pk['hbm_gbs']},
                  'decode': {'ms': dec_ms, 'algorithmic_bytes': dec_bytes, 'gbs': dec_bytes / (dec_ms * 1e-3) / 1e9,
                             'hbm_frac': dec_bytes / (dec_ms * 1e-3) / 1e9 / pk['hbm_gbs'],
                             'note': 'argmax (one read of every heatmap value) + per-map L-BFGS-B fit; the %d-map batch is smaller than L2' % BATCH}}
        check(lib.ttk_hrnet_set_profile(engine.h, 1))
        step_device(prec, gather=False)
        torch.cuda.synchronize()
        per = {}
        ot, ci, ms, fl, by = C.c_int(), C.c_int(), C.c_float(), C.c_double(), C.c_double()
        tot_ms = 0.0
        for i in range(lib.ttk_hrnet_profile_count(engine.h)):
            check(lib.ttk_hrnet_profile_read(engine.h, i, C.byref(ot), C.byref(ci), C.byref(ms), C.byref(fl), C.byref(by)))
            r = per.setdefault((ot.value, ci.value), [0.0, 0.0, 0.0, 0])
            r[0] += ms.value
            r[1] += fl.value
            r[2] += by.value
            r[3] += 1
            tot_ms += ms.value
        check(lib.ttk_hrnet_set_profile(engine.h, 0))
        if dump:
            rows = []
            for (t_, c_), v in sorted(per.items(), key=lambda kv: -kv[1][0]):
                nm = engine.specs[c_][0] if c_ >= 0 else ('fuse_sum' if t_ == 1 else 'final_conv')
                rows.append({'kernel': nm, 'spec_cin_cout_k_stride': engine.specs[c_][2:] if c_ >= 0 else None, 'launches': v[3], 'ms': v[0], 'share': v[0] / tot_ms,
                             'tflops': v[1] / (v[0] * 1e-3) / 1e12, 'gbs': v[2] / (v[0] * 1e-3) / 1e9})
            json.dump({'dtype': prec, 'total_ms': tot_ms, 'rows': rows}, open(dump, 'w'), indent=1)
        (top_type, top_conv), top = max(per.items(), key=lambda kv: kv[1][0])
        name = engine.specs[top_conv][0] if top_conv >= 0 else ('fuse_sum' if top_type == 1 else 'final_conv')
        achieved_tf, achieved_gbs = top[1] / (top[0] * 1e-3) / 1e12, top[2] / (top[0] * 1e-3) / 1e9
        conv_ms, conv_fl, conv_by = (sum(v[j] for k, v in per.items() if k[0] == 0) for j in range(3))
        tpk = tensor_peak[prec]
        ridge = tpk * 1e12 / (pk['hbm_gbs'] * 1e9)
        intensity = top[1] / top[2]
        hbm_bound = intensity < ridge
        return {
            'bound': 'hbm' if hbm_bound else 'tensor', 'dtype': prec,
            'kernel': 'conv %s (%d launches/step, %.1f%% of detector time)' % (name, top[3], 100 * top[0] / tot_ms),
            'achieved': achieved_gbs if hbm_bound else achieved_tf,
            'peak': pk['hbm_gbs'] if hbm_bound else tpk,
            'unit': 'GB/s' if hbm_bound else 'TFLOP/s',
            'frac': (achieved_gbs / pk['hbm_gbs']) if hbm_bound else (achieved_tf / tpk),
            'traffic': ncu_traffic('%s/%s' % (prec, name), BATCH / top[3]),
            'traffic_note': 'dram__bytes_read.sum + dram__bytes_write.sum of this kernel from the committed ncu --set full capture (profiles/ncu_traffic.json), per launch',
            'peak_source': pk['source'] + (', copy bandwidth' if hbm_bound else ', sustained bf16 (kernel timed inside a long step)%s' % (' / 2: kind::tf32 issues at half the bf16 rate' if prec != 'bf16' else '')),
            'intensity_flop_per_byte': intensity, 'ridge_flop_per_byte': ridge,
            'algorithmic_bytes_per_launch': top[2] / top[3], 'algorithmic_flops_per_launch': top[1] / top[3],
            'avg_launch_ms': top[0] / top[3],
            'tensor_achieved_tflops': achieved_tf, 'tensor_frac': achieved_tf / tpk,
            'hbm_achieved_gbs': achieved_gbs, 'hbm_frac': achieved_gbs / pk['hbm_gbs'],
            'all_convs': {'achieved_tflops': conv_fl / (conv_ms * 1e-3) / 1e12, 'tensor_frac': conv_fl / (conv_ms * 1e-3) / 1e12 / tpk,
                          'achieved_gbs': conv_by / (conv_ms * 1e-3) / 1e9, 'hbm_frac': conv_by / (conv_ms * 1e-3) / 1e9 / pk['hbm_gbs'],
                          'share_of_detector_time': conv_ms / tot_ms, 'ms': conv_ms},
            'stages': stages,
        }

    roofline = roofline_of(args.dtype, args.dump_profile or None)
    stages = roofline.pop('stages')
    roofline['whole_step_tflops'] = WASB_GFLOP_PER_STACK * BATCH * args.steps / (head['ms_dev'] * 1e-3) / 1e3
    roofline['whole_step_tflops_note'] = ('against the 344.07 GFLOP per stack of the reference graph; the plan skips the thirteen stage-4 fuse convolutions whose outputs '
                                          'nothing reads (the reference computes and drops them), all_convs counts the executed work')
    roofline_other = None
    if 'bf16' in legs:
        o = 'bf16' if args.dtype != 'bf16' else 'tf32'
        roofline_other = roofline_of(o, (args.dump_profile + '.' + o) if args.dump_profile else None)
        roofline_other.pop('stages')
    # the decode's HBM-bound kernel on its own: 64 maps (231 MB, larger than L2), argmax pass timed by the library's events
    g = torch.Generator(device=dev).manual_seed(0)
    big = torch.randn((64, H, W), device=dev, generator=g) * 0.05
    big[:, 100:103, 200:203] += 1.0
    check(lib.ttk_decode_set_profile(1))
    am_ms = []
    for _ in range(5):
        ops.decode_heatmaps(big, SRC[1], SRC[0], 'table')
        a_ms, f_ms = C.c_float(), C.c_float()
        check(lib.ttk_decode_profile_read(C.byref(a_ms), C.byref(f_ms)))
        am_ms.append((a_ms.value, f_ms.value))
    check(lib.ttk_decode_set_profile(0))
    a_ms, f_ms = sorted(am_ms)[len(am_ms) // 2]
    big_bytes = big.numel() * 4
    stages['decode_argmax_64maps'] = {'ms': a_ms, 'fit_ms': f_ms, 'algorithmic_bytes': big_bytes, 'gbs': big_bytes / (a_ms * 1e-3) / 1e9,
                                      'hbm_frac': big_bytes / (a_ms * 1e-3) / 1e9 / pk['hbm_gbs'],
                                      'note': 'argmax_partial_kernel alone on 64 maps of 704x1280 (231 MB > L2), median of 5, CUDA events on the launching '
                                              'stream; fit_ms is the per-map L-BFGS-B kernel (latency floor, independent of the map count)'}
    del big

    # ---- stock PyTorch eager on this GPU (SURVEY.md section 2a's bar) and the CPU baselines (BASELINE.md section 3) ----
    eager = None
    if not args.no_eager_baseline:
        del xbuf, heat
        torch.cuda.empty_cache()
        eager = gpu_eager_baseline(dev)
        net_ms = roofline['all_convs']['ms'] / roofline['all_convs']['share_of_detector_time']
        eager['speedup_wasb_network'] = {'ours_stacks_per_s': BATCH / (net_ms * 1e-3), 'dtype': args.dtype,
                                         'vs_torch_tf32_default': BATCH / (net_ms * 1e-3) / eager['wasb_forward']['tf32_default'],
                                         'vs_torch_tf32_channels_last': BATCH / (net_ms * 1e-3) / eager['wasb_forward']['tf32_channels_last']}
        if roofline_other is not None:
            o_ms = roofline_other['all_convs']['ms'] / roofline_other['all_convs']['share_of_detector_time']
            eager['speedup_wasb_network'][roofline_other['dtype'] + '_vs_torch_bf16_channels_last'] = BATCH / (o_ms * 1e-3) / eager['wasb_forward']['bf16_channels_last']
        if up_line is not None:
            eager['speedup_uplift'] = {'tf32x3_vs_torch_fp32_sdpa': up_line['value'] / world / eager['uplift_forward']['fp32_sdpa_b4096'],
                                       'fp32_simt_vs_torch_fp32_sdpa': up_line['fp32_simt']['value'] / world / eager['uplift_forward']['fp32_sdpa_b4096']}
        if vit_line is not None and 'vitpose_forward' in eager:
            ev = eager['vitpose_forward']
            eager['speedup_vitpose'] = {'note': 'ours includes pre-processing and decode, the torch figures are the network alone',
                                        'tf32x3_vs_torch_fp32_default': vit_line['value'] / world / ev['fp32_default'],
                                        'tf32x3_vs_torch_tf32_matmul_opt_in': vit_line['value'] / world / ev['tf32_matmul_opt_in']}
            if 'bf16' in ev:
                eager['speedup_vitpose']['bf16_vs_torch_bf16'] = vit_line['bf16']['value'] / world / ev['bf16']
    cpu = None
    if not args.no_cpu_baseline:
        torch.set_num_threads(os.cpu_count())
        n_cpu = 3
        cpu_reference_step(wasb_sd, frames_np, 1)
        sec = cpu_reference_step(wasb_sd, frames_np, n_cpu)
        cpu = {'value': n_cpu / sec, 'unit': 'frames/s', 'cores': torch.get_num_threads(), 'kind': 'port',
               'sample': '%d stacks (after 1 warm-up) through oracle/: numpy fixed-point resize, CPU torch fp32 WASB, SciPy L-BFGS-B decode, B=1 per forward' % n_cpu}
        if up_line is not None:
            cu = cpu_uplift_baseline(up_sd)
            cpu['uplift'] = {'b1_trajectories_per_s': cu['b1'], 'b512_trajectories_per_s': cu['b512'], 'unit': 'trajectories/s',
                             'sample': 'oracle/uplift.py on the host cores: 20 forwards at B=1, one at B=512 (after one warm-up each)'}
        if pipe_line is not None:
            sec, nfr = cpu_pipeline_baseline(wasb_sd, table_sd, up_sd, list(frames_np[:4]))
            cpu['pipeline'] = {'value': nfr / sec, 'unit': 'frames/s', 'seconds': sec, 'frames': nfr,
                               'sample': 'TableTennisPipeline.predict chained through oracle/ on a %d-frame 1080p clip: WASB x2 on %d stacks, HRNet x2 on %d frames, '
                                         'decodes, both filters, uplift (B=1 per forward); a 300-frame clip extrapolates to %.0f s' % (nfr, nfr - 2, nfr, 300 * sec / nfr)}

    def e2e_entry(ms, steps, api, h2d, d2h):
        return {'value': fps(ms, steps), 'unit': 'frames/s', 'ms_per_step': ms / steps, 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h), 'api': api}
    frame_bytes = SRC[0] * SRC[1] * 3
    hm_bytes = BATCH * H * W * 4
    line = {
        'metric': 'frames_per_sec_detect_decode', 'value': value, 'unit': 'frames/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': head['ms_dev'] / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': args.dtype, 'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'api_default_dtype': api_default,
                   'parallelism': 'clip-sharded x%d, NCCL all_gather of (x,y,v) records' % world,
                   'host_sync': host_sync + (' (cudaDeviceScheduleBlockingSync: several ranks share the host cores)' if host_sync == 'blocking' else ' (CUDA default)'),
                   'l2': 'inputs (211 MB of frames) and activations exceed the 126 MB L2',
                   'weights': 'seeded synthetic (synthetic.hrnet_blob_state_dict: random, BN folded; the frames\' bright blob survives to the heatmap so that peaks are genuine)'},
        'e2e': dict(e2e_entry(head['ms_copy_hm'], args.steps, "hubconf.ball_detection('wasb').predict(triples): 32 (prev, cur, next) triples of numpy frames in pageable host memory, every "
                              "frame a separate .copy() as interface.py:275 builds them (96 frames cross PCIe), heatmaps returned as numpy like the reference's default call",
                              3 * BATCH * frame_bytes, BATCH * 24 + hm_bytes),
                    numpy_window_views=e2e_entry(head['ms_view'], sub_steps, 'same call, return_heatmaps=False, triples are views of one clip array (34 distinct frames are recognised and uploaded once)',
                                                 (BATCH + 2) * frame_bytes, BATCH * 24),
                    numpy_window_views_with_heatmaps=e2e_entry(head['ms_view_hm'], sub_steps, 'views of one clip array, heatmaps returned', (BATCH + 2) * frame_bytes, BATCH * 24 + hm_bytes),
                    numpy_copies=e2e_entry(head['ms_copy'], sub_steps, 'copied triples, return_heatmaps=False', 3 * BATCH * frame_bytes, BATCH * 24),
                    pinned_torch=e2e_entry(head['ms_pinned'], args.steps, 'pinned torch frames (views of one clip tensor), return_heatmaps=False', (BATCH + 2) * frame_bytes, BATCH * 24)),
        'gpu_launches': head['launches'] * args.steps,
        'clocks': clocks,
        'roofline': roofline,
        'stages': stages,
        'parity': parity,
        'cpu_baseline': cpu,
        'gpu_eager_baseline': eager,
    }
    for prec, r in other.items():
        line[prec] = {'value': fps(r['ms_dev'], sub_steps), 'unit': 'frames/s', 'ms_per_step': r['ms_dev'] / sub_steps, 'gpu_launches_per_step': r['launches'],
                      'e2e': dict(e2e_entry(r['ms_copy_hm'], sub_steps, 'numpy copied triples, heatmaps returned (the headline e2e call)', 3 * BATCH * frame_bytes, BATCH * 24 + hm_bytes),
                                  pinned_torch=e2e_entry(r['ms_pinned'], sub_steps, 'pinned torch frames, return_heatmaps=False', (BATCH + 2) * frame_bytes, BATCH * 24)),
                      'roofline': roofline_other if roofline_other is not None and roofline_other['dtype'] == prec else None,
                      'note': 'reported separately: %s' % ('bf16 storage and operands, own bound (parity.bf16)' if prec == 'bf16' else 'the API default')}
    if up_line is not None:
        line['uplift'] = up_line
    if vit_line is not None:
        line['vitpose'] = vit_line
    if pipe_line is not None:
        line['pipeline'] = pipe_line
    if clips_line is not None:
        line['clips'] = clips_line
    if calib_line is not None:
        line['calibration'] = calib_line
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    # stdout carries exactly one JSON line: everything else the libraries print (model loaders, and NCCL's version banner, which is a
    # C-level write to file descriptor 1) goes to stderr
    sys.stdout.flush()
    _real_stdout = os.fdopen(os.dup(1), 'w')
    os.dup2(2, 1)
    sys.stdout = sys.stderr
    _orig_print = print

    def print(*a, **k):          # noqa: A001 - the JSON line
        k.setdefault('file', _real_stdout)
        _orig_print(*a, **k)
        _real_stdout.flush()
    main()
