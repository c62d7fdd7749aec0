"""WASB at the bench config (32 stacks, 1080p frames -> 1280x704, synthetic.hrnet_blob_state_dict) in six arithmetic classes, timed in
one process and alternating: the 'tf32' tensor-core path (default), 'tf32x3' (3xTF32 tensor-core products, fp32-level), the 16-bit
tensor-core paths 'bf16' and 'fp16' (each on its own preprocessed input), the SIMT 'fp32' path, and stock PyTorch strict-fp32 cuDNN
(oracle.hrnet.wasb_forward with cudnn.allow_tf32 off, cudnn.benchmark on).  Network only: the input is the preprocessed batch.  Prints
JSON with the GPU name and power limit and writes it to the given path:

    python tools/time_wasb.py [out.json] [rounds] [steps]
"""
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import hrnet as ohr  # noqa: E402
from upliftingtabletennis_b200 import ops, synthetic  # noqa: E402
from upliftingtabletennis_b200.detector import WASBNet  # noqa: E402

B, W, H = 32, 1280, 704


def gpu_info():
    q = 'name,power.limit,clocks.max.sm'
    try:
        line = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=' + q, '--format=csv,noheader'], capture_output=True, text=True,
                              timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in line.split(',')]
    except (OSError, ValueError, subprocess.SubprocessError):
        name, power, clock = torch.cuda.get_device_name(0), None, None
    return {'gpu': name, 'power_limit': power, 'sm_max_clock': clock}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join('profiles', 'wasb_timing.json')
    rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    steps = int(sys.argv[3]) if len(sys.argv) > 3 else 3
    dev = torch.device('cuda:0')
    sd = synthetic.hrnet_blob_state_dict(ohr.state_dict_layout(9, 3), seed=1)
    m = WASBNet().to(dev).eval()
    m.load_state_dict(sd)
    frames = torch.from_numpy(synthetic.frames_1080p(B + 2, seed=100)).to(dev)
    x = ops.preprocess_stacks(frames, 3, 1, B, W, H, layout='nhwc16', dtype=torch.float32)
    x16 = {p: ops.preprocess_stacks(frames, 3, 1, B, W, H, layout='nhwc16', dtype=dt) for p, dt in (('bf16', torch.bfloat16), ('fp16', torch.float16))}
    x_nchw = x[..., :9].permute(0, 3, 1, 2).contiguous()
    sd_dev = {k: v.to(dev) for k, v in sd.items()}

    def torch_strict():
        with torch.no_grad():
            return ohr.wasb_forward(sd_dev, x_nchw)

    arms = {p: (lambda p=p: m.heatmaps_from_nhwc16(x16.get(p, x), p)) for p in ('tf32', 'tf32x3', 'bf16', 'fp16', 'fp32')}
    arms['torch_fp32_strict'] = torch_strict
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.allow_tf32, torch.backends.cudnn.benchmark = False, True
    try:
        outs = {}
        for k, fn in arms.items():          # warm-up: module loads, tensor maps, cuDNN algorithm selection
            outs[k] = fn()
            fn()
        torch.cuda.synchronize()
        ref = outs['fp32']
        max_diff = {k: float((v - ref).abs().max()) for k, v in outs.items()}
        del outs
        samples = {k: [] for k in arms}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(rounds):
            for k, fn in arms.items():
                torch.cuda.synchronize()
                e0.record()
                for _ in range(steps):
                    fn()
                e1.record()
                torch.cuda.synchronize()
                samples[k].append(B * steps / (e0.elapsed_time(e1) * 1e-3))
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cudnn.benchmark = old
    med = {k: sorted(v)[len(v) // 2] for k, v in samples.items()}
    res = {'workload': 'WASB forward, %d stacks of 1080p frames resized to %dx%d, synthetic.hrnet_blob_state_dict(seed=1); network only' % (B, W, H),
           **gpu_info(), 'unit': 'stacks/s', 'rounds': rounds, 'steps_per_sample': steps, 'median': med, 'samples': samples,
           'tf32x3_over_tf32': med['tf32x3'] / med['tf32'], 'tf32x3_over_simt_fp32': med['tf32x3'] / med['fp32'],
           'tf32x3_over_torch_fp32_strict': med['tf32x3'] / med['torch_fp32_strict'],
           'fp16_over_bf16': med['fp16'] / med['bf16'], 'fp16_over_tf32': med['fp16'] / med['tf32'],
           'max_abs_diff_vs_simt_fp32': max_diff, 'max_abs_simt_fp32': float(ref.abs().max())}
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, 'w') as f:
        json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
