"""Per-launch table of one detector pass (ttk_hrnet_set_profile): python tools/layer_profile.py [tf32|tf32x3|bf16|fp32] [batch] [out.json]."""
import ctypes as C
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from upliftingtabletennis_b200 import ops, synthetic  # noqa: E402
from upliftingtabletennis_b200._lib import check, lib  # noqa: E402
from upliftingtabletennis_b200.detector import WASBNet  # noqa: E402

prec = sys.argv[1] if len(sys.argv) > 1 else 'tf32'
n = int(sys.argv[2]) if len(sys.argv) > 2 else 32
dev = torch.device('cuda:0')
m = WASBNet(dtype=prec).to(dev).eval()
m.load_state_dict(synthetic.hrnet_state_dict(m.engine.state_dict_layout(), seed=1))
frames = torch.from_numpy(synthetic.frames_1080p(n + 2, seed=5)).to(dev)
x = ops.preprocess_stacks(frames, 3, 1, n, 1280, 704, layout='nhwc16', dtype=m.storage_dtype)
for _ in range(3):
    hm = m.heatmaps_from_nhwc16(x, prec)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(5):
    hm = m.heatmaps_from_nhwc16(x, prec)
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / 5
print('%s: %.2f ms per %d stacks = %.0f stacks/s (network only)' % (prec, ms, n, n / ms * 1e3))
eng = m.engine
check(lib.ttk_hrnet_set_profile(eng.h, 1))
hm = m.heatmaps_from_nhwc16(x, prec)
torch.cuda.synchronize()
per, tot = {}, 0.0
ot, ci, t, fl, by = C.c_int(), C.c_int(), C.c_float(), C.c_double(), C.c_double()
for i in range(lib.ttk_hrnet_profile_count(eng.h)):
    check(lib.ttk_hrnet_profile_read(eng.h, i, C.byref(ot), C.byref(ci), C.byref(t), C.byref(fl), C.byref(by)))
    r = per.setdefault((ot.value, ci.value), [0.0, 0.0, 0.0, 0])
    r[0] += t.value; r[1] += fl.value; r[2] += by.value; r[3] += 1
    tot += t.value
check(lib.ttk_hrnet_set_profile(eng.h, 0))
rows = []
for (t_, c_), v in sorted(per.items(), key=lambda kv: -kv[1][0]):
    nm = eng.specs[c_][0] if c_ >= 0 else ('fuse_sum' if t_ == 1 else 'final_conv')
    rows.append({'kernel': nm, 'spec_cin_cout_k_stride': eng.specs[c_][2:] if c_ >= 0 else None, 'simt_fallback': t_ == 3, 'launches': v[3], 'ms': v[0], 'share': v[0] / tot,
                 'tflops': v[1] / (v[0] * 1e-3) / 1e12, 'gbs': v[2] / (v[0] * 1e-3) / 1e9})
print('profiled total %.2f ms' % tot)
for r in rows[:45]:
    print('%-42s %-18s n=%2d ms=%6.3f share=%5.1f%% tf=%6.0f gbs=%5.0f%s' % (r['kernel'], r['spec_cin_cout_k_stride'], r['launches'], r['ms'], 100 * r['share'], r['tflops'], r['gbs'],
                                                                        ' (SIMT fallback)' if r['simt_fallback'] else ''))
if len(sys.argv) > 3:
    json.dump({'precision': prec, 'batch': n, 'total_ms': tot, 'ms_per_pass': ms, 'rows': rows}, open(sys.argv[3], 'w'), indent=1)
