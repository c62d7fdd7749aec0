"""The 3xTF32 ('tf32x3') path of the WASB / HRNet detectors: every convolution of the plan against float64 on unrounded operands, the
network against the CPU oracle and the golden file at the strict fp32 bar, the full-size batch against the SIMT fp32 path, batch
invariance, and the hub entry points.  The tests marked gpu need a B200: run with `-m gpu`."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import decode as odec
from oracle import hrnet as ohr
from oracle import preprocess as opre


def _fp32_bar(ref):
    """the strict fp32 path's bar: |d| <= 1e-4 max|h| + 1e-5"""
    return 1e-4 * float(np.abs(ref).max()) + 1e-5


def _margin_ok(maps, bound):
    """maps whose top-2 margin exceeds twice the bound"""
    flat = maps.reshape(maps.shape[0], -1)
    top2 = torch.topk(flat, 2, dim=1).values
    return (top2[:, 0] - top2[:, 1]) > 2 * bound


@pytest.fixture(scope='module')
def dev():
    assert torch.cuda.is_available()
    return torch.device('cuda:0')


def test_tf32x3_accepted_without_gpu():
    """The HRNet shells take 'tf32x3' through dtype= and compute_dtype, and the library sizes its workspace (fp32 storage, like TF32)
    without a device."""
    from upliftingtabletennis_b200 import _lib
    from upliftingtabletennis_b200.detector import MyHRNet, WASBNet
    m = WASBNet(dtype='tf32x3')
    assert m.compute_dtype == 'tf32x3' and m.storage_dtype == torch.float32
    m.compute_dtype = 'fp32'
    m.compute_dtype = '3xtf32'
    assert m.compute_dtype == 'tf32x3'
    assert MyHRNet(dtype='tf32x3').compute_dtype == 'tf32x3' and MyHRNet().compute_dtype == 'tf32'
    ws = _lib.lib.ttk_hrnet_workspace_bytes(m.engine.h, 2, 704, 1280, _lib.TF32X3)
    assert ws > 0 and ws == _lib.lib.ttk_hrnet_workspace_bytes(m.engine.h, 2, 704, 1280, _lib.TF32)


@pytest.mark.gpu
@pytest.mark.parametrize('shape', [(2, 24, 200), (1, 10, 130), (1, 40, 72), (1, 16, 520)])
def test_every_conv_x3_vs_float64(dev, shape):
    """debug_conv path 4 for every convolution of the plan (bias, residual on / off, ReLU) against a float64 convolution of the
    unrounded fp32 inputs and weights: TF32's bar, now against exact operands.  Every convolution has an x3 kernel."""
    from upliftingtabletennis_b200._lib import lib, ptr, stream_ptr
    from upliftingtabletennis_b200.detector import WASBNet
    m = WASBNet().to(dev).eval()
    sd = ohr.random_state_dict(9, 3, seed=123)
    m.load_state_dict(sd)
    m._sync()
    eng = m.engine
    n, H, W = shape
    rng = np.random.default_rng(H * W)
    specs = ohr.conv_specs(9, 3)
    worst = 0.0
    for idx, (name, bn, cin, cout, k, stride) in enumerate(eng.specs[:-1]):
        cin_p, cout_p = (cin + 15) // 16 * 16, (cout + 15) // 16 * 16
        x = torch.zeros((n, H, W, cin_p), dtype=torch.float32)
        x[..., :cin] = torch.from_numpy(rng.standard_normal((n, H, W, cin)).astype(np.float32))
        Ho, Wo = (H + stride - 1) // stride, (W + stride - 1) // stride
        res = torch.zeros((n, Ho, Wo, cout_p), dtype=torch.float32)
        res[..., :cout] = torch.from_numpy(rng.standard_normal((n, Ho, Wo, cout)).astype(np.float32))
        xd, rd = x.to(dev), res.to(dev)
        w, b = ohr.fold_bn(sd, specs[idx])
        w32 = torch.from_numpy(w.astype(np.float32))
        conv = F.conv2d(x[..., :cin].permute(0, 3, 1, 2).double(), w32.double(), None, stride=stride, padding=k // 2)
        conv = conv + torch.from_numpy(b.astype(np.float32)).double()[None, :, None, None]
        for use_res in (True, False):
            out = torch.full((n, Ho, Wo, cout_p), float('nan'), dtype=torch.float32, device=dev)
            rc = lib.ttk_hrnet_debug_conv(eng.h, idx, ptr(xd), n, H, W, ptr(rd) if use_res else None, 1, 4, ptr(out), stream_ptr())
            torch.cuda.synchronize()
            assert rc == 0, (name, rc)
            ref = conv + res[..., :cout].permute(0, 3, 1, 2).double() if use_res else conv
            ref = torch.relu(ref).permute(0, 2, 3, 1)
            y = out.cpu()
            assert torch.isfinite(y).all(), name
            err = float((ref - y[..., :cout].double()).abs().max())
            bar = 2e-5 * (float(ref.abs().max()) + 1.0)
            assert err <= bar, (name, use_res, err, bar)
            worst = max(worst, err / bar)
            assert float(y[..., cout:].abs().max() if cout_p > cout else 0.0) == 0.0
    print('x3 convolutions %s: worst error / bar = %.3f' % (shape, worst))
    x = torch.zeros((1, 8, 8, 16), device=dev)
    out = torch.zeros((1, 8, 8, 64), device=dev)
    assert lib.ttk_hrnet_debug_conv(eng.h, 0, ptr(x), 1, 8, 8, None, 1, 5, ptr(out), stream_ptr()) == -1      # paths are 0-4


@pytest.mark.gpu
@pytest.mark.parametrize('shape', [(1, 88, 160), (3, 40, 72), (2, 8, 8), (2, 64, 200)])
def test_network_x3_vs_oracle(dev, shape):
    """WASB and the 13-channel HRNet table detector on the x3 path against the CPU oracle at the strict path's bar."""
    from upliftingtabletennis_b200.detector import MyHRNet, WASBNet
    B, H, W = shape
    rng = np.random.default_rng(B * 1000 + H)
    sd = ohr.random_state_dict(9, 3, seed=77)
    x = rng.standard_normal((B, 9, H, W)).astype(np.float32)
    ref = ohr.wasb_forward(sd, torch.from_numpy(x)).numpy()
    m = WASBNet(dtype='tf32x3').to(dev).eval()
    m.load_state_dict(sd)
    y, _ = m(torch.from_numpy(x).to(dev))
    err = np.abs(y.cpu().numpy() - ref).max()
    assert err <= _fp32_bar(ref), (err, _fp32_bar(ref))
    sdt = ohr.random_state_dict(3, 13, seed=78)
    xt = rng.standard_normal((B, 3, H, W)).astype(np.float32)
    reft = ohr.hrnet_forward(sdt, torch.from_numpy(xt)).numpy()
    t = MyHRNet(dtype='tf32x3').to(dev).eval()
    t.load_state_dict(sdt)
    yt = t(torch.from_numpy(xt).to(dev)).cpu().numpy()
    assert yt.shape == reft.shape
    assert np.abs(yt - reft).max() <= _fp32_bar(reft), (np.abs(yt - reft).max(), _fp32_bar(reft))


@pytest.mark.gpu
def test_network_x3_golden(dev, golden):
    from upliftingtabletennis_b200.detector import MyHRNet, WASBNet
    g = golden('hrnet')
    m = WASBNet(dtype='tf32x3').to(dev).eval()
    m.load_state_dict(ohr.random_state_dict(9, 3, seed=int(g['wasb_seed'])))
    y, _ = m(torch.from_numpy(g['wasb_x']).to(dev))
    np.testing.assert_allclose(y.cpu().numpy(), g['wasb_y'], rtol=0, atol=_fp32_bar(g['wasb_y']))
    t = MyHRNet(dtype='tf32x3').to(dev).eval()
    t.load_state_dict(ohr.random_state_dict(3, 13, seed=int(g['table_seed'])))
    yt = t(torch.from_numpy(g['table_x']).to(dev))
    np.testing.assert_allclose(yt.cpu().numpy(), g['table_y'], rtol=0, atol=_fp32_bar(g['table_y']))


@pytest.mark.gpu
def test_full_size_x3_vs_simt_fp32(dev):
    """32 stacks of 1080p frames with a moving blob -> WASB @1280x704 on the x3 path against the SIMT fp32 path on the same GPU: the
    fp32 bar on the heatmaps, the same peak index wherever the top-2 margin exceeds twice the bar, decoded coordinates within 1e-2 px
    there; three stacks also against the CPU oracle."""
    from upliftingtabletennis_b200 import ops, synthetic
    from upliftingtabletennis_b200.detector import WASBNet
    B = 32
    frames_np = synthetic.frames_1080p(B + 2, seed=100)
    frames = torch.from_numpy(frames_np).to(dev)
    sd = synthetic.hrnet_blob_state_dict(ohr.state_dict_layout(9, 3), seed=1)
    m = WASBNet(dtype='tf32x3').to(dev).eval()
    m.load_state_dict(sd)
    x = ops.preprocess_stacks(frames, 3, 1, B, 1280, 704, layout='nhwc16', dtype=torch.float32)
    h3 = m.heatmaps_from_nhwc16(x, 'tf32x3')
    h32 = m.heatmaps_from_nhwc16(x, 'fp32')
    bar = _fp32_bar(h32.cpu().numpy())
    err = float((h3 - h32).abs().max())
    assert err <= bar, (err, bar)
    pos3, idx3, _ = ops.decode_heatmaps(h3[:, 0], 1920, 1080, 'table', return_debug=True)
    pos32, idx32, _ = ops.decode_heatmaps(h32[:, 0], 1920, 1080, 'table', return_debug=True)
    sure = _margin_ok(h32[:, 0], bar)
    same = idx3 == idx32
    assert int(sure.sum()) >= 16          # the rule is not vacuous
    assert bool(same[sure].all())
    d = (pos3 - pos32)[:, :2].abs().max(dim=1).values
    assert float(d[sure].max()) <= 1e-2, d
    print('x3 vs SIMT fp32 at 32 x 1280x704: max|dh| %.2e (bar %.2e), maps under the margin rule %d, index match fraction %.4f, '
          'max coord diff there %.2e px' % (err, bar, int(sure.sum()), float(same.float().mean()), float(d[sure].max())))
    for s in (0, 13, 31):
        ref = ohr.wasb_forward(sd, torch.from_numpy(opre.preprocess_stack(list(frames_np[s:s + 3]), 1280, 704))[None]).numpy()
        tol = _fp32_bar(ref)
        assert np.abs(h3[s:s + 1].cpu().numpy() - ref).max() <= tol, s
        ref_pos, ref_idx, _ = odec.decode_heatmaps(ref[:, 0], 1920, 1080, odec.TABLE)
        flat = np.sort(ref.ravel())
        if flat[-1] - flat[-2] > 2 * tol:
            assert int(idx3[s]) == int(ref_idx[0])
            assert np.abs(pos3.cpu().numpy()[s, :2] - ref_pos[0, :2]).max() < 1e-2


@pytest.mark.gpu
def test_x3_batch_invariance_and_profile(dev):
    """A stack's heatmap is bit-identical alone, inside a batch of 5, and with sub-batches of 1 / 4 / 16; the profile shows every
    convolution on an x3 tensor-core kernel (op type 0, none on the SIMT fallback, op type 3)."""
    from upliftingtabletennis_b200._lib import check, lib
    from upliftingtabletennis_b200.detector import WASBNet
    m = WASBNet(dtype='tf32x3').to(dev).eval()
    m.load_state_dict(ohr.random_state_dict(9, 3, seed=5))
    x = torch.from_numpy(np.random.default_rng(6).standard_normal((5, 9, 72, 264)).astype(np.float32)).to(dev)
    runs = []
    try:
        for sb in (16, 4, 1):
            check(lib.ttk_hrnet_set_subbatch(m.engine.h, sb))
            runs.append(m(x)[0])
        alone = m(x[2:3])[0]
    finally:
        check(lib.ttk_hrnet_set_subbatch(m.engine.h, 16))
    for y in runs[1:]:
        assert torch.equal(y, runs[0])
    assert torch.equal(alone[0], runs[0][2])
    # the plan without the fused BasicBlock / bottleneck kernels: 72 convolutions - 13 unread - the final layer, + 3 sums + the final layer
    assert m.engine.last_launches() == 72 - 13 - 1 + 3 + 1
    check(lib.ttk_hrnet_set_profile(m.engine.h, 1))
    try:
        m(x)
        torch.cuda.synchronize()
        ot, ci = C.c_int(), C.c_int()
        types = []
        for i in range(lib.ttk_hrnet_profile_count(m.engine.h)):
            check(lib.ttk_hrnet_profile_read(m.engine.h, i, C.byref(ot), C.byref(ci), None, None, None))
            types.append(ot.value)
    finally:
        check(lib.ttk_hrnet_set_profile(m.engine.h, 0))
    assert types.count(0) == 72 - 13 - 1 and types.count(1) == 3 and types.count(2) == 1 and 3 not in types


@pytest.fixture(scope='module')
def weights(tmp_path_factory):
    """A synthetic weights tree in the reference's checkpoint format (oracle weights)."""
    import os
    from oracle.gen_golden import write_checkpoints
    hub = tmp_path_factory.mktemp('torchhome')
    torch.hub.set_dir(str(hub))
    w = os.path.join(str(hub), 'checkpoints', 'tt_uplifting_extracted', 'weights')
    write_checkpoints(w)
    return w


@pytest.mark.gpu
def test_hub_detectors_x3_match_fp32(weights, golden):
    """ball_detection('wasb', dtype='tf32x3') and table_detection('hrnet', dtype='tf32x3') against the fp32 detectors on the same frames:
    heatmaps within the fp32 bar, decoded positions within 2e-3 image px on maps under the margin rule."""
    import hubconf
    g = golden('interface')
    frames = list(g['frames'])
    triples = [(frames[i - 1], frames[i], frames[i + 1]) for i in range(1, 5)]
    bd3, bd32 = hubconf.ball_detection('wasb', dtype='tf32x3'), hubconf.ball_detection('wasb', dtype='fp32')
    assert bd3.model.compute_dtype == 'tf32x3'
    pos3, hm3 = bd3.predict(triples)
    pos32, hm32 = bd32.predict(triples)
    bar = _fp32_bar(hm32)
    assert np.abs(hm3 - hm32).max() <= bar, (np.abs(hm3 - hm32).max(), bar)
    sure = _margin_ok(torch.from_numpy(hm32[:, 0]), bar).numpy()
    assert np.abs(pos3[sure, :2] - pos32[sure, :2]).max(initial=0.0) <= 2e-3
    td3, td32 = hubconf.table_detection('hrnet', dtype='tf32x3'), hubconf.table_detection('hrnet', dtype='fp32')
    assert td3.model.compute_dtype == 'tf32x3'
    tpos3, thm3 = td3.predict(frames[:2])
    tpos32, thm32 = td32.predict(frames[:2])
    tbar = _fp32_bar(thm32)
    assert np.abs(thm3 - thm32).max() <= tbar, (np.abs(thm3 - thm32).max(), tbar)
    maps = torch.from_numpy(thm32.reshape(-1, *thm32.shape[-2:]))
    tsure = _margin_ok(maps, tbar).numpy().reshape(tpos32.shape[:2])
    assert np.abs(tpos3[..., :2] - tpos32[..., :2])[tsure].max(initial=0.0) <= 2e-3
    print('hub x3 vs fp32: ball maps under the margin rule %d / %d, table %d / %d' % (sure.sum(), sure.size, tsure.sum(), tsure.size))
