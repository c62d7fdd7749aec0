"""The fp16 ('fp16') path of the WASB / HRNet detectors: the bf16 path's kernels with IEEE fp16 storage and operands.  Pre-processing
bit for bit, every convolution of the plan against float64 on fp16-rounded operands, the network against the CPU oracle (and against
stock PyTorch in fp16) and the golden file at TF32's bar, the full-size batch against the SIMT fp32 path, the launch structure, batch
invariance and the hub entry points.  The tests marked gpu need a B200: run with `-m gpu`."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import hrnet as ohr

TF32_BOUND = 1e-2            # TF32's heatmap bar, of max|h_ref|
TF32_COORD_PX = 0.05         # TF32's coordinate bar (image px) on maps under the margin rule
TORCH_FP16_FACTOR, TORCH_FP16_FLOOR = 4.0, 2e-3     # against stock PyTorch in fp16: <= 4x its error + 2e-3 max|h|
CONV_REL, CONV_ABS = 2.0 ** -11, 2e-5                # one fp16 output rounding + fp32 accumulation


def _margin_ok(maps, bound):
    """maps whose top-2 margin exceeds twice the bound"""
    flat = maps.reshape(maps.shape[0], -1)
    top2 = torch.topk(flat, 2, dim=1).values
    return (top2[:, 0] - top2[:, 1]) > 2 * bound


@pytest.fixture(scope='module')
def dev():
    assert torch.cuda.is_available()
    return torch.device('cuda:0')


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


def test_fp16_names_and_storage():
    from upliftingtabletennis_b200 import _lib
    from upliftingtabletennis_b200.precision import canonical, lib_enum, storage_dtype
    for name in ('fp16', 'f16', 'float16', 'half', 'FP16', torch.float16):
        assert canonical(name) == 'fp16'
        assert storage_dtype(name) == torch.float16
    assert lib_enum('half') == _lib.F16 == 4
    assert storage_dtype('bf16') == torch.bfloat16 and storage_dtype('tf32') == torch.float32
    with pytest.raises(ValueError):
        canonical('fp8')


def test_fp16_accepted_without_gpu():
    """The HRNet shells take 'fp16' through dtype= and compute_dtype; the workspace of the 2-byte path is the bf16 one."""
    from upliftingtabletennis_b200 import _lib
    from upliftingtabletennis_b200.detector import MyHRNet, WASBNet
    m = WASBNet(dtype='fp16')
    assert m.compute_dtype == 'fp16' and m.storage_dtype == torch.float16
    m.compute_dtype = 'tf32'
    m.compute_dtype = 'half'
    assert m.compute_dtype == 'fp16'
    t = MyHRNet(dtype=torch.float16)
    assert t.compute_dtype == 'fp16' and MyHRNet().compute_dtype == 'tf32'
    for B, H, W in ((2, 704, 1280), (1, 88, 160), (40, 64, 200)):
        ws = _lib.lib.ttk_hrnet_workspace_bytes(m.engine.h, B, H, W, _lib.F16)
        assert ws > 0 and ws == _lib.lib.ttk_hrnet_workspace_bytes(m.engine.h, B, H, W, _lib.BF16)


def test_fp16_refused_by_vitpose_and_uplift():
    from upliftingtabletennis_b200.uplift import get_model
    from upliftingtabletennis_b200.vitpose import VitPose
    with pytest.raises(NotImplementedError):
        VitPose(in_frames=3, resolution=(160, 96), dtype='fp16')
    with pytest.raises(NotImplementedError):
        get_model('connectstage', 'large', 'dynamic', 'new', dtype=torch.float16)
    up = get_model('connectstage', 'large', 'dynamic', 'new')
    with pytest.raises(NotImplementedError):
        up.compute_dtype = 'half'


def test_pipeline_fp16_refused_before_weights(tmp_path, monkeypatch):
    """TableTennisPipeline(dtype='fp16') raises before any weights are located: the hub directory stays untouched."""
    from upliftingtabletennis_b200 import interface
    hub = tmp_path / 'torchhome'
    monkeypatch.setattr(torch.hub, 'get_dir', lambda: str(hub))

    def no_weights(*a, **k):
        raise AssertionError('weights were looked up')
    monkeypatch.setattr(interface, '_get_weights_path', no_weights)
    for dt in ('fp16', torch.float16, 'half'):
        with pytest.raises(NotImplementedError, match='compute_dtype'):
            interface.TableTennisPipeline(dtype=dt)
    assert not hub.exists()


@pytest.mark.gpu
@pytest.mark.parametrize('res', [(1280, 704), (1920, 1088)])
def test_preprocess_fp16_bit_exact(dev, res):
    """NHWC16 fp16 = the float32 values rounded to nearest-even (channels 9..15 zero), 1080p sources."""
    from oracle.gen_golden import synthetic_frames
    from upliftingtabletennis_b200 import ops
    frames = synthetic_frames(np.random.default_rng(7), 4, 1080, 1920)
    w, h = res
    fd = torch.from_numpy(np.stack(frames)).to(dev)
    nhwc = ops.preprocess_stacks(fd, 3, 1, 2, w, h, layout='nhwc16', dtype=torch.float32)
    nh = ops.preprocess_stacks(fd, 3, 1, 2, w, h, layout='nhwc16', dtype=torch.float16)
    assert nh.dtype == torch.float16 and torch.equal(nh, nhwc.to(torch.float16))
    # single-frame stacks at the source size (the un-staged kernel)
    src = fd[:, :h // 2, :w // 2].contiguous()
    n1 = ops.preprocess_stacks(src, 1, 1, 2, w // 2, h // 2, layout='nhwc16', dtype=torch.float16)
    assert torch.equal(n1, ops.preprocess_stacks(src, 1, 1, 2, w // 2, h // 2, layout='nhwc16', dtype=torch.float32).to(torch.float16))
    with pytest.raises(ValueError):
        ops.preprocess_stacks(fd, 3, 1, 2, w, h, layout='nhwc16', dtype=torch.float64)


@pytest.mark.gpu
@pytest.mark.parametrize('shape', [(2, 24, 200), (1, 10, 130), (1, 40, 72), (1, 16, 520)])
def test_every_conv_f16_vs_float64(dev, shape):
    """ttk_hrnet_debug_conv_f16 for every convolution of the plan, tcgen05 and SIMT (bias, residual on / off, ReLU), against a float64
    convolution of the fp16-rounded input, weights and residual: |y - ref| <= 2^-11 |ref| + 2e-5 (max|ref| + 1).  Padded output
    channels are zero.  Every convolution has a tcgen05 kernel."""
    from upliftingtabletennis_b200._lib import lib, ptr, stream_ptr
    from upliftingtabletennis_b200.detector import WASBNet
    m = WASBNet().to(dev).eval()
    sd = ohr.random_state_dict(9, 3, seed=123)
    m.load_state_dict(sd)
    m._sync()
    eng = m.engine
    n, H, W = shape
    rng = np.random.default_rng(H * W + 1)
    specs = ohr.conv_specs(9, 3)
    worst = {0: 0.0, 1: 0.0}
    for idx, (name, bn, cin, cout, k, stride) in enumerate(eng.specs[:-1]):
        cin_p, cout_p = (cin + 15) // 16 * 16, (cout + 15) // 16 * 16
        x = torch.zeros((n, H, W, cin_p), dtype=torch.float16)
        x[..., :cin] = torch.from_numpy(rng.standard_normal((n, H, W, cin)).astype(np.float32)).half()
        Ho, Wo = (H + stride - 1) // stride, (W + stride - 1) // stride
        res = torch.zeros((n, Ho, Wo, cout_p), dtype=torch.float16)
        res[..., :cout] = torch.from_numpy(rng.standard_normal((n, Ho, Wo, cout)).astype(np.float32)).half()
        xd, rd = x.to(dev), res.to(dev)
        w, b = ohr.fold_bn(sd, specs[idx])
        w16 = torch.from_numpy(w.astype(np.float32)).half().double()         # the host folds in fp64, rounds to fp32, then to fp16
        conv = F.conv2d(x[..., :cin].permute(0, 3, 1, 2).double(), w16, None, stride=stride, padding=k // 2)
        conv = conv + torch.from_numpy(b.astype(np.float32)).double()[None, :, None, None]
        for simt in (0, 1):
            for use_res in (True, False):
                out = torch.full((n, Ho, Wo, cout_p), float('nan'), dtype=torch.float16, device=dev)
                rc = lib.ttk_hrnet_debug_conv_f16(eng.h, idx, ptr(xd), n, H, W, ptr(rd) if use_res else None, 1, simt, ptr(out), stream_ptr())
                torch.cuda.synchronize()
                assert rc == 0, (name, simt, rc)
                ref = conv + res[..., :cout].permute(0, 3, 1, 2).double() if use_res else conv
                ref = torch.relu(ref).permute(0, 2, 3, 1)
                y = out.cpu().double()
                assert torch.isfinite(y).all(), (name, simt)
                err = (ref - y[..., :cout]).abs()
                bar = CONV_REL * ref.abs() + CONV_ABS * (float(ref.abs().max()) + 1.0)
                assert bool((err <= bar).all()), (name, simt, use_res, float(err.max()), float((err / bar).max()))
                worst[simt] = max(worst[simt], float((err / bar).max()))
                if cout_p > cout:
                    assert float(y[..., cout:].abs().max()) == 0.0, (name, simt)
    print('fp16 convolutions %s: worst error / bar = %.3f (tcgen05), %.3f (SIMT)' % (shape, worst[0], worst[1]))
    bad = torch.zeros((1, 8, 8, 16), dtype=torch.float16, device=dev)
    assert lib.ttk_hrnet_debug_conv_f16(eng.h, len(eng.specs) - 1, ptr(bad), 1, 8, 8, None, 1, 0, ptr(bad), stream_ptr()) == -1


def _torch_fp16(forward, sd, x, dev):
    """Stock PyTorch in fp16 on this GPU: the oracle's functional forward (F.conv2d + eval-mode F.batch_norm, cuDNN) with every
    floating-point tensor of the state dict and the input cast to float16."""
    sd16 = {k: (v.to(dev).half() if v.is_floating_point() else v.to(dev)) for k, v in sd.items()}
    with torch.no_grad():
        return forward(sd16, torch.from_numpy(x).to(dev).half()).float().cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize('shape', [(1, 88, 160), (3, 40, 72), (2, 8, 8), (2, 64, 200)])
def test_network_f16_vs_oracle(dev, shape):
    """WASB and the 13-channel HRNet on the fp16 path against the CPU oracle: TF32's bar, and within 4x the error of stock PyTorch in
    fp16 (plus 2e-3 max|h|)."""
    from upliftingtabletennis_b200.detector import MyHRNet, WASBNet
    B, H, W = shape
    rng = np.random.default_rng(B * 1000 + H + 7)
    cases = []
    sd = ohr.random_state_dict(9, 3, seed=77)
    x = rng.standard_normal((B, 9, H, W)).astype(np.float32)
    m = WASBNet(dtype='fp16').to(dev).eval()
    m.load_state_dict(sd)
    cases.append(('wasb', m(torch.from_numpy(x).to(dev))[0].cpu().numpy(), ohr.wasb_forward(sd, torch.from_numpy(x)).numpy(),
                  _torch_fp16(ohr.wasb_forward, sd, x, dev)))
    sdt = ohr.random_state_dict(3, 13, seed=78)
    xt = rng.standard_normal((B, 3, H, W)).astype(np.float32)
    t = MyHRNet(dtype=torch.float16).to(dev).eval()
    t.load_state_dict(sdt)
    cases.append(('hrnet', t(torch.from_numpy(xt).to(dev)).cpu().numpy(), ohr.hrnet_forward(sdt, torch.from_numpy(xt)).numpy(),
                  _torch_fp16(ohr.hrnet_forward, sdt, xt, dev)))
    for name, y, ref, y_torch in cases:
        assert y.shape == ref.shape and np.isfinite(y).all()
        scale = float(np.abs(ref).max())
        err, err_torch = float(np.abs(y - ref).max()), float(np.abs(y_torch - ref).max())
        assert err <= TF32_BOUND * scale, (name, err, scale)
        assert err <= TORCH_FP16_FACTOR * err_torch + TORCH_FP16_FLOOR * scale, (name, err, err_torch, scale)
        print('%s %s: fp16 max|d|/max|h| %.2e, stock PyTorch fp16 %.2e' % (name, shape, err / scale, err_torch / scale))


@pytest.mark.gpu
def test_network_f16_golden(dev, golden):
    from upliftingtabletennis_b200.detector import MyHRNet, WASBNet
    g = golden('hrnet')
    m = WASBNet(dtype='fp16').to(dev).eval()
    m.load_state_dict(ohr.random_state_dict(9, 3, seed=int(g['wasb_seed'])))
    y, _ = m(torch.from_numpy(g['wasb_x']).to(dev))
    np.testing.assert_allclose(y.cpu().numpy(), g['wasb_y'], rtol=0, atol=TF32_BOUND * np.abs(g['wasb_y']).max())
    t = MyHRNet(dtype='fp16').to(dev).eval()
    t.load_state_dict(ohr.random_state_dict(3, 13, seed=int(g['table_seed'])))
    yt = t(torch.from_numpy(g['table_x']).to(dev))
    np.testing.assert_allclose(yt.cpu().numpy(), g['table_y'], rtol=0, atol=TF32_BOUND * np.abs(g['table_y']).max())


@pytest.mark.gpu
def test_full_size_f16_vs_simt_fp32(dev):
    """32 stacks of 1080p frames with a moving blob -> WASB @1280x704 on the fp16 path against the SIMT fp32 path on the same GPU:
    finite, TF32's heatmap bar, the same peak index on every map under the margin rule, decoded coordinates within 0.05 px there and
    within one heatmap pixel elsewhere; fp16's max-abs error is below bf16's on the same batch."""
    from upliftingtabletennis_b200 import ops, synthetic
    from upliftingtabletennis_b200.detector import WASBNet
    B = 32
    frames = torch.from_numpy(synthetic.frames_1080p(B + 2, seed=100)).to(dev)
    sd = synthetic.hrnet_blob_state_dict(ohr.state_dict_layout(9, 3), seed=1)
    m = WASBNet(dtype='fp16').to(dev).eval()
    m.load_state_dict(sd)
    x32 = ops.preprocess_stacks(frames, 3, 1, B, 1280, 704, layout='nhwc16', dtype=torch.float32)
    h32 = m.heatmaps_from_nhwc16(x32, 'fp32')
    h16 = m.heatmaps_from_nhwc16(ops.preprocess_stacks(frames, 3, 1, B, 1280, 704, layout='nhwc16', dtype=torch.float16))
    hb = m.heatmaps_from_nhwc16(ops.preprocess_stacks(frames, 3, 1, B, 1280, 704, layout='nhwc16', dtype=torch.bfloat16))
    assert bool(torch.isfinite(h16).all())
    scale = float(h32.abs().max())
    err, err_bf16 = float((h16 - h32).abs().max()), float((hb - h32).abs().max())
    assert err <= TF32_BOUND * scale, (err, scale)
    assert err < err_bf16, (err, err_bf16)
    pos16, idx16, _ = ops.decode_heatmaps(h16[:, 0], 1920, 1080, 'table', return_debug=True)
    pos32, idx32, _ = ops.decode_heatmaps(h32[:, 0], 1920, 1080, 'table', return_debug=True)
    sure = _margin_ok(h32[:, 0], TF32_BOUND * scale)
    same = idx16 == idx32
    assert int(sure.sum()) >= 16          # the rule is not vacuous
    assert bool(same[sure].all())
    d = (pos16 - pos32)[:, :2].abs().max(dim=1).values
    assert float(d[sure].max()) <= TF32_COORD_PX, d
    assert float(d.max()) <= 1920 / 1280 + TF32_COORD_PX, d
    print('fp16 vs SIMT fp32 at 32 x 1280x704: max|dh|/max|h| %.2e (bf16 %.2e), maps under the margin rule %d, index match fraction '
          '%.4f, max coord diff %.2e px (%.2e under the rule)' % (err / scale, err_bf16 / scale, int(sure.sum()), float(same.float().mean()),
                                                                 float(d.max()), float(d[sure].max())))


def _profile_types(m, x):
    from upliftingtabletennis_b200._lib import check, lib
    check(lib.ttk_hrnet_set_profile(m.engine.h, 1))
    try:
        y = m.heatmaps_from_nhwc16(x)
        torch.cuda.synchronize()
        ot, ci = C.c_int(), C.c_int()
        types = []
        for i in range(lib.ttk_hrnet_profile_count(m.engine.h)):
            check(lib.ttk_hrnet_profile_read(m.engine.h, i, C.byref(ot), C.byref(ci), None, None, None))
            types.append((ot.value, ci.value))
    finally:
        check(lib.ttk_hrnet_set_profile(m.engine.h, 0))
    return y, types


@pytest.mark.gpu
def test_f16_structure(dev):
    """The fp16 forward launches exactly the bf16 forward's kernels (launch count and profile op sequence, fused blocks and bottleneck
    included); without block fusion it has 12 more launches, and forced SIMT agrees with tcgen05, both within TF32's bar."""
    from upliftingtabletennis_b200._lib import check, lib
    from upliftingtabletennis_b200.detector import WASBNet
    m = WASBNet(dtype='fp16').to(dev).eval()
    m.load_state_dict(ohr.random_state_dict(9, 3, seed=5))
    x = torch.from_numpy(np.random.default_rng(6).standard_normal((3, 72, 264, 16)).astype(np.float32)).to(dev)
    x[..., 9:] = 0
    y16, t16 = _profile_types(m, x.half())
    n16 = m.engine.last_launches()
    _, tb = _profile_types(m, x.bfloat16())
    assert n16 == m.engine.last_launches() and t16 == tb
    assert 3 not in [t for t, _ in t16]          # no convolution on the SIMT fallback
    scale = float(y16.abs().max())
    try:
        check(lib.ttk_hrnet_set_block_fusion(m.engine.h, 0))
        y_nf = m.heatmaps_from_nhwc16(x.half())
        assert m.engine.last_launches() == n16 + 12
    finally:
        check(lib.ttk_hrnet_set_block_fusion(m.engine.h, 1))
    try:
        check(lib.ttk_hrnet_set_force_simt(m.engine.h, 1))
        y_simt = m.heatmaps_from_nhwc16(x.half())
    finally:
        check(lib.ttk_hrnet_set_force_simt(m.engine.h, 0))
    assert float((y_nf - y16).abs().max()) <= TF32_BOUND * scale
    assert float((y_simt - y16).abs().max()) <= TF32_BOUND * scale
    print('fp16 structure: %d launches; no fusion max|d|/max|h| %.2e, SIMT %.2e' % (
        n16, float((y_nf - y16).abs().max()) / scale, float((y_simt - y16).abs().max()) / scale))


@pytest.mark.gpu
def test_f16_batch_invariance(dev):
    """A stack's heatmap is bit-identical alone, inside a batch of 5, and with sub-batches of 16 / 4 / 1."""
    from upliftingtabletennis_b200._lib import check, lib
    from upliftingtabletennis_b200.detector import WASBNet
    m = WASBNet(dtype='fp16').to(dev).eval()
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


@pytest.mark.gpu
def test_hub_detectors_f16_match_fp32(weights, golden):
    """ball_detection('wasb', dtype='fp16') and table_detection('hrnet', dtype=torch.float16) against the fp32 detectors on the same
    frames: heatmaps within TF32's bar, decoded positions within 0.05 image px on maps under the margin rule and within one heatmap
    pixel elsewhere."""
    import hubconf
    g = golden('interface')
    frames = list(g['frames'])
    img_w = frames[0].shape[1]
    triples = [(frames[i - 1], frames[i], frames[i + 1]) for i in range(1, 5)]
    bd16, bd32 = hubconf.ball_detection('wasb', dtype='fp16'), hubconf.ball_detection('wasb', dtype='fp32')
    assert bd16.model.compute_dtype == 'fp16'
    pos16, hm16 = bd16.predict(triples)
    pos32, hm32 = bd32.predict(triples)
    bar = TF32_BOUND * np.abs(hm32).max()
    assert np.abs(hm16 - hm32).max() <= bar, (np.abs(hm16 - hm32).max(), bar)
    sure = _margin_ok(torch.from_numpy(hm32[:, 0]), bar).numpy()
    d = np.abs(pos16[:, :2] - pos32[:, :2]).max(axis=1)
    assert d[sure].max(initial=0.0) <= TF32_COORD_PX
    assert d.max() <= img_w / hm32.shape[-1] + TF32_COORD_PX, d
    td16, td32 = hubconf.table_detection('hrnet', dtype=torch.float16), hubconf.table_detection('hrnet', dtype='fp32')
    assert td16.model.compute_dtype == 'fp16'
    tpos16, thm16 = td16.predict(frames[:2])
    tpos32, thm32 = td32.predict(frames[:2])
    tbar = TF32_BOUND * np.abs(thm32).max()
    assert np.abs(thm16 - thm32).max() <= tbar, (np.abs(thm16 - thm32).max(), tbar)
    maps = torch.from_numpy(thm32.reshape(-1, *thm32.shape[-2:]))
    tsure = _margin_ok(maps, tbar).numpy().reshape(tpos32.shape[:2])
    td = np.abs(tpos16[..., :2] - tpos32[..., :2]).max(axis=-1)
    assert td[tsure].max(initial=0.0) <= TF32_COORD_PX
    assert td.max() <= img_w / thm32.shape[-1] + TF32_COORD_PX, td
    print('hub fp16 vs fp32: ball maps under the margin rule %d / %d, table %d / %d' % (sure.sum(), sure.size, tsure.sum(), tsure.size))
