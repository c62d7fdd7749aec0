"""Uplifting transformer at its input edges.

The tf32x3 path's two kernels (gemm3_umma.cu, uplift3.cu's attention) against float64 through their test hooks, and the whole model in
all three precisions against the fp32 oracle on inputs the golden fixtures never reach: sequence lengths on both sides of every attention
template switch (T = 51 / 52 / 53, the longest T = 63), odd B T (a half-filled CTA in the table-token stage), trajectories with 0, 1 or 2
valid frames or with holes, no / all table keypoints visible, times seconds into a clip with gaps, the tf32x3 chunk boundary, and the
reference's second mask format {-1e9, 0}.  The tests without the gpu marker check the float64 reference and the input generator on the
CPU."""
import math

import numpy as np
import pytest
import torch

from oracle import uplift as oup

UPLIFT_ATOL, UPLIFT_RTOL = 1e-4, 1e-4          # the fp32-level bar of test_gpu_parity.py
NTAB, D, HEADS, HD = 13, 128, 4, 32
EDGE_SHAPES = [(1, 2), (3, 3), (5, 13), (4, 51), (3, 52), (3, 53), (5, 63)]
FPS = (25.0, 30.0, 50.0, 60.0, 120.0)
OFFSETS = (0.0, 3.3, 60.0)


# ------------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------------
def edge_trajectories(rng, B, T):
    """(ball (B,T,2), table (B,13,3), mask (B,T), times (B,T)) float32, padded rows zero as _uplifting_transform writes them.
    Trajectory b takes the b-th entry of: holes (a valid prefix with frames 1 and T // 2 dropped), 0 valid frames, T, 1, 2, T - 1;
    table visibility none / all / mixed and a time offset of 0, 3.3 or 60 s in turn; frames are 1 to 3 frame periods apart."""
    ball = np.zeros((B, T, 2), np.float32)
    mask = np.zeros((B, T), np.float32)
    times = np.zeros((B, T), np.float32)
    table = np.zeros((B, NTAB, 3), np.float32)
    for b in range(B):
        kind = ('holes', 0, T, 1, 2, T - 1)[b % 6]
        n = max(T - 1, 1) if kind == 'holes' else kind
        fps = float(rng.choice(FPS))
        dt = np.cumsum(rng.choice([1, 1, 1, 2, 3], n)) / fps
        ball[b, :n, 0] = 0.2 + 0.3 * dt + rng.normal(0, 0.002, n)
        ball[b, :n, 1] = 0.6 - 1.2 * dt + 2.5 * dt * dt + rng.normal(0, 0.002, n)
        times[b, :n] = OFFSETS[b % 3] + dt
        mask[b, :n] = 1.0
        if kind == 'holes':
            mask[b, [1, T // 2]] = 0.0
        table[b, :, 0] = rng.uniform(0.2, 0.8, NTAB)
        table[b, :, 1] = rng.uniform(0.4, 0.9, NTAB)
        vis = (np.zeros(NTAB), np.ones(NTAB), np.arange(NTAB) % 3 != 0)[b % 3]
        table[b, :, 2] = vis
    return ball, table, mask, times


def additive(mask):
    """{0, 1} -> the reference's other mask format {-1e9, 0}."""
    return np.where(mask == 0, np.float32(-1e9), np.float32(0.0)).astype(np.float32)


# ------------------------------------------------------------------------------------------------
# float64 reference of the attention kernel (order of operations of oracle.uplift.attention)
# ------------------------------------------------------------------------------------------------
def stage_layout(mode, table, mask, times, mask_additive):
    """Per stage: sequence length, row masks (float64, additive), row times (float32, NaN = not rotated)."""
    table, mask, times = (np.asarray(a, np.float32) for a in (table, mask, times))
    B, T = mask.shape
    m = mask.astype(np.float64) if mask_additive else np.where(mask == 0, -np.inf, 0.0)
    if mode == 0:
        tm = np.concatenate([np.zeros((B, 1)), np.where(table[:, :, 2] == 1, 0.0, -np.inf)], 1)
        tt = np.concatenate([[np.nan], np.arange(NTAB, dtype=np.float32) / np.float32(100.0)]).astype(np.float32)
        return NTAB + 1, np.repeat(tm, T, 0), np.broadcast_to(tt, (B * T, NTAB + 1))
    if mode == 1:
        return T, m, times
    return T + 1, np.concatenate([np.zeros((B, 1)), m], 1), np.concatenate([np.full((B, 1), np.nan, np.float32), times], 1)


def attention_ref(mode, qkv, table, mask, times, inv_freq, mask_additive=False, first_only=False):
    """float64 attention of qkv [rows][384] (bias included) -> [rows][128] ([sequences][128] when first_only).
    The RoPE angle is formed in float32 like the reference and the kernels: pos = rint(t / 0.002f), angle = pos * inv_freq; a float64
    angle would differ by up to ulp(angle) ~ 1e-3 rad at a minute into a clip.  A finite mask is added in float32, again like the
    reference: -1e9 absorbs the score (ulp(1e9) = 64), so a padded query row weighs the valid keys uniformly."""
    S, m, t = stage_layout(mode, table, mask, times, mask_additive)
    nseq = m.shape[0]
    x = torch.as_tensor(np.asarray(qkv, np.float64)).view(nseq, S, 3, HEADS, HD).permute(2, 0, 3, 1, 4)
    q, k, v = x[0], x[1], x[2]
    pos = np.rint(t / np.float32(0.002)).astype(np.float32)
    ang = torch.as_tensor((pos[:, :, None] * np.asarray(inv_freq, np.float32)[None, None, :]).astype(np.float64))
    rot = ~torch.isnan(ang)
    c = torch.where(rot, torch.cos(ang), torch.ones_like(ang))[:, None]
    s = torch.where(rot, torch.sin(ang), torch.zeros_like(ang))[:, None]

    def rope(a):
        out = torch.empty_like(a)
        out[..., 0::2] = a[..., 0::2] * c - a[..., 1::2] * s
        out[..., 1::2] = a[..., 0::2] * s + a[..., 1::2] * c
        return out
    q, k = rope(q), rope(k)
    sc = (q @ k.transpose(-2, -1)) / math.sqrt(HD)
    mm = torch.as_tensor(m)
    msum = (mm[:, None, None, :] + mm[:, None, :, None]).expand_as(sc)
    finite = torch.isfinite(msum) & (msum != 0)
    sc = torch.where(finite, (sc + msum).float().double(), sc + msum)
    mx = sc.max(-1, keepdim=True).values
    mx = torch.where(torch.isinf(mx), torch.zeros_like(mx), mx)
    e = torch.exp(sc - mx)
    den = e.sum(-1, keepdim=True)
    a = torch.where(den > 0, e / den, torch.zeros_like(e))
    o = (a @ v).transpose(1, 2).reshape(nseq, S, D)
    return (o[:, 0] if first_only else o.reshape(nseq * S, D)).numpy()


def attention_inputs(mode, B, T, seed):
    rng = np.random.default_rng(seed)
    ball, table, mask, times = edge_trajectories(rng, B, T)
    S = NTAB + 1 if mode == 0 else (T if mode == 1 else T + 1)
    nseq = B * T if mode == 0 else B
    qkv = (rng.standard_normal((nseq * S, 3 * D)) * 1.5).astype(np.float32)
    inv = oup.random_state_dict(0)['firststage.layers.0.attn.rotary_emb.inv_freq'].numpy()
    return qkv, table, mask, times, inv


# ------------------------------------------------------------------------------------------------
# CPU checks: the reference, the specification of the mask formats, the generator
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('mask_additive', [False, True])
@pytest.mark.parametrize('mode,T', [(0, 3), (1, 2), (1, 53), (2, 2), (2, 63)])
def test_attention_reference_matches_oracle(mode, T, mask_additive):
    """The float64 reference above agrees with oracle.uplift.attention (float32) at float32 level on the edge inputs."""
    B = 3
    _, table, mask, times, inv = attention_inputs(mode, B, T, seed=10 * T + mode)
    if mask_additive:
        mask = additive(mask)
    S, m, t = stage_layout(mode, table, mask, times, mask_additive)
    nseq = m.shape[0]
    # the oracle takes the layer input: its qkv projection, repeated here in float32, gives the rows of the reference; the output
    # projection is the identity
    g = torch.Generator().manual_seed(mode)
    x = torch.randn(nseq, S, D, generator=g)
    sd = {'p.attn.qkv.weight': torch.randn(3 * D, D, generator=g) * 0.15, 'p.attn.qkv.bias': torch.randn(3 * D, generator=g) * 0.1,
          'p.attn.proj.weight': torch.eye(D), 'p.attn.rotary_emb.inv_freq': torch.from_numpy(inv)}
    qkv = torch.nn.functional.linear(x, sd['p.attn.qkv.weight'], sd['p.attn.qkv.bias']).reshape(nseq * S, 3 * D).numpy()
    ref = attention_ref(mode, qkv, table, mask, times, inv, mask_additive)
    tt = torch.from_numpy(np.ascontiguousarray(t if mode == 1 else t[:, 1:]))
    out = oup.attention(sd, 'p.', x, torch.from_numpy(m.astype(np.float32)), tt, 0 if mode == 1 else 1, HEADS)
    err = np.abs(out.reshape(-1, D).double().numpy() - ref).max()
    assert err <= 4e-6 * np.abs(ref).max() + 1e-6, (err, np.abs(ref).max())


def test_oracle_mask_formats():
    """The reference's semantics that ttk_uplift_forward(mask_additive = 1) implements: with {-1e9, 0} masks, valid rows of pos and
    rot equal the {0, 1} result bit for bit, padded rows differ (they attend over the valid frames instead of nothing)."""
    ball, table, mask, times = edge_trajectories(np.random.default_rng(0), 5, 13)
    sd = oup.random_state_dict(5)
    args = [torch.from_numpy(a) for a in (ball, table, mask, times)]
    r1, p1 = oup.uplift_forward(sd, *args)
    r2, p2 = oup.uplift_forward(sd, args[0], args[1], torch.from_numpy(additive(mask)), args[3])
    v = torch.from_numpy(mask).bool()
    assert torch.equal(r1, r2) and torch.equal(p1[v], p2[v])
    assert (p1[~v] - p2[~v]).abs().max() > 0.1


@pytest.mark.parametrize('B,T', EDGE_SHAPES)
def test_edge_generator(B, T):
    """Every batch has a padded frame and a valid one (both mask formats accept it), and the shapes promised above."""
    ball, table, mask, times = edge_trajectories(np.random.default_rng(B * T), B, T)
    assert mask.min() == 0 and mask.max() == 1
    counts = mask.sum(1)
    assert counts[0] < T and mask[0, 0] == 1                      # holes
    if B > 1:
        assert counts[1] == 0
    if B > 2:
        assert counts[2] == T and (table[1, :, 2] == 1).all() and (table[0, :, 2] == 0).all()
    assert times.max() > 60.0 or B < 3
    assert (B * T) % 2 == (1 if (B, T) in ((3, 3), (5, 13), (3, 53), (5, 63)) else 0)


# ------------------------------------------------------------------------------------------------
# GPU: kernels against float64
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def dev():
    assert torch.cuda.is_available(), 'gpu tests need a CUDA device'
    from upliftingtabletennis_b200 import _lib
    _lib.require_device()
    return torch.device('cuda:0')


def _rna_tf32(t):
    """tf32(x) rounded to nearest, ties away (cvt.rna), as the library splits the weights."""
    b = t.contiguous().view(torch.int32)
    return ((b + 0x1000) & ~0x1FFF).view(torch.float32)


GEMM3_LAYERS = {          # name: N, LayerNorm on load, bias, ReLU, residual (aliasing C), out_stats -- the four calls of a layer
    'qkv': (384, True, True, 0, False, False),
    'proj': (128, False, False, 0, True, True),
    'fc1': (128, True, True, 1, False, False),
    'fc2': (128, False, True, 0, True, True),
}
GEMM3_M = [1, 2, 28, 128, 129, 700, 3 * 148 * 128 + 77]


@pytest.mark.gpu
@pytest.mark.parametrize('layer,M,big_mean', [(layer, M, False) for layer in GEMM3_LAYERS for M in GEMM3_M] +
                         [(layer, M, True) for layer in GEMM3_LAYERS for M in (129, 700)])
def test_gemm3_vs_float64(dev, layer, M, big_mean):
    """gemm3 against float64 with the kernel's own float32 LayerNorm statistics as inputs.  M = 3 148 128 + 77 walks every CTA over at
    least three tiles (accumulator double buffer and ring phases wrapping); big_mean rows (mean 50, std 0.05) stress LayerNorm on load
    and the row statistics of the output.  out_stats is checked against float64 statistics of the kernel's own C, which separates the
    two-pass / Chan-merge arithmetic from the GEMM.  Measured on a B200 (1000 W): C 1.3e-6 of max|C| (bar 1e-5), mean 4.9e-7 of
    |mean| + std (bar 1e-6), rstd 4.5e-6 relative (bar 1e-5; 2.6e-5 on the big-mean rows before the epilogue took its chunk sums about
    the row's first value)."""
    from upliftingtabletennis_b200._lib import check, lib, ptr, stream_ptr
    N, ln, has_bias, relu, res, stats = GEMM3_LAYERS[layer]
    g = torch.Generator(device='cpu').manual_seed(M * 7 + N + big_mean)
    A = torch.randn(M, D, generator=g)
    if big_mean:
        A = 50.0 + 0.05 * A if ln else 0.01 * A
    W = torch.randn(N, D, generator=g) / D ** 0.5
    bias = torch.randn(N, generator=g) * 0.1 if has_bias else None
    gamma = torch.rand(D, generator=g) * 0.4 + 0.8
    beta = torch.randn(D, generator=g) * 0.05
    R = (50.0 + 0.05 * torch.randn(M, N, generator=g)) if big_mean else torch.randn(M, N, generator=g)
    st = None
    if ln:
        a64 = A.double()
        mu = a64.mean(1)
        st = torch.stack([mu, 1.0 / torch.sqrt(((a64 - mu[:, None]) ** 2).mean(1) + 1e-5)], 1).float()
    A, W, gamma, beta, R = (t.to(dev) for t in (A, W, gamma, beta, R))
    bias = bias.to(dev) if bias is not None else None
    st = st.to(dev) if st is not None else None
    w_hi = _rna_tf32(W)
    w_lo = (W - w_hi).contiguous()
    C = R.clone() if res else torch.full((M, N), float('nan'), device=dev)
    out_stats = torch.full((M, 2), float('nan'), device=dev) if stats else None
    check(lib.ttk_uplift_debug_gemm3(ptr(A), ptr(w_hi), ptr(w_lo), ptr(bias), ptr(C) if res else None, ptr(C), M, N, relu, ptr(st),
                                     ptr(gamma) if ln else None, ptr(beta) if ln else None, ptr(out_stats), stream_ptr()))
    torch.cuda.synchronize()
    a = A.double()
    if ln:
        a = (a - st[:, :1].double()) * st[:, 1:].double() * gamma.double() + beta.double()
    ref = a @ W.double().t()
    if bias is not None:
        ref = ref + bias.double()
    if relu:
        ref = torch.relu(ref)
    if res:
        ref = ref + R.double()
    err = (C.double() - ref).abs().max().item()
    scale = ref.abs().max().item()
    print('gemm3 %s M %d big_mean %d: max|C - ref| = %.2e of max|ref| %.2e' % (layer, M, big_mean, err, scale))
    assert err <= 1e-5 * scale, (err, scale)
    if stats:
        c = C.double()
        mu = c.mean(1)
        sd = ((c - mu[:, None]) ** 2).mean(1).sqrt()
        rstd = 1.0 / torch.sqrt(sd ** 2 + 1e-5)
        e_mu = ((out_stats[:, 0].double() - mu).abs() / (mu.abs() + sd)).max().item()
        e_rs = ((out_stats[:, 1].double() - rstd).abs() / rstd).max().item()
        print('gemm3 %s M %d big_mean %d: stats mean %.2e, rstd %.2e relative' % (layer, M, big_mean, e_mu, e_rs))
        assert e_mu <= 1e-6 and e_rs <= 1e-5, (e_mu, e_rs)


@pytest.mark.gpu
def test_gemm3_rejects_stats_of_wide_output(dev):
    from upliftingtabletennis_b200._lib import lib, ptr, stream_ptr
    a = torch.zeros(4, D, device=dev)
    w = torch.zeros(384, D, device=dev)
    c = torch.zeros(4, 384, device=dev)
    s = torch.zeros(4, 2, device=dev)
    assert lib.ttk_uplift_debug_gemm3(ptr(a), ptr(w), ptr(w), None, None, ptr(c), 4, 384, 0, None, None, None, ptr(s), stream_ptr()) == -4
    assert b'row statistics need N = 128' in lib.ttk_last_error()


ATTENTION_CASES = [           # (mode, first_only, B, T): table-token stage with B T odd, both sides of the SMAX switches, T = 2 and 63
    (0, False, 3, 3), (0, True, 3, 3), (0, False, 5, 13), (0, True, 5, 13),
    (1, False, 3, 2), (1, False, 4, 52), (1, False, 5, 53), (1, False, 5, 63),
    (2, False, 3, 2), (2, False, 4, 51), (2, False, 5, 52), (2, False, 5, 63),
]


@pytest.mark.gpu
@pytest.mark.parametrize('mask_additive', [False, True])
@pytest.mark.parametrize('mode,first_only,B,T', ATTENTION_CASES)
def test_attention3_vs_float64(dev, mode, first_only, B, T, mask_additive):
    """attention3 (the instantiation the model picks for this stage and T) against float64 on edge masks, no / all / some table
    keypoints visible and times up to a minute into a clip.  Measured on a B200 (1000 W): at most 0.11 of the bar (2.1e-6 at max|ref| 4.7)."""
    from upliftingtabletennis_b200._lib import check, lib, ptr, stream_ptr
    qkv, table, mask, times, inv = attention_inputs(mode, B, T, seed=100 * T + 10 * mode + first_only)
    if mask_additive:
        mask = additive(mask)
    ref = attention_ref(mode, qkv, table, mask, times, inv, mask_additive, first_only)
    t = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (qkv, table, mask, times, inv)]
    o = torch.full(ref.shape, float('nan'), device=dev)
    check(lib.ttk_uplift_debug_attention3(mode, int(first_only), ptr(t[0]), ptr(o), ptr(t[1]), ptr(t[2]), ptr(t[3]), ptr(t[4]), B, T,
                                          int(mask_additive), stream_ptr()))
    torch.cuda.synchronize()
    err = np.abs(o.cpu().double().numpy() - ref).max()
    scale = np.abs(ref).max()
    print('attention3 mode %d first_only %d B %d T %d additive %d: max err %.2e of max|ref| %.2e' % (mode, first_only, B, T, mask_additive, err, scale))
    assert err <= 4e-6 * scale + 1e-6, (err, scale)


# ------------------------------------------------------------------------------------------------
# GPU: the model against the fp32 oracle
# ------------------------------------------------------------------------------------------------
PRECISIONS = ('tf32x3', 'fp32', 'bf16')
SEEDS = {'connectstage': 31, 'multistage': 32}


@pytest.fixture(scope='module')
def models(dev):
    from upliftingtabletennis_b200.uplift import get_model
    out = {}
    for name, seed in SEEDS.items():
        sd = oup.random_state_dict(seed)
        m = get_model(name, 'large', 'dynamic', 'new').to(dev).eval()
        m.load_state_dict(sd)
        out[name] = (m, sd)
    return out


def _oracle(sd, name, ball, table, mask, times):
    r, p = oup.uplift_forward(sd, *(torch.from_numpy(a) for a in (ball, table, mask, times)), use_skipconnection=(name == 'connectstage'))
    return r.numpy(), p.numpy()


def _check_bar(prec, rot, pos, r_ref, p_ref, rows):
    """The precision's bar: fp32-level (and tf32x3 pos <= 3e-5) on every row, or bf16 relative L2 per trajectory on `rows`."""
    if prec != 'bf16':
        np.testing.assert_allclose(pos, p_ref, rtol=UPLIFT_RTOL, atol=UPLIFT_ATOL)
        np.testing.assert_allclose(rot, r_ref, rtol=UPLIFT_RTOL, atol=UPLIFT_ATOL)
        if prec == 'tf32x3':
            assert np.abs(pos - p_ref).max() < 3e-5
        return
    assert np.isfinite(pos).all() and np.isfinite(rot).all()
    for b in range(pos.shape[0]):
        if rows[b].any():
            ref = p_ref[b][rows[b]]
            rel = np.linalg.norm(pos[b][rows[b]] - ref) / (np.linalg.norm(ref) + 1e-6)
            assert rel < 5e-2, (b, rel)
    assert np.linalg.norm(rot - r_ref) / np.linalg.norm(r_ref) < 5e-2


@pytest.mark.gpu
@pytest.mark.parametrize('B,T', EDGE_SHAPES)
@pytest.mark.parametrize('name', list(SEEDS))
def test_model_edges_vs_oracle(dev, models, name, B, T):
    """Every precision against the oracle on the edge batch, and every trajectory run alone equals its row of the batch bit for bit.
    Measured on a B200 (1000 W): max |pos - oracle| 2.7e-5 for tf32x3 (bar 3e-5), 1.2e-5 for fp32 (bar 1e-4).  With an odd B T the
    tf32x3 path used to stop with a misaligned-address fault (its qkv buffer started 16 bytes off the 32 its stores need)."""
    m, sd = models[name]
    ball, table, mask, times = edge_trajectories(np.random.default_rng(1000 * B + T), B, T)
    r_ref, p_ref = _oracle(sd, name, ball, table, mask, times)
    args = [torch.from_numpy(a).to(dev) for a in (ball, table, mask, times)]
    for prec in PRECISIONS:
        m.compute_dtype = prec
        rot, pos = m(*args)
        rot, pos = rot.cpu(), pos.cpu()
        print('%s %s B %d T %d: max|pos - oracle| %.2e, max|rot - oracle| %.2e' % (name, prec, B, T, np.abs(pos.numpy() - p_ref).max(),
                                                                                    np.abs(rot.numpy() - r_ref).max()))
        _check_bar(prec, rot.numpy(), pos.numpy(), r_ref, p_ref, mask.astype(bool))
        for b in range(B):       # through the engine: a lone trajectory's mask may be all zeros or all ones
            r1, p1 = m.engine.forward(*(a[b:b + 1] for a in args), prec)
            assert torch.equal(r1[0].cpu(), rot[b]) and torch.equal(p1[0].cpu(), pos[b]), (prec, b)
    m.compute_dtype = 'tf32x3'


@pytest.mark.gpu
def test_tf32x3_chunk_boundary(dev, models):
    """B = 4097 on the tf32x3 path runs as a chunk of 4096 and one of 1 trajectory; both sides of the boundary match a lone run bit for
    bit and the oracle."""
    from upliftingtabletennis_b200.uplift import UpliftEngine
    m, sd = models['connectstage']
    B, T = UpliftEngine.TF32X3_CHUNK + 1, 5
    ball, table, mask, times = edge_trajectories(np.random.default_rng(4097), B, T)
    args = [torch.from_numpy(a).to(dev) for a in (ball, table, mask, times)]
    rot, pos = m.engine.forward(*args, 'tf32x3')
    sel = slice(B - 2, B)
    r_ref, p_ref = _oracle(sd, 'connectstage', ball[sel], table[sel], mask[sel], times[sel])
    _check_bar('tf32x3', rot[sel].cpu().numpy(), pos[sel].cpu().numpy(), r_ref, p_ref, None)
    for b in (B - 2, B - 1):
        r1, p1 = m.engine.forward(*(a[b:b + 1] for a in args), 'tf32x3')
        assert torch.equal(r1[0], rot[b]) and torch.equal(p1[0], pos[b]), b


@pytest.mark.gpu
@pytest.mark.parametrize('B,T', [(5, 13), (3, 53)])
@pytest.mark.parametrize('name', list(SEEDS))
def test_model_additive_mask(dev, models, name, B, T):
    """{-1e9, 0} masks follow the reference on ALL rows: a padded row attends uniformly over the valid frames (over all frames of a
    fully padded trajectory) instead of to nothing.  Valid rows and rot are those of the {0, 1} call, bit for bit.  Measured on a B200
    (1000 W): max |pos - oracle| 2.8e-5 for tf32x3, 1.1e-5 for fp32 on all rows."""
    m, sd = models[name]
    ball, table, mask, times = edge_trajectories(np.random.default_rng(7 * B + T), B, T)
    assert (mask.sum(1) == 0).any()
    madd = additive(mask)
    r_ref, p_ref = _oracle(sd, name, ball, table, madd, times)
    valid = mask.astype(bool)
    args = [torch.from_numpy(a).to(dev) for a in (ball, table, mask, times)]
    args_add = [args[0], args[1], torch.from_numpy(madd).to(dev), args[3]]
    for prec in PRECISIONS:
        m.compute_dtype = prec
        r01, p01 = (t.cpu().numpy() for t in m(*args))
        rot, pos = (t.cpu().numpy() for t in m(*args_add))
        print('%s %s additive mask B %d T %d: max|pos - oracle| %.2e' % (name, prec, B, T, np.abs(pos - p_ref).max()))
        _check_bar(prec, rot, pos, r_ref, p_ref, np.ones_like(valid))
        assert np.array_equal(rot, r01) and np.array_equal(pos[valid], p01[valid]), prec
    m.compute_dtype = 'tf32x3'


@pytest.mark.gpu
@pytest.mark.parametrize('T', [1, 64])
def test_seq_len_out_of_range(dev, models, T):
    """T outside [2, 63] is refused before any kernel is launched: the outputs keep their contents."""
    from upliftingtabletennis_b200 import _lib
    from upliftingtabletennis_b200._lib import lib, ptr, stream_ptr
    m, _ = models['connectstage']
    B = 2
    z = torch.zeros
    mask = z(B, T, device=dev)
    mask[0, 0] = 1.0
    with pytest.raises(_lib.TtkError, match='seq_len'):
        m(z(B, T, 2, device=dev), torch.ones(B, NTAB, 3, device=dev), mask, z(B, T, device=dev))
    assert m.engine.last_launches() == 0
    ws = torch.empty(lib.ttk_uplift_workspace_bytes(m.engine.h, B, T, _lib.TF32X3), dtype=torch.uint8, device=dev)
    rot = torch.full((B, 3), float('nan'), device=dev)
    pos = torch.full((B, T, 3), float('nan'), device=dev)
    args = [z(B, T, 2, device=dev), torch.ones(B, NTAB, 3, device=dev), mask, z(B, T, device=dev)]
    rc = lib.ttk_uplift_forward(m.engine.h, *(ptr(a) for a in args), B, T, 0, _lib.TF32X3, ptr(rot), ptr(pos), ptr(ws), ws.numel(),
                                stream_ptr())
    torch.cuda.synchronize()
    assert rc == -1 and b'seq_len' in lib.ttk_last_error() and lib.ttk_uplift_last_launches(m.engine.h) == 0
    assert rot.isnan().all() and pos.isnan().all()
