"""The tensor-core convolution engine (csrc/igemm.cu) on every path the model uses, against exact-operand fp64 references.

Reference operands are exactly what the hardware reads: activations (and dy) truncated to TF32, weights read back from
the packed buffer (pack rounds to TF32 with ties away from zero, checked separately against the fp64 effective kernel).
Every reference is an fp64 convolution on the GPU; dgrad and wgrad references are its autograd.  The bound is per
element:  |y - ref| <= TAU * absref + EPS * |ref|,  where absref is the same op on |x|, |w| (+ |bias|, |prior|, |addend|)
and bounds the fp32 accumulation error at every position, so an error confined to small-magnitude elements (a border,
a tail tile, a wrong halo) is seen.  EPS covers __expf / tanhf and the final fp32 roundings (a few ulps).

Each case pins the engine (VP_HALO=0/1, read on every call, which also bypasses the autotuner) and asserts which kernel
actually ran (vp_conv_last_launch): halo mode falls back to box mode silently on ineligible geometries, and split_k = 0
must really split (memset + atomics) on the rows marked auto-split.

Largest ratio max((|y - ref| - EPS |ref|) / absref) per family, measured over all cases on a B200 (1000 W power limit;
printed at the end of a -s run):  forward 1.5e-6, dgrad 2.0e-6, wgrad 2.3e-6, epilogues 1.7e-6, actgrad 7.5e-7, so
TAU = 2^-17 = 7.6e-6 is 3.4x the largest.  Exact mode (3xTF32, against the UNROUNDED operands): 1.4e-6, EXACT_BOUND 2^-19.
"""
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import savp_oracle as O

TAU = 2.0 ** -17
EPS = 2.0 ** -20
RATIOS = {}

gpu = pytest.mark.gpu
PLAIN, POOLED, UPSAMPLED = range(3)
NONE, RELU, LRELU, SIGMOID, TANH = range(5)
BOX, HALO, WG_TAPS, WG_ROWS = range(4)


@pytest.fixture(scope='module')
def L():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from video_prediction_b200 import lib
    lib.lib()
    yield lib
    if RATIOS:
        print('\nlargest error ratio per family: ' + ', '.join('%s %.3g' % kv for kv in sorted(RATIOS.items())))


# ------------------------------------------------------------------ operands
def rnd(*s, seed=0, scale=1.0, device='cuda'):
    g = torch.Generator(device='cpu').manual_seed(seed)
    return (torch.randn(*s, generator=g) * scale).to(device)


def trunc(t):
    """What the tensor core reads of an fp32 activation: the top 19 bits."""
    return (t.contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)


def rna(t):
    """TF32 rounding to nearest, ties away from zero (cvt.rna.tf32.f32, what pack applies to weights)."""
    return ((t.contiguous().view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)


def ceil4(v):
    return (v + 3) // 4 * 4


# ------------------------------------------------------------------ fp64 references
def conv_ref(x, P, ke, s, p, transposed, osp):
    """What the engine computes, in the precision of x / P.  x [N,D,H,W,K]; P [taps, Nout, K] (taps in (d,h,w) order of
    ke); result [N, *osp, Nout].  transposed = 0: out[o] = sum_r x[s*o + r - p] P[r];  1: out[s*o + r - p] += x[o] P[r]."""
    w = P.reshape(ke[0], ke[1], ke[2], P.shape[1], P.shape[2])
    xn = x.permute(0, 4, 1, 2, 3)
    if not transposed:
        after = [(o - 1) * st + k - pp - d for o, st, k, pp, d in zip(osp, s, ke, p, x.shape[1:4])]
        xn = F.pad(xn, (p[2], after[2], p[1], after[1], p[0], after[0]))
        y = F.conv3d(xn, w.permute(3, 4, 0, 1, 2), stride=s)
    else:
        y = F.conv_transpose3d(xn, w.permute(4, 3, 0, 1, 2), stride=s)
        full = y.shape[2:]
        y = F.pad(y, (-p[2], osp[2] + p[2] - full[2], -p[1], osp[1] + p[1] - full[1], -p[0], osp[0] + p[0] - full[0]))
    return y.permute(0, 2, 3, 4, 1)


def _bil4(i):
    return 0.25 if i in (0, 3) else (0.75 if i in (1, 2) else 0.0)


def keff64(w, kind, k, cmap, ci_int):
    """The effective tap matrices pack builds, in fp64 and unrounded: [taps, co, ci_int] (cmap -1 columns zero)."""
    kh, kw = k[1], k[2]
    w = w.double().reshape(k[0] * kh * kw, w.shape[-2], w.shape[-1])            # [tap][ci_ref][co]
    if kind == PLAIN:
        taps = w
    elif kind == POOLED:
        w4 = w.reshape(kh, kw, w.shape[1], w.shape[2])
        taps = torch.zeros(kh + 1, kw + 1, w.shape[1], w.shape[2], dtype=w.dtype, device=w.device)
        for a in (0, 1):
            for b in (0, 1):
                taps[a:a + kh, b:b + kw] += 0.25 * w4
        taps = taps.reshape(-1, w.shape[1], w.shape[2])
    else:
        w4 = w.reshape(kh, kw, w.shape[1], w.shape[2])
        taps = torch.zeros(kh + 3, kw + 3, w.shape[1], w.shape[2], dtype=w.dtype, device=w.device)
        for p_ in range(kh + 3):
            for q in range(kw + 3):
                for i in range(kh):
                    for j in range(kw):
                        bw = _bil4(p_ + i - (kh - 1)) * _bil4(q + j - (kw - 1))
                        if bw:
                            taps[p_, q] += bw * w4[i, j]
        taps = taps.reshape(-1, w.shape[1], w.shape[2])
    out = torch.zeros(taps.shape[0], taps.shape[2], ci_int, dtype=w.dtype, device=w.device)
    for j, cr in enumerate(cmap):
        if cr >= 0:
            out[:, :, j] = taps[:, cr, :]
    return out


def act64(v, act, alpha):
    if act == RELU:
        return torch.relu(v)
    if act == LRELU:
        return O.lrelu(v, alpha)
    if act == SIGMOID:
        return torch.sigmoid(v)
    if act == TANH:
        return torch.tanh(v)
    return v


def check(family, y, ref, absref, what, tau=None):
    """|y - ref| <= tau * absref + EPS * |ref| element by element; records the largest ratio of the family."""
    tau = TAU if tau is None else tau
    assert bool(torch.isfinite(y).all()), '%s: non-finite output (%d elements)' % (what, int((~torch.isfinite(y)).sum()))
    slack = ((y.double() - ref).abs() - EPS * ref.abs()).clamp(min=0)
    ratio = float((slack / absref.clamp(min=1e-300)).max()) if slack.numel() else 0.0
    RATIOS[family] = max(RATIOS.get(family, 0.0), ratio)
    bad = slack > tau * absref
    if bool(bad.any()):
        i = int(bad.flatten().nonzero()[0])
        raise AssertionError('%s: %d elements out of bound (ratio %.3g > tau %.3g); first at flat index %d: got %r, ref %r, absref %r'
                             % (what, int(bad.sum()), ratio, tau, i, float(y.flatten()[i]), float(ref.flatten()[i]),
                                float(absref.flatten()[i])))


# ------------------------------------------------------------------ geometries
class Geo(object):
    """One convolution: x [n, d, h, w, cs] (cs = internal channels = ci_ref + padding, or a concat layout `segs`),
    reference kernel k (kd, kh, kw), engine pad p, co outputs.  halo / halo_d: halo mode serves forward / dgrad;
    split / split_d: split_k = 0 splits the forward / dgrad in (box, halo) mode (measured on a B200: the split choice
    depends on the SM count); wg: weight-gradient kernel, wg_split: split_k = 0 splits it."""

    def __init__(self, name, kind, k, s, p, tr, xs, ci, co, cs=None, segs=None, halo=True, halo_d=True, split=(False, False),
                 split_d=(False, False), wg=WG_TAPS, wg_split=True):
        self.name, self.kind, self.k, self.s, self.p, self.tr, self.xs, self.ci, self.co = name, kind, k, s, p, tr, xs, ci, co
        self.segs = segs
        if segs:
            from video_prediction_b200.models.savp_model import ConcatSpec
            spec = ConcatSpec(segs)
            self.cs, self.cmap = spec.cstride, spec.cmap
            assert spec.ref_channels == ci
        else:
            self.cs = cs or ceil4(ci)
            self.cmap = list(range(ci)) + [-1] * (self.cs - ci)
        self.halo, self.halo_d, self.split, self.split_d, self.wg, self.wg_split = halo, halo_d, split, split_d, wg, wg_split
        self.ke = k if kind == PLAIN else ((1, k[1] + 1, k[2] + 1) if kind == POOLED else (1, k[1] + 3, k[2] + 3))
        sp = xs[1:]
        if tr:
            self.osp = tuple(d * st for d, st in zip(sp, s))
        else:
            self.osp = tuple((d + 2 * pp - kk) // st + 1 for d, pp, kk, st in zip(sp, p, self.ke, s))

    def __repr__(self):
        return self.name


def _segs53():
    return [('a', 32), ('b', 3), ('c', 3), ('d', 3), ('e', 3), ('f', 9)]     # 53 reference channels in a 60-wide buffer


S1, S2, S122, S222 = (1, 1, 1), (1, 2, 2), (1, 2, 2), (2, 2, 2)
GEOMS = [
    # ConvLSTM gate convolutions h0..h2 (5x5, SAME)
    Geo('gate_h0', PLAIN, (1, 5, 5), S1, (0, 2, 2), False, (3, 1, 32, 32), 72, 128, wg=WG_ROWS, split=(True, True), split_d=(True, True)),
    Geo('gate_h1', PLAIN, (1, 5, 5), S1, (0, 2, 2), False, (3, 1, 16, 16), 136, 256, wg=WG_ROWS, split=(True, True), split_d=(True, True)),
    Geo('gate_h2', PLAIN, (1, 5, 5), S1, (0, 2, 2), False, (5, 1, 8, 8), 264, 512, wg=WG_ROWS, split=(True, True), split_d=(True, True), wg_split=False),
    # conv_pool2d h0..h2 (h0: 14 channels in a 16-wide buffer)
    Geo('pool_h0', POOLED, (1, 5, 5), S2, (0, 2, 2), False, (2, 1, 64, 64), 14, 32, cs=16, split=(True, True)),
    Geo('pool_h1', POOLED, (1, 3, 3), S2, (0, 1, 1), False, (2, 1, 32, 32), 40, 64, split=(True, True), split_d=(False, True)),
    Geo('pool_h2', POOLED, (1, 3, 3), S2, (0, 1, 1), False, (3, 1, 16, 16), 72, 128, split=(True, True), split_d=(False, True), wg_split=False),
    # upsample_conv2d h3, h5 (transposed; dy is the shifted operand of the weight gradient)
    Geo('up_h3', UPSAMPLED, (1, 3, 3), S2, (0, 2, 2), True, (3, 1, 8, 8), 136, 64, split=(True, True), split_d=(True, True), wg_split=False),
    Geo('up_h5', UPSAMPLED, (1, 3, 3), S2, (0, 2, 2), True, (2, 1, 32, 32), 72, 32, split=(True, True), split_d=(True, True)),
    # 3x3 heads: masks 53 -> 8 from a 60-channel concat buffer; the scratch image (sigmoid, written into a slice)
    Geo('masks', PLAIN, (1, 3, 3), S1, (0, 1, 1), False, (2, 1, 64, 64), 53, 8, segs=_segs53(), split=(False, True)),
    Geo('scratch', PLAIN, (1, 3, 3), S1, (0, 1, 1), False, (2, 1, 64, 64), 32, 3),
    # posterior 4x4 s2
    Geo('posterior', PLAIN, (1, 4, 4), S2, (0, 1, 1), False, (5, 1, 32, 32), 64, 128, split=(True, True), split_d=(False, True)),
    # video discriminator (3-D; the first layer runs on the CUDA cores / its own kernels)
    Geo('d_conv0_1', PLAIN, (4, 4, 4), S122, (1, 1, 1), False, (2, 10, 64, 64), 32, 64, split=(False, True)),
    Geo('d_conv1_0', PLAIN, (3, 3, 3), S1, (1, 1, 1), False, (2, 9, 32, 32), 64, 64, split=(False, True), split_d=(False, True)),
    Geo('d_conv1_1', PLAIN, (4, 4, 4), S122, (1, 1, 1), False, (2, 9, 32, 32), 64, 128, split=(True, True), split_d=(False, True)),
    Geo('d_conv2_0', PLAIN, (3, 3, 3), S1, (1, 1, 1), False, (2, 8, 16, 16), 128, 128, split=(True, True), split_d=(True, True)),
    Geo('d_conv2_1', PLAIN, (4, 4, 4), S222, (1, 1, 1), False, (2, 8, 16, 16), 128, 256, split=(True, True), split_d=(True, True)),
    Geo('d_conv3_0', PLAIN, (3, 3, 3), S1, (1, 1, 1), False, (3, 4, 8, 8), 256, 256, split=(True, True), split_d=(True, True)),
    # image discriminator (2-D analogue), where it differs
    Geo('i_conv0_1', PLAIN, (1, 4, 4), S2, (0, 1, 1), False, (3, 1, 64, 64), 32, 64, split=(False, True), split_d=(False, True)),
    Geo('i_conv2_1', PLAIN, (1, 4, 4), S2, (0, 1, 1), False, (3, 1, 16, 16), 128, 256, split=(True, True), split_d=(True, True), wg_split=False),
    Geo('i_conv3_0', PLAIN, (1, 3, 3), S1, (0, 1, 1), False, (3, 1, 8, 8), 256, 256, split=(True, True), split_d=(True, True), wg_split=False),
    # edges: W = 24 / H = 12 (stacked halo sub-tiles, partial tile in h); W = 20 (halo ineligible); 8x8 planes, odd n
    Geo('e_w24_h12', PLAIN, (1, 3, 3), S1, (0, 1, 1), False, (3, 1, 12, 24), 40, 64, split=(False, True), split_d=(False, True)),
    Geo('e_w20', PLAIN, (1, 3, 3), S1, (0, 1, 1), False, (2, 1, 12, 20), 40, 64, halo=False, halo_d=False),
    Geo('e_8x8_n5', PLAIN, (1, 3, 3), S1, (0, 1, 1), False, (5, 1, 8, 8), 64, 64, split=(False, True), split_d=(False, True), wg_split=False),
    # k_tail 1, 2, 3 (the last 32-channel chunk holds 4, 12, 20 channels)
    Geo('e_ktail1', PLAIN, (1, 3, 3), S1, (0, 1, 1), False, (2, 1, 16, 16), 36, 32, split=(False, True)),
    Geo('e_ktail2', PLAIN, (1, 3, 3), S1, (0, 1, 1), False, (2, 1, 16, 16), 44, 48, split=(False, True), split_d=(False, True)),
    Geo('e_ktail3', PLAIN, (1, 3, 3), S1, (0, 1, 1), False, (2, 1, 16, 16), 52, 32, split=(False, True)),
    # Cout 7 (n_pad 16, scalar stores); Cout 264 (n_pad 288 = two 144-wide tiles)
    Geo('e_cout7', PLAIN, (1, 3, 3), S1, (0, 1, 1), False, (2, 1, 16, 16), 32, 7),
    Geo('e_cout264', PLAIN, (1, 3, 3), S1, (0, 1, 1), False, (2, 1, 8, 8), 64, 264, split=(False, True), split_d=(True, True), wg_split=False),
]
BY_NAME = {g.name: g for g in GEOMS}


class Setup(object):
    """Operands of one geometry: x in a buffer 4 channels wider than the view (padding channels and cmap -1 slots hold
    7.0), weights, packed weights (both layouts) read back as fp64 [taps, rows, cols]."""

    def __init__(self, L, g, seed=0):
        self.g = g
        n = g.xs[0]
        taps_ref = g.k[0] * g.k[1] * g.k[2]
        self.w = rnd(*(g.k if g.k[0] > 1 else g.k[1:]), g.ci, g.co, seed=seed + 1, scale=1.0 / math.sqrt(taps_ref * g.ci))
        self.cmap_t = torch.tensor(g.cmap, dtype=torch.int32, device='cuda')
        self.xbuf = rnd(*g.xs, g.cs + 4, seed=seed)
        pad = torch.tensor([c < 0 for c in g.cmap] + [True] * 4, device='cuda')
        self.xbuf[..., pad] = 7.0
        self.real = torch.tensor([c >= 0 for c in g.cmap], device='cuda')       # real channels of the view
        self.bias = rnd(g.co, seed=seed + 2, scale=0.5)
        self.wp, self.n_pad, self.kc = L.pack_weights(self.w, g.k, g.ci, g.co, g.kind, L.WLAYOUT_FWD, ci_int=g.cs, cmap=self.cmap_t)
        self.wpd, self.n_pad_d, self.kc_d = L.pack_weights(self.w, g.k, g.ci, g.co, g.kind, L.WLAYOUT_DGRAD, ci_int=g.cs,
                                                           cmap=self.cmap_t)
        taps = L.eff_taps(g.k, g.kind)
        self.P = self.wp.view(taps, self.n_pad, self.kc * 32)[:, :g.co, :g.cs].double()
        self.Pd = self.wpd.view(taps, self.n_pad_d, self.kc_d * 32)[:, :g.cs, :g.co].double()
        self.geom = L.geom(g.ke, g.s, g.p, g.tr)
        self.geom_d = L.geom(g.ke, g.s, g.p, not g.tr)
        self.oshape = (n,) + g.osp
        cos = ceil4(g.co) + 4                                           # dy lives in a wider buffer too
        self.dybuf = rnd(*self.oshape, cos, seed=seed + 3)
        self.dybuf[..., g.co:] = 7.0

    def x_ref(self):
        """fp64 view as the semantics define it: truncated, the padding slots zero."""
        return trunc(self.xbuf[..., :self.g.cs]).double() * self.real.double()

    def dy_ref(self):
        return trunc(self.dybuf[..., :self.g.co]).double()

    def fwd64(self, x, P):
        g = self.g
        return conv_ref(x, P, g.ke, g.s, g.p, g.tr, g.osp)


def _engine(monkeypatch, halo):
    monkeypatch.setenv('VP_HALO', '1' if halo else '0')


def _expect(L, halo_requested, halo_eligible, auto_rows, split_k, what):
    kernel, splits = L.last_launch()
    want = HALO if (halo_requested and halo_eligible) else BOX
    assert kernel == want, '%s: kernel %d ran, expected %d' % (what, kernel, want)
    if split_k == 0 and auto_rows[1 if want == HALO else 0]:
        assert splits > 1, '%s: split_k = 0 did not split' % what
    if split_k == 1:
        assert splits == 1, what
    return kernel, splits


# ------------------------------------------------------------------ semantics of the fp64 reference, pinned in fp64 (CPU)
@pytest.mark.parametrize('name', ['pool_h0', 'pool_h1', 'up_h3', 'up_h5'])
def test_reference_conv_matches_the_oracle_ops_in_fp64(name):
    """conv_ref with the fp64 effective kernel and the engine's (ke, s, p) equals O.conv_pool2d / O.upsample_conv2d."""
    g = BY_NAME[name]
    n = 2
    w = rnd(g.k[1], g.k[2], g.ci, g.co, seed=1, device='cpu').double()
    xr = rnd(n, g.xs[2], g.xs[3], g.ci, seed=2, device='cpu').double()
    xi = torch.zeros(n, 1, g.xs[2], g.xs[3], g.cs, dtype=torch.float64)
    for j, cr in enumerate(g.cmap):
        if cr >= 0:
            xi[..., j] = xr[:, None, ..., cr]
    y = conv_ref(xi, keff64(w, g.kind, g.k, g.cmap, g.cs), g.ke, g.s, g.p, g.tr, g.osp)[:, 0]
    zero = torch.zeros(g.co, dtype=torch.float64)
    want = O.conv_pool2d(xr, w, zero) if g.kind == POOLED else O.upsample_conv2d(xr, w, zero)
    assert y.shape == want.shape
    assert float((y - want).abs().max()) <= 1e-12 * float(want.abs().max())


def test_reference_conv_matches_conv2d_same_in_fp64():
    g = BY_NAME['gate_h1']
    w = rnd(5, 5, 8, 16, seed=1, device='cpu').double()
    x = rnd(2, 1, 16, 16, 8, seed=2, device='cpu').double()
    y = conv_ref(x, w.reshape(25, 8, 16).transpose(1, 2), g.ke, g.s, g.p, False, (1, 16, 16))
    want = O.conv2d_tf(x[:, 0], w, padding='SAME')
    assert float((y[:, 0] - want).abs().max()) <= 1e-12 * float(want.abs().max())


# ------------------------------------------------------------------ pack
@gpu
@pytest.mark.parametrize('g', GEOMS, ids=repr)
def test_pack_against_fp64_effective_kernel(L, g):
    """Packed weights = rna(keff) within 2^-11 |keff| (+ the fp32 sums of the pooled / upsampled taps); the DGRAD layout is
    the FWD layout transposed, bit for bit; the padding of both is zero."""
    S = Setup(L, g)
    kref = keff64(S.w, g.kind, g.k, g.cmap, g.cs)
    kabs = keff64(S.w.abs(), g.kind, g.k, g.cmap, g.cs)
    err = (S.P - kref).abs()
    assert bool((err <= 2.0 ** -11 * kref.abs() + 2.0 ** -21 * kabs).all()), 'pack: max err %g' % float(err.max())
    assert torch.equal(S.P, rna(S.P.float()).double())                      # TF32 values
    assert torch.equal(S.Pd, S.P.transpose(1, 2))
    taps = L.eff_taps(g.k, g.kind)
    full = S.wp.view(taps, S.n_pad, S.kc * 32)
    assert float(full[:, g.co:].abs().sum()) == 0 and float(full[:, :, g.cs:].abs().sum()) == 0


# ------------------------------------------------------------------ forward
def _run_fwd(L, S, out, view, act=NONE, alpha=0.2, split_k=1, accumulate=0, bias=True):
    L.conv_igemm(L.tensor_view(S.xbuf, S.g.cs), S.geom, S.wp, S.n_pad, S.kc, view, S.bias if bias else None, act, alpha,
                 split_k, accumulate)
    torch.cuda.synchronize()


def _out_buffer(S, slice_off=None):
    """Dense [n, osp, co] when co % 4 == 0, else co in a ceil4(co)-wide buffer; slice_off puts it into a wider buffer."""
    g = S.g
    width = ceil4(g.co) if slice_off is None else slice_off + ceil4(g.co) + 4
    return torch.full(S.oshape + (width,), float('nan'), device='cuda')


def _sentinel_check(buf, before, off, c):
    mask = torch.ones(buf.shape[-1], dtype=torch.bool, device='cuda')
    mask[off:off + c] = False
    assert torch.equal(buf[..., mask].view(torch.int32), before[..., mask].view(torch.int32)), 'channels outside the view changed'


@gpu
@pytest.mark.parametrize('split_k', [1, 0])
@pytest.mark.parametrize('halo', [False, True], ids=['box', 'halo'])
@pytest.mark.parametrize('g', GEOMS, ids=repr)
def test_forward(L, monkeypatch, g, halo, split_k):
    _engine(monkeypatch, halo)
    S = Setup(L, g)
    out = _out_buffer(S)
    if g.co % 4:
        out[..., g.co:] = -123.5
    before = out.clone()
    _run_fwd(L, S, out, L.tensor_view(out, g.co), split_k=split_k)
    _expect(L, halo, g.halo, g.split, split_k, '%s fwd' % g.name)
    _sentinel_check(out, before, 0, g.co)
    x = S.x_ref()
    ref = S.fwd64(x, S.P) + S.bias.double()
    absref = S.fwd64(x.abs(), S.P.abs()) + S.bias.double().abs()
    check('forward', out[..., :g.co], ref, absref, '%s forward' % g.name)


@gpu
@pytest.mark.parametrize('act', [NONE, RELU, LRELU, SIGMOID, TANH], ids=['none', 'relu', 'lrelu', 'sigmoid', 'tanh'])
@pytest.mark.parametrize('halo', [False, True], ids=['box', 'halo'])
@pytest.mark.parametrize('name', ['gate_h0', 'pool_h1', 'masks', 'd_conv1_0', 'e_cout7', 'e_w24_h12'])
def test_forward_epilogues(L, monkeypatch, name, halo, act):
    g = BY_NAME[name]
    _engine(monkeypatch, halo)
    S = Setup(L, g, seed=10)
    out = _out_buffer(S)
    _run_fwd(L, S, out, L.tensor_view(out, g.co), act=act, split_k=0)
    _expect(L, halo, g.halo, g.split if act == NONE else (False, False), 0, '%s act %d' % (name, act))
    x = S.x_ref()
    pre = S.fwd64(x, S.P) + S.bias.double()
    absref = S.fwd64(x.abs(), S.P.abs()) + S.bias.double().abs()
    check('epilogues', out[..., :g.co], act64(pre, act, 0.2), absref, '%s act %d' % (name, act))


@gpu
@pytest.mark.parametrize('halo', [False, True], ids=['box', 'halo'])
def test_forward_sigmoid_into_a_slice_of_a_wider_buffer(L, monkeypatch, halo):
    """The scratch-image head: 3 channels, sigmoid, written at channel offset 8 of a 20-channel buffer."""
    g = BY_NAME['scratch']
    _engine(monkeypatch, halo)
    S = Setup(L, g, seed=20)
    out = _out_buffer(S, slice_off=8)
    out[..., :8] = -123.5
    out[..., 8 + g.co:] = 321.25
    before = out.clone()
    _run_fwd(L, S, out, L.tensor_view(out, g.co, 8), act=SIGMOID, split_k=0)
    _expect(L, halo, g.halo, (False, False), 0, 'scratch head')
    _sentinel_check(out, before, 8, g.co)
    x = S.x_ref()
    pre = S.fwd64(x, S.P) + S.bias.double()
    absref = S.fwd64(x.abs(), S.P.abs()) + S.bias.double().abs()
    check('epilogues', out[..., 8:8 + g.co], torch.sigmoid(pre), absref, 'scratch head')


@gpu
@pytest.mark.parametrize('mode', ['acc1', 'acc2_none', 'acc2_lrelu', 'acc2_sigmoid', 'acc2_tanh', 'acc1_split3', 'acc2_split3',
                                  'split3'])
@pytest.mark.parametrize('halo', [False, True], ids=['box', 'halo'])
@pytest.mark.parametrize('name', ['gate_h1', 'pool_h0', 'up_h5', 'd_conv2_1', 'e_cout264'])
def test_forward_accumulate(L, monkeypatch, name, halo, mode):
    """accumulate = 1: out += conv (no bias, act NONE); accumulate = 2: out = act(out + conv + bias), the prior added
    BEFORE the activation.  An explicit split_k > 1 adds atomically into the output as the caller left it (cleared for a
    plain call)."""
    g = BY_NAME[name]
    _engine(monkeypatch, halo)
    S = Setup(L, g, seed=30)
    acc = 0 if mode == 'split3' else (1 if mode.startswith('acc1') else 2)
    act = {'acc2_lrelu': LRELU, 'acc2_sigmoid': SIGMOID, 'acc2_tanh': TANH}.get(mode, NONE)
    split_k = 3 if mode.endswith('split3') else 1
    prior = torch.zeros(S.oshape + (g.co,), device='cuda') if acc == 0 else rnd(*S.oshape, g.co, seed=31)
    out = prior.clone()
    _run_fwd(L, S, out, L.tensor_view(out, g.co), act=act, split_k=split_k, accumulate=acc, bias=acc != 1)
    kernel, splits = _expect(L, halo, g.halo, (False, False), split_k, '%s %s' % (name, mode))
    assert splits > 1 if split_k == 3 else splits == 1
    x = S.x_ref()
    pre = S.fwd64(x, S.P) + prior.double() + (S.bias.double() if acc != 1 else 0)
    absref = S.fwd64(x.abs(), S.P.abs()) + prior.double().abs() + (S.bias.double().abs() if acc != 1 else 0)
    check('epilogues', out, act64(pre, act, 0.2), absref, '%s %s' % (name, mode))


# ------------------------------------------------------------------ dgrad
@gpu
@pytest.mark.parametrize('split_k', [1, 0])
@pytest.mark.parametrize('halo', [False, True], ids=['box', 'halo'])
@pytest.mark.parametrize('g', GEOMS, ids=repr)
def test_dgrad(L, monkeypatch, g, halo, split_k):
    """dx = conv^T(dy): the same engine with the transposed flag flipped (strided 3-D: 4 or 8 output phases), against
    the autograd of the forward reference."""
    _engine(monkeypatch, halo)
    S = Setup(L, g, seed=40)
    dx = torch.full(g.xs + (g.cs,), float('nan'), device='cuda')
    L.conv_igemm(L.tensor_view(S.dybuf, g.co), S.geom_d, S.wpd, S.n_pad_d, S.kc_d, L.tensor_view(dx, g.cs), None, NONE, 0.0,
                 split_k, 0)
    torch.cuda.synchronize()
    _expect(L, halo, g.halo_d, g.split_d, split_k, '%s dgrad' % g.name)
    dy = S.dy_ref()
    x = torch.zeros(g.xs + (g.cs,), dtype=torch.float64, device='cuda', requires_grad=True)
    (ref,) = torch.autograd.grad(S.fwd64(x, S.P), x, dy)
    (absref,) = torch.autograd.grad(S.fwd64(x, S.P.abs()), x, dy.abs())
    check('dgrad', dx, ref, absref, '%s dgrad' % g.name)


@gpu
@pytest.mark.parametrize('halo', [False, True], ids=['box', 'halo'])
@pytest.mark.parametrize('name', ['gate_h1', 'pool_h1', 'up_h5', 'masks', 'd_conv0_1', 'd_conv2_1', 'e_cout7'])
def test_dgrad_accumulate(L, monkeypatch, name, halo):
    """accumulate = 1 (the generator's dgrad into a gradient that already holds another consumer's part)."""
    g = BY_NAME[name]
    _engine(monkeypatch, halo)
    S = Setup(L, g, seed=50)
    prior = rnd(*g.xs, g.cs, seed=51)
    dx = prior.clone()
    L.conv_igemm(L.tensor_view(S.dybuf, g.co), S.geom_d, S.wpd, S.n_pad_d, S.kc_d, L.tensor_view(dx, g.cs), None, NONE, 0.0, 1, 1)
    torch.cuda.synchronize()
    _expect(L, halo, g.halo_d, g.split_d, 1, '%s dgrad accumulate' % name)
    dy = S.dy_ref()
    x = torch.zeros(g.xs + (g.cs,), dtype=torch.float64, device='cuda', requires_grad=True)
    (ref,) = torch.autograd.grad(S.fwd64(x, S.P), x, dy)
    (absref,) = torch.autograd.grad(S.fwd64(x, S.P.abs()), x, dy.abs())
    check('dgrad', dx, ref + prior.double(), absref + prior.double().abs(), '%s dgrad accumulate' % name)


def _act_deriv64(y, act, alpha):
    y = y.double()
    if act == LRELU:
        return torch.where(y > 0, torch.ones_like(y), torch.full_like(y, alpha))
    if act == RELU:
        return (y > 0).double()
    if act == SIGMOID:
        return y * (1 - y)
    return 1 - y * y


@gpu
@pytest.mark.parametrize('acc', [0, 2])
@pytest.mark.parametrize('addend', [False, True], ids=['plain', 'addend'])
@pytest.mark.parametrize('act', [LRELU, RELU, SIGMOID], ids=['lrelu', 'relu', 'sigmoid'])
@pytest.mark.parametrize('halo', [False, True], ids=['box', 'halo'])
@pytest.mark.parametrize('name', ['d_conv1_0', 'd_conv2_1', 'i_conv0_1'])
def test_conv_igemm_actgrad(L, monkeypatch, name, halo, act, addend, acc):
    """out = (conv^T(dy) + [out] + addend) * act'(y): the discriminator towers' dgrad fused with the previous layer's
    activation backward, act' evaluated from the activation OUTPUT y."""
    g = BY_NAME[name]
    _engine(monkeypatch, halo)
    S = Setup(L, g, seed=60)
    shape = g.xs + (g.cs,)
    y = rnd(*shape, seed=61)
    y = torch.sigmoid(y) if act == SIGMOID else torch.where(y > 0, y, 0.2 * y if act == LRELU else torch.zeros_like(y))
    add = rnd(*shape, seed=62) if addend else None
    prior = rnd(*shape, seed=63)
    dx = prior.clone() if acc == 2 else torch.full(shape, float('nan'), device='cuda')
    L.conv_igemm_actgrad(L.tensor_view(S.dybuf, g.co), S.geom_d, S.wpd, S.n_pad_d, S.kc_d, L.tensor_view(dx, g.cs), y.data_ptr(),
                         add.data_ptr() if addend else 0, act, 0.2, accumulate=acc)
    torch.cuda.synchronize()
    _expect(L, halo, g.halo_d, (False, False), 1, '%s actgrad' % name)
    dy = S.dy_ref()
    x = torch.zeros(shape, dtype=torch.float64, device='cuda', requires_grad=True)
    (conv,) = torch.autograd.grad(S.fwd64(x, S.P), x, dy)
    (absref,) = torch.autograd.grad(S.fwd64(x, S.P.abs()), x, dy.abs())
    pre, apre = conv, absref
    if acc == 2:
        pre, apre = pre + prior.double(), apre + prior.double().abs()
    if addend:
        pre, apre = pre + add.double(), apre + add.double().abs()
    d = _act_deriv64(y, act, 0.2)
    check('actgrad', dx, pre * d, apre * d.abs(), '%s actgrad act %d addend %d acc %d' % (name, act, addend, acc))


# ------------------------------------------------------------------ wgrad
def _wgrad_case(L, g, split_k, seed=70):
    S = Setup(L, g, seed=seed)
    taps = L.eff_taps(g.k, g.kind)
    dwp = torch.full((taps * S.n_pad * S.kc * 32,), 0.25, device='cuda')          # wgrad adds into it
    L.conv_wgrad(L.tensor_view(S.xbuf, g.cs), L.tensor_view(S.dybuf, g.co), S.geom, dwp, S.n_pad, S.kc, split_k)
    torch.cuda.synchronize()
    kernel, splits = L.last_launch()
    xw = trunc(S.xbuf[..., :g.cs]).double()                 # the engine's operand: every channel of the view, padding slots too
    dy = S.dy_ref()
    Pv = torch.zeros(taps, g.co, g.cs, dtype=torch.float64, device='cuda', requires_grad=True)
    (ref,) = torch.autograd.grad(S.fwd64(xw, Pv), Pv, dy)
    (absref,) = torch.autograd.grad(S.fwd64(xw.abs(), Pv), Pv, dy.abs())
    full = dwp.view(taps, S.n_pad, S.kc * 32)
    check('wgrad', full[:, :g.co, :g.cs], ref + 0.25, absref, '%s wgrad' % g.name)
    rest = torch.ones_like(full, dtype=torch.bool)
    rest[:, :g.co, :g.cs] = False
    assert bool((full[rest] == 0.25).all()), '%s wgrad: padding rows / columns of dwpacked changed' % g.name
    return kernel, splits


@gpu
@pytest.mark.parametrize('split_k', [1, 0])
@pytest.mark.parametrize('g', GEOMS, ids=repr)
def test_wgrad(L, monkeypatch, g, split_k):
    """Row mode for the 5x5 gates, tap groups (merged wide-N MMAs) elsewhere; split_k = 0 splits the pixel loop."""
    monkeypatch.delenv('VP_WGRAD_ROW', raising=False)
    monkeypatch.delenv('VP_WGRAD_MERGE', raising=False)
    kernel, splits = _wgrad_case(L, g, split_k)
    assert kernel == g.wg, '%s wgrad: kernel %d ran, expected %d' % (g.name, kernel, g.wg)
    assert splits == 1 if split_k == 1 else (splits > 1) == g.wg_split, '%s wgrad: %d splits' % (g.name, splits)


@gpu
@pytest.mark.parametrize('knob', ['VP_WGRAD_MERGE', 'VP_WGRAD_ROW'])
@pytest.mark.parametrize('name', ['gate_h0', 'gate_h2', 'pool_h0', 'up_h3', 'masks', 'd_conv0_1', 'd_conv1_0', 'd_conv2_1',
                                  'd_conv3_0', 'e_cout7', 'e_cout264'])
def test_wgrad_knobs(L, monkeypatch, name, knob):
    """VP_WGRAD_MERGE=0 (one MMA per tap instead of merged wide-N MMAs) and VP_WGRAD_ROW=0 (tap groups for the 5x5 gates)."""
    g = BY_NAME[name]
    monkeypatch.delenv('VP_WGRAD_ROW', raising=False)
    monkeypatch.delenv('VP_WGRAD_MERGE', raising=False)
    monkeypatch.setenv(knob, '0')
    kernel, _ = _wgrad_case(L, g, 0, seed=80)
    assert kernel == (WG_TAPS if knob == 'VP_WGRAD_ROW' else g.wg)


# ------------------------------------------------------------------ fp32-exact mode at kernel level
@gpu
def test_tf32_residual_is_x_minus_its_truncation(L):
    x = rnd(3, 1000, 4, seed=90) * torch.logspace(-20, 20, 4, device='cuda')
    x[0, :4] = torch.tensor([0.0, -0.0, 1.0, -1.5 * 2.0 ** -126], device='cuda')     # (denormals are flushed: fast math)
    lo = L.tf32_residual(x)
    torch.cuda.synchronize()
    assert torch.equal(lo.view(torch.int32), (x - trunc(x)).view(torch.int32))


@gpu
@pytest.mark.parametrize('layout', ['fwd', 'dgrad'])
def test_residual_pack_is_rna_of_what_rounding_dropped(L, layout):
    g = BY_NAME['masks']
    S = Setup(L, g, seed=91)
    lay = (L.WLAYOUT_FWD if layout == 'fwd' else L.WLAYOUT_DGRAD)
    hi, n_pad, kc = L.pack_weights(S.w, g.k, g.ci, g.co, g.kind, lay, ci_int=g.cs, cmap=S.cmap_t)
    lo, _, _ = L.pack_weights(S.w, g.k, g.ci, g.co, g.kind, lay | L.WLAYOUT_RESIDUAL, ci_int=g.cs, cmap=S.cmap_t)
    torch.cuda.synchronize()
    k = keff64(S.w, PLAIN, g.k, g.cmap, g.cs).float()                      # exact: PLAIN copies the fp32 weights
    if layout == 'dgrad':
        k = k.transpose(1, 2)
    full = torch.zeros(9, n_pad, kc * 32, device='cuda')
    full[:, :k.shape[1], :k.shape[2]] = k
    assert torch.equal(hi.view(9, n_pad, kc * 32).view(torch.int32), rna(full).view(torch.int32))
    assert torch.equal(lo.view(9, n_pad, kc * 32).view(torch.int32), rna(full - rna(full)).view(torch.int32))


EXACT_BOUND = 2.0 ** -19      # per element, relative to absref (fp32 accumulation of the three passes): 1.4e-6 measured


def _exact_operands(L, g, seed):
    S = Setup(L, g, seed=seed)
    S.wp_lo, _, _ = L.pack_weights(S.w, g.k, g.ci, g.co, g.kind, L.WLAYOUT_FWD | L.WLAYOUT_RESIDUAL, ci_int=g.cs, cmap=S.cmap_t)
    S.wpd_lo, _, _ = L.pack_weights(S.w, g.k, g.ci, g.co, g.kind, L.WLAYOUT_DGRAD | L.WLAYOUT_RESIDUAL, ci_int=g.cs,
                                    cmap=S.cmap_t)
    S.xbuf = S.xbuf[..., :g.cs].contiguous()                # conv3x takes the residual of the whole buffer
    S.xbuf[..., ~S.real] = 0.0
    S.dybuf = S.dybuf[..., :g.co].contiguous() if g.co % 4 == 0 else S.dybuf
    S.dybuf[..., g.co:] = 0.0
    S.K = keff64(S.w, g.kind, g.k, g.cmap, g.cs)             # unrounded fp64 effective kernel
    return S


def _max_ratio(y, ref, absref):
    return float(((y.double() - ref).abs() / absref.clamp(min=1e-300)).max())


@gpu
@pytest.mark.parametrize('act', [NONE, LRELU, SIGMOID], ids=['none', 'lrelu', 'sigmoid'])
@pytest.mark.parametrize('halo', [False, True], ids=['box', 'halo'])
@pytest.mark.parametrize('name', ['gate_h1', 'pool_h1', 'd_conv1_1'])
def test_conv3x_forward_is_fp32_exact(L, monkeypatch, name, halo, act):
    """savp_model.conv3x (x_hi W_hi + x_lo W_hi + x_hi W_lo, the last pass adding bias and activation) against fp64 with
    the UNROUNDED operands: at least 30x closer than one TF32 pass, and within EXACT_BOUND."""
    from video_prediction_b200.models.savp_model import conv3x
    g = BY_NAME[name]
    _engine(monkeypatch, halo)
    S = _exact_operands(L, g, seed=100)
    out3 = torch.full(S.oshape + (g.co,), float('nan'), device='cuda')
    conv3x(S.xbuf, g.cs, S.geom, S.wp, S.wp_lo, S.n_pad, S.kc, L.tensor_view(out3, g.co), S.bias, act, 0.2)
    out1 = torch.full_like(out3, float('nan'))
    _run_fwd(L, S, out1, L.tensor_view(out1, g.co), act=act, split_k=1)
    x = S.xbuf.double()
    pre = S.fwd64(x, S.K) + S.bias.double()
    ref = act64(pre, act, 0.2)
    absref = S.fwd64(x.abs(), S.K.abs()) + S.bias.double().abs()
    r3, r1 = _max_ratio(out3, ref, absref), _max_ratio(out1, ref, absref)
    RATIOS['exact'] = max(RATIOS.get('exact', 0.0), r3)
    assert r3 * 30 <= r1, '%s: 3xTF32 %.3g vs one pass %.3g' % (name, r3, r1)
    assert r3 <= EXACT_BOUND, '%s: 3xTF32 ratio %.3g' % (name, r3)


@gpu
@pytest.mark.parametrize('halo', [False, True], ids=['box', 'halo'])
@pytest.mark.parametrize('name', ['d_conv1_0', 'd_conv2_1'])
def test_conv3x_actgrad_is_fp32_exact(L, monkeypatch, name, halo):
    """conv3x with the fused activation gradient (the discriminator dgrad in exact mode)."""
    from video_prediction_b200.models.savp_model import conv3x
    g = BY_NAME[name]
    _engine(monkeypatch, halo)
    S = _exact_operands(L, g, seed=110)
    shape = g.xs + (g.cs,)
    y = torch.sigmoid(rnd(*shape, seed=111))
    add = rnd(*shape, seed=112)
    dx = torch.full(shape, float('nan'), device='cuda')
    conv3x(S.dybuf, g.co, S.geom_d, S.wpd, S.wpd_lo, S.n_pad_d, S.kc_d, L.tensor_view(dx, g.cs), None, NONE, 0.2,
           aux=(y.data_ptr(), add.data_ptr(), SIGMOID))
    dx1 = torch.full(shape, float('nan'), device='cuda')
    L.conv_igemm_actgrad(L.tensor_view(S.dybuf, g.co), S.geom_d, S.wpd, S.n_pad_d, S.kc_d, L.tensor_view(dx1, g.cs), y.data_ptr(),
                         add.data_ptr(), SIGMOID, 0.2)
    torch.cuda.synchronize()
    dy = S.dybuf[..., :g.co].double()
    x = torch.zeros(shape, dtype=torch.float64, device='cuda', requires_grad=True)
    (conv,) = torch.autograd.grad(S.fwd64(x, S.K), x, dy)
    (absref,) = torch.autograd.grad(S.fwd64(x, S.K.abs()), x, dy.abs())
    d = _act_deriv64(y, SIGMOID, 0.2)
    ref, absref = (conv + add.double()) * d, (absref + add.double().abs()) * d
    r3, r1 = _max_ratio(dx, ref, absref), _max_ratio(dx1, ref, absref)
    RATIOS['exact'] = max(RATIOS.get('exact', 0.0), r3)
    assert r3 * 30 <= r1, '%s: 3xTF32 %.3g vs one pass %.3g' % (name, r3, r1)
    assert r3 <= EXACT_BOUND, '%s: 3xTF32 ratio %.3g' % (name, r3)


@gpu
@pytest.mark.parametrize('name', ['gate_h0', 'pool_h1', 'up_h3', 'd_conv1_0', 'masks'])
def test_three_pass_wgrad_is_fp32_exact(L, name):
    """The weight gradient as ConvLayer.wgrad issues it in exact mode: x^T dy + x_lo^T dy + x^T dy_lo (split_k = 0)."""
    g = BY_NAME[name]
    S = _exact_operands(L, g, seed=120)
    taps = L.eff_taps(g.k, g.kind)
    xv, dyv = L.tensor_view(S.xbuf, g.cs), L.tensor_view(S.dybuf, g.co)
    dwp3 = torch.zeros(taps * S.n_pad * S.kc * 32, device='cuda')
    L.conv_wgrad(xv, dyv, S.geom, dwp3, S.n_pad, S.kc, split_k=0)
    L.conv_wgrad(L.tensor_view(L.tf32_residual(S.xbuf), g.cs), dyv, S.geom, dwp3, S.n_pad, S.kc, split_k=0)
    L.conv_wgrad(xv, L.tensor_view(L.tf32_residual(S.dybuf), g.co), S.geom, dwp3, S.n_pad, S.kc, split_k=0)
    dwp1 = torch.zeros_like(dwp3)
    L.conv_wgrad(xv, dyv, S.geom, dwp1, S.n_pad, S.kc, split_k=0)
    torch.cuda.synchronize()
    x, dy = S.xbuf.double(), S.dybuf[..., :g.co].double()
    Pv = torch.zeros(taps, g.co, g.cs, dtype=torch.float64, device='cuda', requires_grad=True)
    (ref,) = torch.autograd.grad(S.fwd64(x, Pv), Pv, dy)
    (absref,) = torch.autograd.grad(S.fwd64(x.abs(), Pv), Pv, dy.abs())
    sl = (slice(None), slice(0, g.co), slice(0, g.cs))
    r3 = _max_ratio(dwp3.view(taps, S.n_pad, -1)[sl], ref, absref)
    r1 = _max_ratio(dwp1.view(taps, S.n_pad, -1)[sl], ref, absref)
    RATIOS['exact'] = max(RATIOS.get('exact', 0.0), r3)
    assert r3 * 30 <= r1, '%s: 3xTF32 %.3g vs one pass %.3g' % (name, r3, r1)
    assert r3 <= EXACT_BOUND, '%s: 3xTF32 ratio %.3g' % (name, r3)


# ------------------------------------------------------------------ the autotuner
@gpu
def test_autotuner_times_an_accumulating_call_on_a_snapshot(L, monkeypatch):
    """_pick_engine times both engines with repeated launches; an accumulate = 1 dgrad must still leave P + conv (the
    output is snapshotted and restored), and the choice is then cached."""
    monkeypatch.setattr(L, '_ENGINE_CHOICE', {})
    monkeypatch.delenv('VP_HALO', raising=False)
    monkeypatch.delenv('VP_AUTOTUNE', raising=False)
    g = Geo('autotune', PLAIN, (1, 3, 3), S1, (0, 1, 1), False, (3, 1, 24, 40), 48, 80)
    S = Setup(L, g, seed=130)
    prior = rnd(*g.xs, g.cs, seed=131)
    dx = prior.clone()
    L.conv_igemm(L.tensor_view(S.dybuf, g.co), S.geom_d, S.wpd, S.n_pad_d, S.kc_d, L.tensor_view(dx, g.cs), None, NONE, 0.0, 1, 1)
    torch.cuda.synchronize()
    assert len(L._ENGINE_CHOICE) == 1
    dy = S.dy_ref()
    x = torch.zeros(g.xs + (g.cs,), dtype=torch.float64, device='cuda', requires_grad=True)
    (ref,) = torch.autograd.grad(S.fwd64(x, S.P), x, dy)
    (absref,) = torch.autograd.grad(S.fwd64(x, S.P.abs()), x, dy.abs())
    check('dgrad', dx, ref + prior.double(), absref + prior.double().abs(), 'autotuned accumulate dgrad')
    choice = dict(L._ENGINE_CHOICE)
    dx2 = prior.clone()
    L.conv_igemm(L.tensor_view(S.dybuf, g.co), S.geom_d, S.wpd, S.n_pad_d, S.kc_d, L.tensor_view(dx2, g.cs), None, NONE, 0.0, 1, 1)
    torch.cuda.synchronize()
    assert L._ENGINE_CHOICE == choice
    assert L.last_launch()[0] == list(choice.values())[0]
    check('dgrad', dx2, ref + prior.double(), absref + prior.double().abs(), 'cached engine')
