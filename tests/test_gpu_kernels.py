"""GPU unit tests (-m gpu): every hand-written kernel against the oracle's op (fp32 / fp64, torch autograd for the
backward kernels).  HBM-bound kernels are plain fp32 -> tight tolerances; tensor-core convolutions compute on
TF32-truncated operands -> compared with an fp64 reference on TF32-rounded inputs, relative tolerance 2e-3."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import savp_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def L():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from video_prediction_b200 import lib
    lib.lib()
    return lib


def rnd(*s, seed=0, scale=1.0):
    g = torch.Generator(device='cpu').manual_seed(seed)
    return (torch.randn(*s, generator=g) * scale).cuda()


def tf32(x):
    xi = x.contiguous().view(torch.int32)
    xi = (xi + 0x0FFF + ((xi >> 13) & 1)) & ~0x1FFF
    return xi.view(torch.float32)


def close(a, b, tol, what=''):
    err = (a.double().cpu() - b.double().cpu()).abs().max().item()
    sc = b.double().abs().max().item() + 1e-30
    assert err <= tol * max(sc, 1.0), '%s: max err %g (ref max %g)' % (what, err, sc)


# ------------------------------------------------------------------ tensor-core engine
def _ke(L, k, kind):
    return k if kind == L.WKIND_PLAIN else ((1, k[1] + 1, k[2] + 1) if kind == L.WKIND_POOLED else (1, k[1] + 3, k[2] + 3))


def _fwd(L, x, c_used, w, k, s, p, out_shape, kind=0, transposed=False, bias=None, act=0, alpha=0.0, split_k=1):
    ci_ref, co = w.shape[-2], w.shape[-1]
    wp, n_pad, kc = L.pack_weights(w.contiguous(), k, ci_ref, co, kind, L.WLAYOUT_FWD, ci_int=c_used)
    out = torch.zeros(*out_shape, co, device='cuda')
    L.conv_igemm(L.tensor_view(x, c_used), L.geom(_ke(L, k, kind), s, p, transposed), wp, n_pad, kc, L.tensor_view(out, co), bias,
                 act, alpha, split_k)
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize('B,H,Cin,Cout', [(4, 32, 72, 128), (6, 8, 264, 512), (3, 16, 136, 256)])
def test_convlstm_gate_conv(L, B, H, Cin, Cout):
    x, w = rnd(B, H, H, Cin), rnd(5, 5, Cin, Cout, seed=1, scale=0.05)
    y = _fwd(L, x, Cin, w, (1, 5, 5), (1, 1, 1), (0, 2, 2), (B, H, H))
    ref = O.conv2d_tf(tf32(x).double(), tf32(w).double(), padding='SAME')
    close(y, ref, 2e-3, 'gate conv')
    y2 = _fwd(L, x, Cin, w, (1, 5, 5), (1, 1, 1), (0, 2, 2), (B, H, H), split_k=3)
    close(y2, ref, 2e-3, 'gate conv split-k')


def test_conv_pool2d_and_upsample_conv2d(L):
    x, w, b = rnd(2, 64, 64, 16), rnd(5, 5, 14, 32, seed=1, scale=0.1), rnd(32, seed=2)
    y = _fwd(L, x, 14, w, (1, 5, 5), (1, 2, 2), (0, 2, 2), (2, 32, 32), kind=L.WKIND_POOLED, bias=b)
    close(y, O.conv_pool2d(tf32(x)[..., :14].double(), w.double(), b.double()), 2e-3, 'conv_pool2d')
    x, w, b = rnd(2, 8, 8, 136), rnd(3, 3, 136, 64, seed=1, scale=0.05), rnd(64, seed=2)
    y = _fwd(L, x, 136, w, (1, 3, 3), (1, 2, 2), (0, 2, 2), (2, 16, 16), kind=L.WKIND_UPSAMPLED, transposed=True, bias=b)
    close(y, O.upsample_conv2d(tf32(x).double(), w.double(), b.double()), 2e-3, 'upsample_conv2d')


@pytest.mark.parametrize('k,s,cin,cout,shape', [(3, (1, 1, 1), 3, 32, (2, 6, 16, 16)), (4, (1, 2, 2), 32, 64, (2, 10, 32, 32)),
                                                (4, (2, 2, 2), 64, 128, (2, 8, 16, 16))])
def test_conv3d_padded_valid(L, k, s, cin, cout, shape):
    cs = (cin + 3) // 4 * 4
    x, w, b = rnd(*shape, cs), rnd(k, k, k, cin, cout, seed=1, scale=0.05), rnd(cout, seed=2)
    od = tuple((d + 2 - k) // st + 1 for d, st in zip(shape[1:], s))
    y = _fwd(L, x, cin, w, (k, k, k), s, (1, 1, 1), (shape[0],) + od, bias=b, act=L.ACT_LRELU, alpha=0.1)
    xp = F.pad(tf32(x)[..., :cin].double(), (0, 0, 1, 1, 1, 1, 1, 1))
    ref = O.lrelu(O.conv3d_tf_valid(xp, tf32(w).double(), s, b.double()), 0.1)
    close(y, ref, 2e-3, 'conv3d')


def test_dgrad_and_wgrad_match_autograd(L):
    for kind, k, s, p, transposed, xs, ys, cin, cout, fn in [
        (L.WKIND_PLAIN, (1, 5, 5), (1, 1, 1), (0, 2, 2), False, (2, 16, 16), (2, 16, 16), 72, 128,
         lambda x, w: O.conv2d_tf(x, w, padding='SAME')),
        (L.WKIND_POOLED, (1, 3, 3), (1, 2, 2), (0, 1, 1), False, (2, 32, 32), (2, 16, 16), 40, 64,
         lambda x, w: O.conv_pool2d(x, w, torch.zeros(64, device='cuda', dtype=torch.float64))),
        (L.WKIND_UPSAMPLED, (1, 3, 3), (1, 2, 2), (0, 2, 2), True, (2, 8, 8), (2, 16, 16), 136, 64,
         lambda x, w: O.upsample_conv2d(x, w, torch.zeros(64, device='cuda', dtype=torch.float64))),
    ]:
        x, dy = rnd(*xs, cin), rnd(*ys, cout, seed=1)
        w = rnd(k[1], k[2], cin, cout, seed=2, scale=0.05)
        xd = tf32(x).double().requires_grad_(True)
        wd = w.double().requires_grad_(True)
        gx, gw = torch.autograd.grad(fn(xd, wd), (xd, wd), tf32(dy).double())
        wpd, n_pad, kc = L.pack_weights(w, k, cin, cout, kind, L.WLAYOUT_DGRAD, ci_int=cin)
        dx = torch.zeros(*xs, cin, device='cuda')
        L.conv_igemm(L.tensor_view(dy, cout), L.geom(_ke(L, k, kind), s, p, not transposed), wpd, n_pad, kc, L.tensor_view(dx, cin))
        close(dx, gx, 3e-3, 'dgrad kind %d' % kind)
        n_pad, kc = L.pad_to(cout, 16), L.pad_to(cin, 32) // 32
        ke = _ke(L, k, kind)
        dwp = torch.zeros(ke[1] * ke[2] * n_pad * kc * 32, device='cuda')
        L.conv_wgrad(L.tensor_view(x, cin), L.tensor_view(dy, cout), L.geom(ke, s, p, transposed), dwp, n_pad, kc, 4)
        dw = torch.zeros(k[1], k[2], cin, cout, device='cuda')
        L.unpack_wgrad(dwp, k, cin, cout, kind, dw, n_pad, kc, ci_int=cin)
        close(dw, gw, 3e-3, 'wgrad kind %d' % kind)


# ------------------------------------------------------------------ HBM-bound kernels, forward + backward
def test_inorm_act_fwd_bwd(L):
    N, P, C = 3, 256, 16
    x, g, b, dy = rnd(N, P, C) * 2 + 1, rnd(C, seed=1), rnd(C, seed=2), rnd(N, P, C, seed=3)
    y = torch.zeros(N, P, 24, device='cuda')
    st = torch.zeros(N, C, 2, device='cuda')
    L.inorm_act(x.data_ptr(), C, y.data_ptr() + 16, 24, N, P, C, g, b, L.ACT_LRELU, 0.2, st)
    xr = x.double().requires_grad_(True)
    gr, br = g.double().requires_grad_(True), b.double().requires_grad_(True)
    ref = O.lrelu(O.instance_norm(xr, gr, br), 0.2)
    close(y[..., 4:20], ref, 1e-5, 'inorm fwd')
    gx, gg, gb = torch.autograd.grad(ref, (xr, gr, br), dy.double())
    dx, dg, db = torch.zeros_like(x), torch.zeros(C, device='cuda'), torch.zeros(C, device='cuda')
    half = dy * 0.5
    L.inorm_act_bwd(x.data_ptr(), C, [(half.data_ptr(), C), (half.data_ptr(), C)], dx.data_ptr(), C, N, P, C, g, b, st, L.ACT_LRELU, 0.2,
                    dg, db)
    close(dx, gx, 2e-5, 'inorm dx')
    close(dg, gg, 2e-5, 'inorm dgamma')
    close(db, gb, 2e-5, 'inorm dbeta')


def test_lstm_gates_fwd_bwd(L):
    N, P, Fl = 2, 64, 8
    pre, c0 = rnd(N, P, 4 * Fl), rnd(N, P, Fl, seed=1)
    g1, b1, g2, b2 = rnd(4 * Fl, seed=2) * 0.3 + 1, rnd(4 * Fl, seed=3) * 0.1, rnd(Fl, seed=4) * 0.3 + 1, rnd(Fl, seed=5) * 0.1
    c1, h = torch.zeros(N, P, Fl, device='cuda'), torch.zeros(N, P, 12, device='cuda')
    s1, s2 = torch.zeros(N, 4 * Fl, 2, device='cuda'), torch.zeros(N, Fl, 2, device='cuda')
    L.lstm_gates_fwd(pre, N, P, Fl, c0, g1, b1, g2, b2, c1, [(h.data_ptr() + 16, 12)], s1, s2)
    prd, c0d = pre.double().requires_grad_(True), c0.double().requires_grad_(True)
    ps = [t.double().requires_grad_(True) for t in (g1, b1, g2, b2)]
    cat = O.instance_norm(prd, ps[0], ps[1])
    i, j, f, o = torch.split(cat, Fl, dim=-1)
    nc = O.instance_norm(c0d * torch.sigmoid(f + 1.0) + torch.sigmoid(i) * torch.tanh(j), ps[2], ps[3])
    nh = torch.tanh(nc) * torch.sigmoid(o)
    close(c1, nc, 1e-5, 'gates c')
    close(h[..., 4:12], nh, 1e-5, 'gates h')
    dh, dc = rnd(N, P, Fl, seed=6), rnd(N, P, Fl, seed=7)
    grads = torch.autograd.grad((nh * dh.double()).sum() + (nc * dc.double()).sum(), [prd, c0d] + ps)
    dpre, dc0 = torch.zeros_like(pre), torch.zeros_like(c0)
    dgs = [torch.zeros_like(t) for t in (g1, b1, g2, b2)]
    L.lstm_gates_bwd(pre, N, P, Fl, c0, g1, b1, g2, b2, s1, s2, [(dh.data_ptr(), Fl)], dc, dpre, dc0, dgs[0], dgs[1], dgs[2], dgs[3])
    close(dpre, grads[0], 3e-5, 'gates dpre')
    close(dc0, grads[1], 3e-5, 'gates dc_prev')
    for a, b_, nm in zip(dgs, grads[2:], ('dg1', 'db1', 'dg2', 'db2')):
        close(a, b_, 3e-5, 'gates ' + nm)


def test_cdna_and_composite_fwd_bwd(L):
    N, H, W, C, nk = 2, 16, 12, 3, 4
    img = torch.zeros(N, H, W, 4, device='cuda')
    img[..., :C] = torch.rand(N, H, W, C, device='cuda')
    first = torch.zeros_like(img)
    first[..., :C] = torch.rand(N, H, W, C, device='cuda')
    raw = rnd(N, 25 * nk, scale=0.3)
    kern = torch.zeros_like(raw)
    L.cdna_kernel_norm(raw, kern, N, 5, 5, nk)
    rawd = raw.double().view(N, 5, 5, nk).requires_grad_(True)
    k = torch.relu(rawd + torch.tensor(O.identity_kernel((5, 5)), device='cuda')[None, :, :, None] - 1e-12) + 1e-12
    k = k / k.sum(dim=(1, 2), keepdim=True)
    close(kern.view(N, 5, 5, nk), k, 1e-6, 'cdna kernel norm')
    nl = nk + 3
    layers = torch.zeros(N, H, W, 4 * nl, device='cuda')
    L.cdna_apply(img, first, kern, layers.data_ptr(), 4 * nl, N, H, W, 5, 5, nk)
    imgd = img[..., :C].double().requires_grad_(True)
    tr = O.apply_cdna_kernels(imgd, k) + [imgd, first[..., :C].double()]
    for l in range(nk + 2):
        close(layers[..., 4 * l:4 * l + C], tr[l], 1e-5, 'cdna layer %d' % l)
    scratch = torch.rand(N, H, W, C, device='cuda')
    layers[..., 4 * (nl - 1):4 * (nl - 1) + C] = scratch
    logits = rnd(N, H, W, 8, seed=3)
    masks, gen = torch.zeros(N, H, W, 8, device='cuda'), torch.zeros(N, H, W, 4, device='cuda')
    L.composite(logits, 8, layers.data_ptr(), 4 * nl, masks, 8, gen, N * H * W, nl)
    lgd = logits[..., :nl].double().requires_grad_(True)
    scd = scratch.double().requires_grad_(True)
    m = torch.softmax(lgd, dim=-1)
    full = tr + [scd]
    gref = sum(full[l] * m[..., l:l + 1] for l in range(nl))
    close(gen[..., :C], gref, 1e-5, 'composite gen')
    dgen = torch.zeros(N, H, W, 4, device='cuda')
    dgen[..., :C] = rnd(N, H, W, C, seed=4)
    g_l, g_s, g_i, g_r = torch.autograd.grad(gref, (lgd, scd, imgd, rawd), dgen[..., :C].double())
    dlog, dlay = torch.zeros(N, H, W, 8, device='cuda'), torch.zeros(N, H, W, 4 * nl, device='cuda')
    L.composite_bwd(dgen, masks, 8, layers.data_ptr(), 4 * nl, dlog, 8, dlay, 4 * nl, N * H * W, nl)
    close(dlog[..., :nl], g_l, 2e-5, 'composite dlogits')
    close(dlay[..., 4 * (nl - 1):4 * (nl - 1) + C], g_s, 2e-5, 'composite dscratch')
    dimg, dk = torch.zeros(N, H, W, 4, device='cuda'), torch.zeros_like(kern)
    zero = torch.zeros_like(dlay)
    L.cdna_apply_bwd(img, kern, dlay.data_ptr(), 4 * nl, zero.data_ptr(), 4 * nl, dimg, dk, N, H, W, 5, 5, nk)
    close(dimg[..., :C], g_i, 3e-5, 'cdna dimage')
    draw = torch.zeros_like(raw)
    L.cdna_kernel_norm_bwd(raw, kern, dk, draw, N, 5, 5, nk)
    close(draw.view(N, 5, 5, nk), g_r, 3e-5, 'cdna draw')


def test_dense_and_small_lstm_fwd_bwd(L):
    B, K, J = 5, 300, 10
    x, w, b, dy = rnd(B, K), rnd(K, J, seed=1, scale=0.1), rnd(J, seed=2), rnd(B, J, seed=3)
    y = torch.zeros(B, J, device='cuda')
    L.dense_fwd(x, K, w, b, y, J, B, K, J, k_splits=4)
    xd, wd, bd = [t.double().requires_grad_(True) for t in (x, w, b)]
    ref = xd @ wd + bd
    close(y, ref, 1e-5, 'dense fwd')
    gx, gw, gb = torch.autograd.grad(ref, (xd, wd, bd), dy.double())
    dx, dw, db = torch.zeros_like(x), torch.zeros_like(w), torch.zeros_like(b)
    L.dense_bwd(x, K, w, dy, J, B, K, J, dx=dx, dx_stride=K, dw=dw, dbias=db)
    close(dx, gx, 1e-5, 'dense dx'); close(dw, gw, 1e-5, 'dense dw'); close(db, gb, 1e-5, 'dense db')
    U = 8
    gates, c0, dh, dc = rnd(B, 4 * U), rnd(B, U, seed=1), rnd(B, U, seed=2), rnd(B, U, seed=3)
    c1, h1 = torch.zeros(B, U, device='cuda'), torch.zeros(B, U, device='cuda')
    L.lstm_cell_fwd(gates, c0, c1, h1, B, U)
    gd, cd = gates.double().requires_grad_(True), c0.double().requires_grad_(True)
    i, j, f, o = torch.split(gd, U, dim=-1)
    nc = torch.sigmoid(f + 1.0) * cd + torch.sigmoid(i) * torch.tanh(j)
    nh = torch.tanh(nc) * torch.sigmoid(o)
    close(c1, nc, 1e-5, 'lstm c'); close(h1, nh, 1e-5, 'lstm h')
    gg, gc = torch.autograd.grad((nh * dh.double()).sum() + (nc * dc.double()).sum(), (gd, cd))
    dg, dc0 = torch.zeros_like(gates), torch.zeros_like(c0)
    L.lstm_cell_bwd(gates, c0, c1, dh, dc, dg, dc0, B, U)
    close(dg, gg, 1e-5, 'lstm dgates'); close(dc0, gc, 1e-5, 'lstm dc')


def test_wide_dense_tiled_kernels(L):
    """The CDNA-kernel dense layer shapes (K >= 1024, J <= 128) take the tiled kernels; dW is called once over all time steps."""
    for B, K, J in [(32, 2048, 100), (70, 1100, 36), (16, 4096, 1), (5, 1030, 7)]:
        x, w, b, dy = rnd(B, K), rnd(K, J, seed=1, scale=0.05), rnd(J, seed=2), rnd(B, J, seed=3)
        sig = torch.tensor([1.7], device='cuda')
        y = torch.zeros(B, J, device='cuda')
        L.dense_fwd(x, K, w, b, y, J, B, K, J, k_splits=32, inv_scale=sig)
        xd, wd, bd = [t.double().requires_grad_(True) for t in (x, w, b)]
        ref = xd @ (wd / 1.7) + bd
        close(y, ref, 2e-5, 'wide dense fwd')
        gx, gw, gb = torch.autograd.grad(ref, (xd, wd, bd), dy.double())
        dx, dw, db = torch.zeros_like(x), torch.zeros_like(w), torch.zeros_like(b)
        L.dense_bwd(x, K, w, dy, J, B, K, J, dx=dx, dx_stride=K, dw=dw, dbias=db, inv_scale=sig)
        close(dx, gx, 2e-5, 'wide dense dx'); close(dw, gw, 2e-5, 'wide dense dw'); close(db, gb, 2e-5, 'wide dense db')


def test_losses_and_adam(L):
    rows, C = 1000, 3
    pred, tgt = torch.rand(rows, 4, device='cuda'), torch.rand(rows, 4, device='cuda')
    out, dp = torch.zeros(2, device='cuda'), torch.zeros(rows, 4, device='cuda')
    L.pixel_loss(pred.data_ptr(), 4, tgt.data_ptr(), 4, dp.data_ptr(), 4, rows, C, 0, rows * C, 2.0, out[0:1])
    pd = pred[:, :C].double().requires_grad_(True)
    ref = O.l1_loss(pd, tgt[:, :C].double())
    close(out[0:1], ref.reshape(1), 1e-5, 'l1 value')
    close(dp[:, :C], torch.autograd.grad(2.0 * ref, pd)[0], 1e-6, 'l1 grad')
    a, b = rnd(40, 16), rnd(40, 16, seed=1)
    da = torch.zeros_like(a)
    L.cosine_distance(a, b, da, 40, 16, 3.0, out[1:2])
    ad = a.double().requires_grad_(True)
    ref = O.cosine_distance(ad, b.double())
    close(out[1:2], ref.reshape(1), 1e-5, 'cdist value')
    close(da, torch.autograd.grad(3.0 * ref, ad)[0], 1e-5, 'cdist grad')
    n = 1000
    p, g = rnd(n), rnd(n, seed=1)
    m, v = torch.zeros(n, device='cuda'), torch.zeros(n, device='cuda')
    pr, mr, vr = p.clone().cpu(), torch.zeros(n), torch.zeros(n)
    import math
    for t in (1, 2, 3):
        lr_t = torch.tensor([1e-3 * math.sqrt(1 - 0.999 ** t) / (1 - 0.5 ** t)], device='cuda')
        L.adam(p, g, m, v, n, lr_t, 0.5, 0.999)
        pr, mr, vr = O.adam_tf(pr, g.cpu(), mr, vr, 1e-3, 0.5, 0.999, t)
    close(p, pr, 1e-6, 'adam')


def test_spectral_norm_fwd_bwd(L):
    R, Cc = 27 * 4, 32
    W, u, G = rnd(R, Cc, scale=0.1), rnd(1, Cc, seed=1), rnd(R, Cc, seed=2)
    v, s, un, scal = [torch.zeros(n, device='cuda') for n in (R, Cc, Cc, 4)]
    L.spectral_norm_fwd(W, u, R, Cc, v, s, un, scal)
    Wd = W.double().requires_grad_(True)
    Wb, u1 = O.spectral_normed_weight(Wd, u.double())
    sigma = (Wd / Wb).mean()
    close(scal[2:3], sigma.reshape(1), 1e-5, 'sigma')
    close(un, u1.reshape(-1), 1e-5, 'u_new')
    (gW,) = torch.autograd.grad(Wb, Wd, G.double())
    gs, gt, dW = torch.zeros(Cc, device='cuda'), torch.zeros(R, device='cuda'), torch.zeros_like(W)
    L.spectral_norm_bwd(W, u, G, R, Cc, v, s, scal, gs, gt, dW)
    close(dW, gW, 3e-5, 'sn backward')


def test_clip_gather_scatter(L):
    T, NB, P, B, clip = 7, 4, 10, 2, 3
    video = rnd(T, NB, P, 4)
    ts = torch.tensor([1, 4], dtype=torch.int32, device='cuda')
    out = torch.zeros(B, clip, P, 4, device='cuda')
    L.gather_clip(video, ts, out, B, clip, P, NB, 2)
    for b in range(B):
        assert torch.equal(out[b], video[int(ts[b]):int(ts[b]) + clip, 2 + b])
    dv = torch.zeros_like(video)
    L.scatter_clip(out, ts, dv, B, clip, P, NB, 2)
    assert torch.equal(dv[1:4, 2], video[1:4, 2]) and float(dv[:, :2].abs().sum()) == 0.0


@pytest.mark.parametrize('rows,C', [(1000, 32), (77, 64), (513, 128), (9, 256)])
def test_cosine_distance_vectorised_shapes(L, rows, C):
    """The discriminator feature widths: 32 / 64 / 128 channels take the float4 kernel (8 / 16 / 32 lanes per row), 256 the generic one."""
    a, b = rnd(rows, C), rnd(rows, C, seed=1)
    da = torch.full_like(a, 0.25)                                # accumulates
    out = torch.zeros(1, device='cuda')
    L.cosine_distance(a, b, da, rows, C, 3.0, out)
    ad = a.double().requires_grad_(True)
    ref = O.cosine_distance(ad, b.double())
    close(out, ref.reshape(1), 1e-5, 'cosine distance')
    close(da - 0.25, torch.autograd.grad(3.0 * ref, ad)[0], 1e-6, 'cosine distance grad')


def test_conv3d_c4_cuda_core_first_discriminator_layer(L):
    N, D, H, W, C = 2, 5, 16, 12, 3
    x = torch.zeros(N, D, H, W, 4, device='cuda')
    x[..., :C] = torch.rand(N, D, H, W, C, device='cuda')
    w, b, dy = rnd(3, 3, 3, C, 32, seed=1, scale=0.2), rnd(32, seed=2), rnd(N, D, H, W, 32, seed=3)
    sigma = torch.tensor([1.7], device='cuda')
    out = torch.zeros(N, D, H, W, 32, device='cuda')
    L.conv3d_c4_fwd(x, w, sigma, b, out, N, D, H, W, C, 0.1)
    wb = (w.double() / 1.7).requires_grad_(True)
    xp = F.pad(x[..., :C].double(), (0, 0, 1, 1, 1, 1, 1, 1))
    pre = O.conv3d_tf_valid(xp, wb, (1, 1, 1), b.double())
    close(out, O.lrelu(pre, 0.1), 1e-5, 'conv3d_c4 fwd')
    (gw,) = torch.autograd.grad(pre, wb, dy.double())
    g = torch.zeros(27 * C * 32, device='cuda')
    L.conv3d_c4_wgrad(x, dy, g, N, D, H, W, C)
    close(g.view(3, 3, 3, C, 32), gw, 2e-5, 'conv3d_c4 wgrad')


@pytest.mark.parametrize('N,D,H,W,C', [(2, 3, 5, 64, 3), (1, 2, 3, 128, 1), (3, 10, 64, 64, 3)])
def test_conv3d_c4_wgrad_tensor_cores(L, N, D, H, W, C):
    """vp_conv3d_c4_wgrad_tc (float4 voxel rows as the un-swizzled MN-major UMMA operand, one MMA per dx) against the fp64
    weight gradient of the operands the tensor core reads (fp32 truncated to TF32), and against the CUDA-core kernel."""
    def trunc(t):
        return (t.contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)
    x = torch.zeros(N, D, H, W, 4, device='cuda')
    x[..., :C] = torch.rand(N, D, H, W, C, device='cuda') - 0.3
    x[..., C:] = 7.0                                           # padding channels must not leak into real taps
    dy = rnd(N, D, H, W, 32, seed=3)
    wz = torch.zeros(3, 3, 3, C, 32, device='cuda', dtype=torch.float64, requires_grad=True)
    xp = F.pad(trunc(x)[..., :C].double(), (0, 0, 1, 1, 1, 1, 1, 1))
    pre = O.conv3d_tf_valid(xp, wz, (1, 1, 1), None)
    (gw,) = torch.autograd.grad(pre, wz, trunc(dy).double())
    g = torch.full((27 * C * 32,), 0.5, device='cuda')         # accumulates
    L.check(L.lib().vp_conv3d_c4_wgrad_tc(L.ptr(x), L.ptr(dy), L.ptr(g), N, D, H, W, C, L.stream_ptr()))
    torch.cuda.synchronize()
    err = (g.view(3, 3, 3, C, 32).double() - 0.5 - gw).norm() / gw.norm()
    assert err < 2e-4, 'tensor-core first-layer wgrad: rel L2 %g' % err.item()
    g2 = torch.zeros(27 * C * 32, device='cuda')
    L.check(L.lib().vp_conv3d_c4_wgrad(L.ptr(x), L.ptr(dy), L.ptr(g2), N, D, H, W, C, L.stream_ptr()))
    err2 = (g - 0.5 - g2).norm() / g2.norm()
    assert err2 < 3e-3, 'tensor cores vs CUDA cores: rel L2 %g' % err2.item()


@pytest.mark.parametrize('N,D,H,W,C', [(2, 3, 16, 64, 3), (1, 2, 8, 128, 1), (3, 4, 64, 64, 3), (1, 2, 12, 20, 2)])
def test_conv3d_c4_fwd_tensor_cores(L, N, D, H, W, C):
    """vp_conv3d_c4_fwd_tc (flat halo tile of float4 voxels as the un-swizzled K-major operand, LBO = one voxel) against the
    fp64 convolution of the operands the tensor core sees (x truncated to TF32, w / sigma rounded to TF32) and the CUDA-core kernel."""
    def trunc(t):
        return (t.contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)
    x = torch.zeros(N, D, H, W, 4, device='cuda')
    x[..., :C] = torch.rand(N, D, H, W, C, device='cuda') - 0.3
    x[..., C:] = 5.0                                           # padding channels must meet zero weights
    w, b = rnd(3, 3, 3, C, 32, seed=1, scale=0.2), rnd(32, seed=2)
    sigma = torch.tensor([1.7], device='cuda')
    out = torch.full((N, D, H, W, 32), -3.0, device='cuda')
    L.conv3d_c4_fwd_tc(x, w, sigma, b, out, N, D, H, W, C, 0.1)
    xp = F.pad(trunc(x)[..., :C].double(), (0, 0, 1, 1, 1, 1, 1, 1))
    ref = O.lrelu(O.conv3d_tf_valid(xp, tf32(w / sigma).double(), (1, 1, 1), b.double()), 0.1)
    close(out, ref, 2e-5, 'first layer forward on the tensor cores')
    out2 = torch.zeros_like(out)
    L.conv3d_c4_fwd(x, w, sigma, b, out2, N, D, H, W, C, 0.1)
    close(out, out2, 3e-3, 'tensor cores vs CUDA cores')


def test_pack_weights_batch_equals_per_tensor_packs(L):
    """vp_pack_weights_batch (one table-driven launch) writes exactly what the per-tensor launches write."""
    cases = [((1, 5, 5), 72, 128, L.WKIND_PLAIN), ((1, 3, 3), 40, 32, L.WKIND_POOLED), ((1, 3, 3), 64, 16, L.WKIND_UPSAMPLED),
             ((3, 3, 3), 3, 32, L.WKIND_PLAIN), ((1, 4, 4), 136, 264, L.WKIND_PLAIN)]
    entries, refs = [], []
    for i, (k, ci, co, kind) in enumerate(cases):
        w = rnd(*k, ci, co, seed=i, scale=0.1)
        ci_int = ((ci + 3) // 4) * 4 + 4
        cmap = torch.arange(ci_int, dtype=torch.int32, device='cuda')
        cmap[ci:] = -1
        sigma = torch.tensor([1.3 + i], device='cuda') if i % 2 else None
        for layout in (L.WLAYOUT_FWD, L.WLAYOUT_DGRAD):
            ref, n_pad, kc = L.pack_weights(w, k, ci, co, kind, layout, ci_int=ci_int, cmap=cmap, inv_scale=sigma)
            out = torch.full_like(ref, -7.0)
            entries.append((w, k, ci, co, kind, layout, ci_int, cmap, sigma, out))
            refs.append(ref)
    plan = L.PackPlan(entries)
    plan.run()
    torch.cuda.synchronize()
    for e, ref in zip(entries, refs):
        assert torch.equal(e[-1], ref)


def test_image_warp_fwd_bwd(L):
    N, H, W, C = 2, 9, 11, 3
    im = torch.zeros(N, H, W, 4, device='cuda')
    im[..., :C] = torch.rand(N, H, W, C, device='cuda')
    flow = rnd(N, H, W, 2, seed=1) * 2.5 + 0.37          # non-integer displacements, some leaving the image
    out = torch.zeros(N, H, W, 4, device='cuda')
    L.image_warp_fwd(im, 4, flow, out, 4, N, H, W, C)
    imd = im[..., :C].double().requires_grad_(True)
    fd = flow.double().requires_grad_(True)
    ref = O.image_warp(imd, fd)
    close(out[..., :C], ref, 1e-5, 'image_warp fwd')
    dout = torch.zeros(N, H, W, 4, device='cuda')
    dout[..., :C] = rnd(N, H, W, C, seed=2)
    g_im, g_fl = torch.autograd.grad(ref, (imd, fd), dout[..., :C].double())
    dim, dfl = torch.zeros(N, H, W, 4, device='cuda'), torch.zeros(N, H, W, 2, device='cuda')
    L.image_warp_bwd(im, 4, flow, dout, 4, dim, 4, dfl, N, H, W, C)
    close(dim[..., :C], g_im, 2e-5, 'image_warp dim')
    close(dfl, g_fl, 2e-5, 'image_warp dflow')


def test_flow_apply_fwd_bwd(L):
    # transformation='flow': NK bilinear warps of the previous image + the two background slots, against oracle.image_warp + autograd
    N, H, W, NK = 2, 16, 20, 4
    im = torch.zeros(N, H, W, 4, device='cuda')
    im[..., :3] = rnd(N, H, W, 3)
    first = torch.zeros(N, H, W, 4, device='cuda')
    first[..., :3] = rnd(N, H, W, 3, seed=1)
    flows = rnd(N, H, W, 2 * NK, seed=2, scale=2.5)
    ls = 4 * (NK + 3) + 8
    layers = torch.zeros(N, H, W, ls, device='cuda')
    L.flow_apply(im, first, flows, 2 * NK, layers.data_ptr() + 4 * 8, ls, N, H, W, NK)
    imd = im[..., :3].double().requires_grad_(True)
    fd = flows.double().requires_grad_(True)
    outs = [O.image_warp(imd, torch.stack([fd[..., k], fd[..., NK + k]], dim=-1)) for k in range(NK)]
    for k in range(NK):
        close(layers[..., 8 + 4 * k:8 + 4 * k + 3], outs[k], 1e-5, 'flow warp %d' % k)
    close(layers[..., 8 + 4 * NK:8 + 4 * NK + 3], im[..., :3], 0, 'prev image slot')
    close(layers[..., 8 + 4 * NK + 4:8 + 4 * NK + 7], first[..., :3], 0, 'first image slot')
    dA, dB = rnd(N, H, W, ls, seed=3), rnd(N, H, W, 4 * (NK + 3), seed=4)
    dimg = torch.zeros(N, H, W, 4, device='cuda')
    dfl = torch.zeros(N, H, W, 2 * NK, device='cuda')
    L.flow_apply_bwd(im, flows, 2 * NK, dA.data_ptr() + 4 * 8, ls, dB.data_ptr(), 4 * (NK + 3), dimg, dfl, N, H, W, NK)
    loss = sum(((dA[..., 8 + 4 * k:8 + 4 * k + 3] + dB[..., 4 * k:4 * k + 3]).double() * outs[k]).sum() for k in range(NK))
    loss = loss + ((dA[..., 8 + 4 * NK:8 + 4 * NK + 3] + dB[..., 4 * NK:4 * NK + 3]).double() * imd).sum()
    gi, gf = torch.autograd.grad(loss, (imd, fd))
    close(dimg[..., :3], gi, 2e-5, 'flow dimage')
    close(dfl, gf, 2e-5, 'dflows')


# ------------------------------------------------------------------ slab-mapped plane kernels (csrc/planes.cu)
@pytest.mark.parametrize('N,P,C', [(3, 64, 32), (2, 256, 64), (32, 1024, 32), (4, 4096, 32), (32, 4096, 32), (2, 16, 256), (5, 1024, 128)])
def test_slab_instance_norm_fwd_bwd(L, N, P, C):
    """Shapes of the model's instance norms (32-channel 64x64 / 32x32 planes ... 256-channel 4x4) on the cluster / DSMEM kernels:
    an input with a large mean (5 sigma) checks the shifted one-pass variance; two gradient sources, strided destination."""
    x, g, b, dy = rnd(N, P, C) * 0.7 + 3.5, rnd(C, seed=1) * 0.3 + 1, rnd(C, seed=2), rnd(N, P, C, seed=3)
    ys = C + 8
    y = torch.zeros(N, P, ys, device='cuda')
    st = torch.zeros(N, C, 2, device='cuda')
    L.inorm_act(x.data_ptr(), C, y.data_ptr() + 16, ys, N, P, C, g, b, L.ACT_RELU, 0.0, st)
    xr = x.double().requires_grad_(True)
    gr, br = g.double().requires_grad_(True), b.double().requires_grad_(True)
    ref = torch.relu(O.instance_norm(xr, gr, br))
    close(y[..., 4:4 + C], ref, 1e-5, 'slab inorm fwd')
    assert float(y[..., :4].abs().max()) == 0 and float(y[..., 4 + C:].abs().max()) == 0       # neighbours of the slice untouched
    gx, gg, gb = torch.autograd.grad(ref, (xr, gr, br), dy.double())
    dx, dg, db = torch.zeros_like(x), torch.zeros(C, device='cuda'), torch.zeros(C, device='cuda')
    half = dy * 0.5
    L.inorm_act_bwd(x.data_ptr(), C, [(half.data_ptr(), C), (half.data_ptr(), C)], dx.data_ptr(), C, N, P, C, g, b, st, L.ACT_RELU, 0.0,
                    dg, db)
    close(dx, gx, 3e-5, 'slab inorm dx')
    close(dg, gg, 3e-5, 'slab inorm dgamma')
    close(db, gb, 3e-5, 'slab inorm dbeta')


@pytest.mark.parametrize('N,P,Fl', [(32, 1024, 32), (6, 256, 64), (32, 256, 64), (5, 64, 128), (32, 64, 128), (2, 1024, 64), (3, 16, 256)])
def test_slab_lstm_gates_fwd_bwd(L, N, P, Fl):
    pre, c0 = rnd(N, P, 4 * Fl) + 0.8, rnd(N, P, Fl, seed=1)
    g1, b1, g2, b2 = rnd(4 * Fl, seed=2) * 0.3 + 1, rnd(4 * Fl, seed=3) * 0.1, rnd(Fl, seed=4) * 0.3 + 1, rnd(Fl, seed=5) * 0.1
    hs = Fl + 8
    c1, h, h2 = torch.zeros(N, P, Fl, device='cuda'), torch.zeros(N, P, hs, device='cuda'), torch.zeros(N, P, Fl, device='cuda')
    s1, s2 = torch.zeros(N, 4 * Fl, 2, device='cuda'), torch.zeros(N, Fl, 2, device='cuda')
    L.lstm_gates_fwd(pre, N, P, Fl, c0, g1, b1, g2, b2, c1, [(h.data_ptr() + 16, hs), (h2.data_ptr(), Fl)], s1, s2)
    prd, c0d = pre.double().requires_grad_(True), c0.double().requires_grad_(True)
    ps = [t.double().requires_grad_(True) for t in (g1, b1, g2, b2)]
    cat = O.instance_norm(prd, ps[0], ps[1])
    i, j, f, o = torch.split(cat, Fl, dim=-1)
    nc = O.instance_norm(c0d * torch.sigmoid(f + 1.0) + torch.sigmoid(i) * torch.tanh(j), ps[2], ps[3])
    nh = torch.tanh(nc) * torch.sigmoid(o)
    close(c1, nc, 1e-5, 'slab gates c')
    close(h[..., 4:4 + Fl], nh, 2e-5, 'slab gates h')          # __expf / fast tanh: 1.04e-5 measured at 32 x 1024 x 32
    close(h2, nh, 2e-5, 'slab gates h (2nd destination)')
    dh, dc = rnd(N, P, Fl, seed=6), rnd(N, P, Fl, seed=7)
    grads = torch.autograd.grad((nh * dh.double()).sum() + (nc * dc.double()).sum(), [prd, c0d] + ps)
    dpre, dc0 = torch.zeros_like(pre), torch.zeros_like(c0)
    dgs = [torch.zeros_like(t) for t in (g1, b1, g2, b2)]
    L.lstm_gates_bwd(pre, N, P, Fl, c0, g1, b1, g2, b2, s1, s2, [(dh.data_ptr(), Fl)], dc, dpre, dc0, dgs[0], dgs[1], dgs[2], dgs[3])
    close(dpre, grads[0], 5e-5, 'slab gates dpre')
    close(dc0, grads[1], 5e-5, 'slab gates dc_prev')
    for a, b_, nm in zip(dgs, grads[2:], ('dg1', 'db1', 'dg2', 'db2')):
        close(a, b_, 5e-5, 'slab gates ' + nm)


# ------------------------------------------------------------------ losses, sampling and small reductions
def _rel(a, b, scale, tol, what):
    err = float((a.double() - b.double()).abs().max())
    assert err <= tol * scale, '%s: max err %g (scale %g)' % (what, err, scale)


@pytest.mark.parametrize('n', [1, 300, 4096])
@pytest.mark.parametrize('label', [0.0, 1.0])
@pytest.mark.parametrize('kind', ['LSGAN', 'GAN', 'SNGAN'])
def test_gan_loss(L, kind, label, n):
    """Value and gradient against O.gan_loss in fp64, logits up to +-90 (value and gradient finite, the softplus form), the
    loss ACCUMULATED into out; n = 300 and 4096 exceed one block's stride."""
    logits = rnd(n, seed=n) * 3.0
    logits[:min(n, 4)] = torch.tensor([30.0, -30.0, 90.0, -90.0], device='cuda')[:min(n, 4)]
    out = torch.full((1,), 0.5, device='cuda')
    dl = torch.full((n,), float('nan'), device='cuda')
    L.gan_loss(logits, label, n, 2.5, kind, dl, out)
    torch.cuda.synchronize()
    ld = logits.double().requires_grad_(True)
    ref = O.gan_loss(ld, label, kind)
    # gradient of the softplus form (the sigmoid cross-entropy form cancels in fp64 too: sigmoid(30) - 1)
    (g,) = torch.autograd.grad(2.5 * O.gan_loss(ld, label, 'SNGAN' if kind == 'GAN' else kind), ld)
    assert bool(torch.isfinite(out).all()) and bool(torch.isfinite(dl).all())
    _rel(out - 0.5, ref.detach().reshape(1), max(1.0, abs(float(ref))), 1e-5, '%s value' % kind)
    err = (dl.double() - g).abs()
    assert bool((err <= 3e-5 * g.abs() + 1e-38).all()), '%s gradient: max err %g' % (kind, float(err.max()))   # per element


@pytest.mark.parametrize('rows,nz', [(7, 8), (300, 8), (2, 1)])
def test_kl_loss(L, rows, nz):
    mu, lss = rnd(rows, nz, seed=1) * 2, (torch.rand(rows, nz, device='cuda') * 20 - 10)
    lss.view(-1)[:2] = torch.tensor([10.0, -10.0], device='cuda')[:lss.numel()]
    out = torch.full((1,), -1.25, device='cuda')
    L.kl_loss(mu, lss, rows, nz, out)
    torch.cuda.synchronize()
    ref = O.kl_loss(mu.double(), lss.double())
    terms = (1 + lss.double().abs() + mu.double() ** 2 + torch.exp(lss.double())).sum() / rows
    _rel(out + 1.25, ref.reshape(1), float(terms), 2e-6, 'kl value')


def test_sample_z_clips_and_writes_back(L):
    total = 1000
    mu, eps = rnd(total, seed=1), rnd(total, seed=2)
    lss = rnd(total, seed=3) * 9.0                                    # a good share beyond +-10
    lss0 = lss.clone()
    z = torch.full((total,), float('nan'), device='cuda')
    L.sample_z(mu, lss, eps, z, total)
    torch.cuda.synchronize()
    assert int((lss0.abs() > 10).sum()) > 50
    assert torch.equal(lss, lss0.clamp(-10.0, 10.0))
    ref = mu.double() + torch.sqrt(torch.exp(lss.double())) * eps.double()
    err = (z.double() - ref).abs() / (mu.double().abs() + torch.sqrt(torch.exp(lss.double())) * eps.double().abs())
    assert float(err.max()) <= 2e-6


@pytest.mark.parametrize('dz_on', [True, False], ids=['dz', 'no_dz'])
@pytest.mark.parametrize('kl_on', [True, False], ids=['kl', 'no_kl'])
def test_sample_z_bwd(L, dz_on, kl_on):
    """dmu = dz + k mu, dlss = dz eps sqrt(e^l) / 2 + k (e^l - 1) / 2, zero where lss was clipped; kl_scale / dz may be NULL."""
    total = 777
    mu, eps, dz = rnd(total, seed=1), rnd(total, seed=2), rnd(total, seed=3)
    lss = rnd(total, seed=4) * 9.0
    z = torch.zeros(total, device='cuda')
    L.sample_z(mu, lss, eps, z, total)                                # lss now clipped, some exactly +-10
    k = torch.tensor([0.37], device='cuda') if kl_on else None
    dmu, dlss = torch.full_like(mu, float('nan')), torch.full_like(mu, float('nan'))
    L.sample_z_bwd(mu, lss, eps, dz if dz_on else None, dmu, dlss, total, k)
    torch.cuda.synchronize()
    kv = 0.37 if kl_on else 0.0
    d = dz.double() if dz_on else torch.zeros(total, dtype=torch.float64, device='cuda')
    e = torch.exp(lss.double())
    rmu = d + kv * mu.double()
    rl = torch.where(lss.abs() < 10, d * eps.double() * 0.5 * torch.sqrt(e) + kv * 0.5 * (e - 1), torch.zeros_like(e))
    _rel(dmu, rmu, float(rmu.abs().max()) + 1e-30, 1e-6, 'dmu')
    sc = (d.abs() * eps.double().abs() * 0.5 * torch.sqrt(e) + kv * 0.5 * (e + 1))
    assert float(((dlss.double() - rl).abs() / sc.clamp(min=1e-30)).max()) <= 2e-6
    assert bool((dlss[lss.abs() >= 10] == 0).all()) and int((lss.abs() >= 10).sum()) > 50


@pytest.mark.parametrize('two', [False, True], ids=['dy_a', 'dy_a+dy_b'])
@pytest.mark.parametrize('act', [1, 2, 3, 4], ids=['relu', 'lrelu', 'sigmoid', 'tanh'])
def test_act_bwd_on_strided_views(L, act, two):
    rows, c = 301, 6
    pre = rnd(rows, 8, seed=1)
    y = {1: torch.relu(pre), 2: torch.where(pre > 0, pre, 0.2 * pre), 3: torch.sigmoid(pre), 4: torch.tanh(pre)}[act]
    dya, dyb = rnd(rows, 12, seed=2), rnd(rows, 8, seed=3)
    dx = torch.full((rows, 10), -5.5, device='cuda')
    before = dx.clone()
    L.act_bwd(y.data_ptr(), 8, dya.data_ptr() + 8, 12, dyb.data_ptr() if two else 0, 8, dx.data_ptr() + 4, 10, rows, c, act, 0.2)
    torch.cuda.synchronize()
    g = dya[:, 2:2 + c].double() + (dyb[:, :c].double() if two else 0)
    yd = y[:, :c].double()
    d = {1: (yd > 0).double(), 2: torch.where(yd > 0, torch.ones_like(yd), torch.full_like(yd, 0.2)), 3: yd * (1 - yd),
         4: 1 - yd * yd}[act]
    _rel(dx[:, 1:1 + c], g * d, 1.0, 1e-6, 'act_bwd %d' % act)
    assert torch.equal(dx[:, :1], before[:, :1]) and torch.equal(dx[:, 1 + c:], before[:, 1 + c:])


@pytest.mark.parametrize('n,P,c,xs,os_', [(1, 1000, 45, 48, 45), (3, 257, 32, 32, 40), (2, 77, 100, 104, 128)])
def test_colsum_accumulates(L, n, P, c, xs, os_):
    """out[n*out_stride + c] += scale * sum_p x: positions not a multiple of the block's 256 rows, c not a multiple of 32."""
    x = rnd(n, P, xs, seed=1)
    out = rnd(n, os_, seed=2)
    before = out.clone()
    L.colsum(x.data_ptr(), xs, out, n, P, c, scale=0.7, out_stride=os_)
    torch.cuda.synchronize()
    ref = before[:, :c].double() + 0.7 * x[:, :, :c].double().sum(dim=1)
    sc = float((before[:, :c].double().abs() + 0.7 * x[:, :, :c].double().abs().sum(dim=1)).max())
    _rel(out[:, :c], ref, sc, 2e-6, 'colsum')
    assert torch.equal(out[:, c:], before[:, c:])


def test_avgpool_fwd_bwd(L):
    n, P, c, xs = 3, 300, 200, 204
    x = rnd(n, P, xs, seed=1)
    y = torch.full((n, c), float('nan'), device='cuda')
    L.avgpool(x, xs, y, n, P, c)
    dy = rnd(n, c, seed=2)
    dx = torch.full((n, P, xs), 9.0, device='cuda')
    L.avgpool_bwd(dy, dx, xs, n, P, c)
    torch.cuda.synchronize()
    _rel(y, x[:, :, :c].double().mean(dim=1), float(x[:, :, :c].abs().double().mean(dim=1).max()), 2e-6, 'avgpool')
    _rel(dx[:, :, :c], (dy.double() / P)[:, None, :].expand(n, P, c), float(dy.abs().max()) / P, 1e-6, 'avgpool_bwd')
    assert bool((dx[:, :, c:] == 9.0).all())


@pytest.mark.parametrize('accumulate', [0, 1])
def test_axpy_channels_row_mask(L, accumulate):
    rows, c, rpm = 90, 5, 3
    src = rnd(rows, 8, seed=1)
    dst = rnd(rows, 12, seed=2)
    before = dst.clone()
    mask = (torch.arange(rows // rpm, device='cuda') % 4 == 1).int()
    L.axpy_channels(src.data_ptr() + 4, 8, dst.data_ptr() + 12, 12, rows, c, scale=-1.5, row_mask=mask, rows_per_mask=rpm,
                    accumulate=bool(accumulate))
    torch.cuda.synchronize()
    keep = (mask.repeat_interleave(rpm) == 0).double()[:, None]
    ref = (before[:, 3:3 + c].double() if accumulate else 0) + keep * -1.5 * src[:, 1:1 + c].double()
    _rel(dst[:, 3:3 + c], ref, 1.0, 1e-6, 'axpy')
    assert torch.equal(dst[:, :3], before[:, :3]) and torch.equal(dst[:, 3 + c:], before[:, 3 + c:])


def test_select_broadcast_and_copy_are_bit_exact(L):
    n, per = 5, 36
    sel = torch.tensor([1, 0, 0, 1, 1], dtype=torch.int32, device='cuda')
    a, b = rnd(n, per, seed=1), rnd(n, per, seed=2)
    out = torch.full((n, per), float('nan'), device='cuda')
    L.select_rows(sel, a, b, out, n, per)
    N, P, c = 3, 50, 7
    vec = rnd(N, 10, seed=3)
    dst = torch.full((N, P, 16), -2.0, device='cuda')
    L.broadcast_channels(vec, 10, dst.data_ptr() + 4 * 5, 16, N, P, c)
    src = rnd(N * P, 12, seed=4)
    cp = torch.full((N * P, 20), -3.0, device='cuda')
    L.copy_channels(src.data_ptr() + 4 * 2, 12, cp.data_ptr() + 4 * 9, 20, N * P, c)
    torch.cuda.synchronize()
    assert torch.equal(out, torch.where(sel[:, None].bool(), a, b))
    assert torch.equal(dst[..., 5:5 + c], vec[:, None, :c].expand(N, P, c))
    assert bool((dst[..., :5] == -2).all()) and bool((dst[..., 5 + c:] == -2).all())
    assert torch.equal(cp[:, 9:9 + c], src[:, 2:2 + c])
    assert bool((cp[:, :9] == -3).all()) and bool((cp[:, 9 + c:] == -3).all())


@pytest.mark.parametrize('mode', [1, 2, 3], ids=['l2', 'l1_accumulate', 'l2_accumulate'])
def test_pixel_loss_l2_and_accumulate(L, mode):
    rows, C = 1001, 3
    pred, tgt = torch.rand(rows, 4, device='cuda'), torch.rand(rows, 8, device='cuda')
    out = torch.full((1,), 0.75, device='cuda')
    dp = rnd(rows, 4, seed=1)
    before = dp.clone()
    L.pixel_loss(pred.data_ptr(), 4, tgt.data_ptr(), 8, dp.data_ptr(), 4, rows, C, mode, rows * C, 2.0, out)
    torch.cuda.synchronize()
    pd = pred[:, :C].double().requires_grad_(True)
    ref = (O.l2_loss if mode & 1 else O.l1_loss)(pd, tgt[:, :C].double())
    (g,) = torch.autograd.grad(2.0 * ref, pd)
    _rel(out - 0.75, ref.reshape(1), 1.0, 1e-5, 'pixel loss value')
    want = g + (before[:, :C].double() if mode & 2 else 0)
    _rel(dp[:, :C], want, 1.0, 1e-6, 'pixel loss gradient')
    assert torch.equal(dp[:, C:], before[:, C:])
