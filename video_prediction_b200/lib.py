"""ctypes binding of libvp_b200.so (the C ABI declared in include/vp_b200.h).

There is deliberately NO fallback: if the CUDA library is missing or fails to load, importing the
product path raises.  PyTorch is used only for device memory and streams."""
from __future__ import annotations

import ctypes as C
import os

import torch

from . import build as _build

_LIB = None


class VpTensor(C.Structure):
    _fields_ = [('ptr', C.c_void_p), ('n', C.c_int32), ('d', C.c_int32), ('h', C.c_int32), ('w', C.c_int32),
                ('c', C.c_int32), ('cstride', C.c_int32)]


class VpConvGeom(C.Structure):
    _fields_ = [('kd', C.c_int32), ('kh', C.c_int32), ('kw', C.c_int32),
                ('sd', C.c_int32), ('sh', C.c_int32), ('sw', C.c_int32),
                ('pd', C.c_int32), ('ph', C.c_int32), ('pw', C.c_int32),
                ('transposed', C.c_int32)]


ACT_NONE, ACT_RELU, ACT_LRELU, ACT_SIGMOID, ACT_TANH = range(5)
WKIND_PLAIN, WKIND_POOLED, WKIND_UPSAMPLED = range(3)
WLAYOUT_FWD, WLAYOUT_DGRAD = range(2)
WLAYOUT_RESIDUAL = 4


class VpError(RuntimeError):
    pass


def lib():
    """Loads (building first if the sources are newer) libvp_b200.so.  Raises if unavailable."""
    global _LIB
    if _LIB is None:
        path = _build.LIB_PATH
        if _build.needs_build():       # missing, or older than any source under csrc/ / the header
            path = _build.build()
        _LIB = C.CDLL(path)
        _LIB.vp_last_error.restype = C.c_char_p
    return _LIB


def check(rc):
    if rc != 0:
        raise VpError(lib().vp_last_error().decode())


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def tensor_view(t, c=None, c_off=0):
    """vp_tensor view of a contiguous channels-last torch tensor [N,H,W,C] or [N,D,H,W,C],
    optionally restricted to channels [c_off, c_off + c)."""
    assert t.is_contiguous() and t.dtype == torch.float32
    if t.dim() == 4:
        n, h, w, ct = t.shape
        d = 1
    else:
        n, d, h, w, ct = t.shape
    c = ct - c_off if c is None else c
    v = VpTensor(t.data_ptr() + 4 * c_off, n, d, h, w, c, ct)
    v._owner = t          # keeps the storage alive and lets the autotuner snapshot / restore an output it accumulates into
    return v


def geom(k, s=(1, 1, 1), p=(0, 0, 0), transposed=False):
    return VpConvGeom(k[0], k[1], k[2], s[0], s[1], s[2], p[0], p[1], p[2], int(transposed))


_ENGINE_CHOICE = {}     # geometry signature -> 0 (box) / 1 (halo), measured once per process
_PROFILE = None         # list of (kind, algorithmic flops, start event, end event) while profile_engine(True) is active


_PROFILE_REPLAY = False


def profile_engine(on, by_geometry=False, replay=False):
    """Starts / stops recording every tensor-core engine call (algorithmic FLOPs + GPU time).  Stopping returns
    {'igemm' | 'wgrad': dict(calls, flops, ms)} for the whole-engine roofline of bench.py, or with by_geometry the same sums
    per (kind, geometry key, engine).  Timing: CUDA events around the eager call on its launching stream, which for kernels
    shorter than a launch costs on the host (ctypes + tensor-map encoding, ~25 us) measures the HOST, not the GPU; with
    replay=True every call is additionally captured four times into a CUDA graph and the replay is timed (GPU time only,
    operands L2-warm; calls that accumulate into their output are repeated too, so the step's numbers are garbage)."""
    global _PROFILE, _PROFILE_REPLAY
    if on:
        _PROFILE, _PROFILE_REPLAY = [], bool(replay)
        return None
    rec, _PROFILE = _PROFILE or [], None
    torch.cuda.synchronize()
    out = {}
    for kind, flops, e0, e1, key, reps in rec:
        d = out.setdefault((kind, key) if by_geometry else kind, dict(calls=0, flops=0.0, ms=0.0))
        d['calls'] += 1
        d['flops'] += flops
        d['ms'] += e0.elapsed_time(e1) / reps
    return out


def _conv_flops(x_view, g, out_view):
    """Algorithmic FLOPs of a convolution call as SURVEY.md 8(d) counts them: 2 * output positions * Cout * Cin * taps executed
    per output (a transposed convolution executes taps / stride-product taps per output position)."""
    taps = g.kd * g.kh * g.kw
    if g.transposed:
        taps = taps / float(g.sd * g.sh * g.sw)
    return 2.0 * out_view.n * out_view.d * out_view.h * out_view.w * out_view.c * x_view.c * taps


def _profiled(kind, flops, call, key=None):
    if _PROFILE is None:
        return call()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if _PROFILE_REPLAY and not torch.cuda.is_current_stream_capturing():
        call()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(4):
                call()
        g.replay()
        e0.record()
        g.replay()
        e1.record()
        e1.synchronize()
        _PROFILE.append((kind, flops, e0, e1, key, 4))
        del g
        return
    e0.record()
    call()
    e1.record()
    _PROFILE.append((kind, flops, e0, e1, key, 1))


def _conv_key(x_view, g, n_pad, kc, out_view, act, extra):
    return (x_view.n, x_view.d, x_view.h, x_view.w, x_view.c, out_view.n, out_view.d, out_view.h, out_view.w, out_view.c,
            out_view.c == out_view.cstride, g.kd, g.kh, g.kw, g.sd, g.sh, g.sw, g.pd, g.ph, g.pw, g.transposed, n_pad, kc, act, extra)


def _pick_engine(key, call, idempotent, out_view=None):
    """Both engines compute the same convolution; which one is faster depends on the geometry (plane size, taps per halo
    group, N).  The first call of a geometry times both (CUDA-graph replays) and the winner is cached for the process.
    VP_HALO=0/1 or VP_AUTOTUNE=0 pin the engine.  A call that accumulates into its output is timed on a snapshot: the output
    tensor is cloned before and restored after (possible when the view was made by tensor_view), otherwise it is not timed."""
    choice = _ENGINE_CHOICE.get(key)
    if choice is not None:
        return choice
    owner = getattr(out_view, '_owner', None)
    if os.environ.get('VP_AUTOTUNE', '1') == '0' or 'VP_HALO' in os.environ or torch.cuda.is_current_stream_capturing() or \
            (not idempotent and owner is None):
        return -1
    snapshot = owner.clone() if not idempotent else None
    times = []
    for eng in (0, 1):
        check(lib().vp_conv_set_engine(eng))
        call()                                   # warm-up (function attributes, descriptor cache)
        torch.cuda.synchronize()
        # the kernels are shorter than an eager launch costs on the host (ctypes + tensor-map encoding), so 8 launches are
        # captured into a CUDA graph and the replay is timed: GPU time, not launch rate
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(8):
                call()
        g.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        g.replay()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1) * 3.0 / 16.0)      # keeps the unit of the log: milliseconds per 3 launches
        del g
    check(lib().vp_conv_set_engine(-1))
    if snapshot is not None:
        owner.copy_(snapshot)
    choice = 0 if times[0] <= times[1] else 1
    _ENGINE_CHOICE[key] = choice
    if os.environ.get('VP_AUTOTUNE_LOG'):
        import sys
        sys.stderr.write('[autotune] %s box %.1f us halo %.1f us -> %s\n' % (key, times[0] / 3 * 1e3, times[1] / 3 * 1e3, 'halo' if choice else 'box'))
    return choice


def conv_igemm(x_view, g, wpacked, n_pad, kc, out_view, bias=None, act=ACT_NONE, alpha=0.0, split_k=1, accumulate=0):
    if 'igemm' in _SKIP:
        return

    def call():
        check(lib().vp_conv_igemm(C.byref(x_view), C.byref(g), ptr(wpacked), n_pad, kc, C.byref(out_view), ptr(bias),
                                  act, C.c_float(alpha), split_k, int(accumulate), stream_ptr()))
    # an explicit split_k > 1 adds atomically into a caller-cleared output: repeating the call (timing) would change it
    key = _conv_key(x_view, g, n_pad, kc, out_view, act, ('fwd', split_k))
    eng = _pick_engine(key, call, not accumulate and split_k <= 1, out_view if split_k <= 1 else None)
    check(lib().vp_conv_set_engine(eng))
    _profiled('igemm', _conv_flops(x_view, g, out_view), call, (key, eng))
    if eng >= 0:
        check(lib().vp_conv_set_engine(-1))


def conv_igemm_actgrad(x_view, g, wpacked, n_pad, kc, out_view, act_output_addr, addend_addr, act, alpha=0.0, accumulate=0):
    if 'igemm' in _SKIP:
        return

    def call():
        check(lib().vp_conv_igemm_actgrad(C.byref(x_view), C.byref(g), ptr(wpacked), n_pad, kc, C.byref(out_view),
                                          C.c_void_p(act_output_addr), C.c_void_p(addend_addr or 0), act, C.c_float(alpha),
                                          int(accumulate), stream_ptr()))
    key = _conv_key(x_view, g, n_pad, kc, out_view, act, ('actgrad', bool(addend_addr)))
    eng = _pick_engine(key, call, not accumulate, out_view)
    check(lib().vp_conv_set_engine(eng))
    _profiled('igemm', _conv_flops(x_view, g, out_view), call, (key, eng))
    if eng >= 0:
        check(lib().vp_conv_set_engine(-1))


KERNEL_BOX, KERNEL_HALO, KERNEL_WGRAD_TAPS, KERNEL_WGRAD_ROWS = range(4)


def last_launch():
    """(kernel, splits) of this thread's last engine launch: kernel is one of the KERNEL_* codes (-1 before any launch)."""
    info = (C.c_int * 2)()
    check(lib().vp_conv_last_launch(info))
    return info[0], info[1]


def tf32_residual(x):
    """x - tf32_truncate(x) with the layout of x (the 'lo' operand of the fp32-exact 3xTF32 mode)."""
    assert x.is_contiguous() and x.dtype == torch.float32
    lo = torch.empty_like(x)
    check(lib().vp_tf32_residual(ptr(x), ptr(lo), C.c_longlong(x.numel()), stream_ptr()))
    return lo


def exact_mode():
    """VP_EXACT=1: every tensor-core convolution (forward, dgrad, wgrad) runs as three TF32 passes
    hi*hi + lo*hi + hi*lo with fp32 accumulation = fp32-exact up to 2^-21 (debug / parity mode, ~3x the conv time)."""
    return os.environ.get('VP_EXACT', '0') == '1'


def conv_wgrad(x_view, dy_view, g, dwpacked, n_pad, kc, split_k=1):
    if 'wgrad' in _SKIP:
        return
    taps = g.kd * g.kh * g.kw / (float(g.sd * g.sh * g.sw) if g.transposed else 1.0)
    flops = 2.0 * dy_view.n * dy_view.d * dy_view.h * dy_view.w * dy_view.c * x_view.c * taps
    _profiled('wgrad', flops, lambda: check(lib().vp_conv_wgrad(C.byref(x_view), C.byref(dy_view), C.byref(g), ptr(dwpacked), n_pad, kc,
                                                               split_k, stream_ptr())),
              (_conv_key(x_view, g, n_pad, kc, dy_view, 0, ('wgrad', split_k)), -1))


def eff_taps(k, kind):
    if kind == WKIND_POOLED:
        return (k[1] + 1) * (k[2] + 1)
    if kind == WKIND_UPSAMPLED:
        return (k[1] + 3) * (k[2] + 3)
    return k[0] * k[1] * k[2]


def pad_to(v, m):
    return (v + m - 1) // m * m


def choose_n_pad(rows):
    """GEMM-N padding: multiple of 16; above 256 either a multiple of 128 (128-wide tiles) or the fewest equal tiles."""
    n = pad_to(rows, 16)
    if n <= 256 or n % 128 == 0:
        return n
    tiles = -(-n // 256)
    bn = pad_to(-(-rows // tiles), 16)
    return tiles * bn


def pack_weights(w, k, ci_ref, co, kind, layout, ci_int=None, cmap=None, inv_scale=None, out=None):
    """Returns (wpacked, n_pad, kc)."""
    ci_int = ci_ref if ci_int is None else ci_int
    rows, cols = (co, ci_int) if (layout & 3) == WLAYOUT_FWD else (ci_int, co)
    n_pad, kc = choose_n_pad(rows), pad_to(cols, 32) // 32
    taps = eff_taps(k, kind)
    if out is None:
        out = torch.empty(taps * n_pad * kc * 32, device=w.device, dtype=torch.float32)
    elif 'pack' in _SKIP:
        return out, n_pad, kc
    check(lib().vp_pack_weights(ptr(w), k[0], k[1], k[2], ci_ref, co, kind, layout, ptr(cmap), ci_int,
                                ptr(inv_scale), ptr(out), n_pad, kc, stream_ptr()))
    return out, n_pad, kc


class PackJob(C.Structure):
    """vp_pack_job (include/vp_b200.h)."""
    _fields_ = [('w', C.c_void_p), ('wpacked', C.c_void_p), ('cmap', C.c_void_p), ('inv_scale', C.c_void_p),
                ('kd', C.c_int), ('kh', C.c_int), ('kw', C.c_int), ('ci_ref', C.c_int), ('co', C.c_int), ('kind', C.c_int),
                ('layout', C.c_int), ('ci_int', C.c_int), ('n_pad', C.c_int), ('kc', C.c_int), ('block_begin', C.c_int),
                ('reserved', C.c_int)]


class PackPlan(object):
    """A fixed set of weight tensors repacked by ONE launch (vp_pack_weights_batch).  Every entry is the argument list of a
    pack_weights call whose output buffer already exists: (w, k, ci_ref, co, kind, layout, ci_int, cmap, inv_scale, out)."""

    def __init__(self, entries):
        import numpy as np
        jobs = (PackJob * len(entries))()
        blocks = 0
        self.keep = entries                                   # the table holds raw pointers: keep the tensors alive
        for j, (w, k, ci_ref, co, kind, layout, ci_int, cmap, inv_scale, out) in zip(jobs, entries):
            ci_int = ci_ref if ci_int is None else ci_int
            rows, cols = (co, ci_int) if (layout & 3) == WLAYOUT_FWD else (ci_int, co)
            n_pad, kc = choose_n_pad(rows), pad_to(cols, 32) // 32
            total = eff_taps(k, kind) * n_pad * kc * 32
            assert out.numel() == total and w.is_contiguous()
            j.w, j.wpacked = w.data_ptr(), out.data_ptr()
            j.cmap = cmap.data_ptr() if cmap is not None else None
            j.inv_scale = inv_scale.data_ptr() if inv_scale is not None else None
            j.kd, j.kh, j.kw, j.ci_ref, j.co, j.kind, j.layout, j.ci_int = k[0], k[1], k[2], ci_ref, co, kind, layout, ci_int
            j.n_pad, j.kc, j.block_begin = n_pad, kc, blocks
            blocks += -(-total // 256)
        self.njobs, self.blocks = len(entries), blocks
        raw = np.frombuffer(bytes(jobs), dtype=np.uint8).copy()
        self.table = torch.from_numpy(raw).to(entries[0][0].device)

    def run(self):
        if 'pack' in _SKIP:
            return
        check(lib().vp_pack_weights_batch(ptr(self.table), self.njobs, self.blocks, stream_ptr()))


def unpack_wgrad(dwpacked, k, ci_ref, co, kind, dw, n_pad, kc, ci_int=None, cmap=None):
    if 'pack' in _SKIP:
        return
    ci_int = ci_ref if ci_int is None else ci_int
    check(lib().vp_unpack_wgrad(ptr(dwpacked), k[0], k[1], k[2], ci_ref, co, kind, ptr(cmap), ci_int, ptr(dw),
                                n_pad, kc, stream_ptr()))


# ---------------------------------------------------------------------------------- HBM-bound kernels
def _f(v):
    return C.c_float(v)


_SKIP = set(filter(None, os.environ.get('VP_SKIP', '').split(',')))   # timing ablations only (wrong results): kernel families not launched


def inorm_act(x_addr, x_cs, y_addr, y_cs, n, positions, c, gamma, beta, act=ACT_NONE, alpha=0.0, stats=None, eps=1e-6):
    if 'inorm' in _SKIP:
        return
    check(lib().vp_inorm_act(C.c_void_p(x_addr), x_cs, C.c_void_p(y_addr), y_cs, n, positions, c, ptr(gamma), ptr(beta), _f(eps), act, _f(alpha),
                             ptr(stats), stream_ptr()))


def lstm_gates_fwd(pre, n, positions, filters, c_prev, g1, b1, g2, b2, c_new, h_dsts, stats1=None, stats2=None,
                   forget_bias=1.0, eps=1e-6):
    if 'gates' in _SKIP:
        return
    """h_dsts: list of (address:int, cstride:int)."""
    k = len(h_dsts)
    pa = (C.c_void_p * k)(*[C.c_void_p(a) for a, _ in h_dsts])
    sa = (C.c_int * k)(*[s for _, s in h_dsts])
    check(lib().vp_lstm_gates_fwd(ptr(pre), n, positions, filters, ptr(c_prev), ptr(g1), ptr(b1), ptr(g2), ptr(b2),
                                  _f(forget_bias), _f(eps), ptr(c_new), pa, sa, k, ptr(stats1), ptr(stats2),
                                  stream_ptr()))


def broadcast_channels(vec, vec_stride, dst_addr, dst_cs, n, positions, c):
    check(lib().vp_broadcast_channels(ptr(vec), vec_stride, C.c_void_p(dst_addr), dst_cs, n, positions, c, stream_ptr()))


def copy_channels(src_addr, src_cs, dst_addr, dst_cs, rows, c):
    if 'copy' in _SKIP:
        return
    check(lib().vp_copy_channels(C.c_void_p(src_addr), src_cs, C.c_void_p(dst_addr), dst_cs, C.c_longlong(rows), c,
                                 stream_ptr()))


def select_rows(sel, a, b, out, n, per_row):
    check(lib().vp_select_rows(ptr(sel), ptr(a), ptr(b), ptr(out), n, C.c_longlong(per_row), stream_ptr()))


def avgpool(x, x_cs, y, n, positions, c):
    check(lib().vp_avgpool(ptr(x), x_cs, ptr(y), n, positions, c, stream_ptr()))


def dense_fwd(x, x_stride, w, bias, y, y_stride, b, k, j, k_splits=1, inv_scale=None):
    if 'dense' in _SKIP:
        return
    check(lib().vp_dense_fwd(ptr(x), x_stride, ptr(w), ptr(bias), ptr(inv_scale), ptr(y), y_stride, b, k, j, k_splits,
                             stream_ptr()))


def lstm_cell_fwd(gates, c_prev, c_new, h_new, b, units, forget_bias=1.0):
    check(lib().vp_lstm_cell_fwd(ptr(gates), ptr(c_prev), ptr(c_new), ptr(h_new), b, units, _f(forget_bias), stream_ptr()))


def sample_z(mu, lss, eps, z, total):
    check(lib().vp_sample_z(ptr(mu), ptr(lss), ptr(eps), ptr(z), total, stream_ptr()))


def cdna_kernel_norm(raw, out, b, kh, kw, nk):
    check(lib().vp_cdna_kernel_norm(ptr(raw), ptr(out), b, kh, kw, nk, stream_ptr()))


def cdna_apply(image, first, kernels, layers_addr, layers_cs, n, h, w, kh, kw, nk):
    if 'cdna' in _SKIP:
        return
    check(lib().vp_cdna_apply(ptr(image), ptr(first), ptr(kernels), C.c_void_p(layers_addr), layers_cs, n, h, w, kh, kw, nk,
                              stream_ptr()))


def flow_apply(image, first, flows, flows_cs, layers_addr, layers_cs, n, h, w, nk):
    check(lib().vp_flow_apply(ptr(image), ptr(first), ptr(flows), flows_cs, C.c_void_p(layers_addr), layers_cs, n, h, w, nk, stream_ptr()))


def flow_apply_bwd(image, flows, flows_cs, da_addr, da_cs, db_addr, db_cs, dimage, dflows, n, h, w, nk):
    check(lib().vp_flow_apply_bwd(ptr(image), ptr(flows), flows_cs, C.c_void_p(da_addr), da_cs, C.c_void_p(db_addr), db_cs, ptr(dimage),
                                  ptr(dflows), n, h, w, nk, stream_ptr()))


def composite(logits, logits_cs, layers_addr, layers_cs, masks, masks_cs, gen, positions, num_layers):
    if 'cdna' in _SKIP:
        return
    check(lib().vp_composite(ptr(logits), logits_cs, C.c_void_p(layers_addr), layers_cs, ptr(masks), masks_cs, ptr(gen),
                             C.c_longlong(positions), num_layers, stream_ptr()))


# ---------------------------------------------------------------------------------- backward / losses / optimizer
def _srcs(srcs):
    """srcs: list of (address:int, cstride:int) gradient sources to be summed."""
    k = len(srcs)
    return (C.c_void_p * k)(*[C.c_void_p(a) for a, _ in srcs]), (C.c_int * k)(*[s for _, s in srcs]), k


def addr(a):
    return C.c_void_p(a)


def inorm_act_bwd(x_addr, x_cs, dy_srcs, dx_addr, dx_cs, n, positions, c, gamma, beta, stats, act, alpha, dgamma, dbeta):
    if 'inorm' in _SKIP:
        return
    pa, sa, k = _srcs(dy_srcs)
    check(lib().vp_inorm_act_bwd(addr(x_addr), x_cs, pa, sa, k, addr(dx_addr), dx_cs, n, positions, c, ptr(gamma), ptr(beta),
                                 ptr(stats), act, _f(alpha), ptr(dgamma), ptr(dbeta), stream_ptr()))


def lstm_gates_bwd(pre, n, positions, filters, c_prev, g1, b1, g2, b2, stats1, stats2, dh_srcs, dc_next, dpre, dc_prev,
                   dg1, db1, dg2, db2, forget_bias=1.0):
    if 'gates' in _SKIP:
        return
    pa, sa, k = _srcs(dh_srcs)
    check(lib().vp_lstm_gates_bwd(ptr(pre), n, positions, filters, ptr(c_prev), ptr(g1), ptr(b1), ptr(g2), ptr(b2), ptr(stats1),
                                  ptr(stats2), _f(forget_bias), pa, sa, k, ptr(dc_next), ptr(dpre), ptr(dc_prev), ptr(dg1),
                                  ptr(db1), ptr(dg2), ptr(db2), stream_ptr()))


def composite_bwd(dgen, masks, masks_cs, layers_addr, layers_cs, dlogits, dlogits_cs, dlayers, dlayers_cs, positions, num_layers):
    if 'cdna' in _SKIP:
        return
    check(lib().vp_composite_bwd(ptr(dgen), ptr(masks), masks_cs, addr(layers_addr), layers_cs, ptr(dlogits), dlogits_cs,
                                 ptr(dlayers), dlayers_cs, C.c_longlong(positions), num_layers, stream_ptr()))


def cdna_apply_bwd(image, kernels, da_addr, da_cs, db_addr, db_cs, dimage, dkernels, n, h, w, kh, kw, nk):
    if 'cdna' in _SKIP:
        return
    check(lib().vp_cdna_apply_bwd(ptr(image), ptr(kernels), addr(da_addr), da_cs, addr(db_addr), db_cs, ptr(dimage), ptr(dkernels),
                                  n, h, w, kh, kw, nk, stream_ptr()))


def cdna_kernel_norm_bwd(raw, out, dout, draw, b, kh, kw, nk):
    check(lib().vp_cdna_kernel_norm_bwd(ptr(raw), ptr(out), ptr(dout), ptr(draw), b, kh, kw, nk, stream_ptr()))


def dense_bwd(x, x_stride, w, dy, dy_stride, b, k, j, dx=None, dx_stride=0, dx_accumulate=False, dw=None, dbias=None,
              inv_scale=None):
    if 'dense' in _SKIP:
        return
    check(lib().vp_dense_bwd(ptr(x), x_stride, ptr(w), ptr(inv_scale), ptr(dy), dy_stride, ptr(dx), dx_stride,
                             int(dx_accumulate), ptr(dw), ptr(dbias), b, k, j, stream_ptr()))


def lstm_cell_bwd(gates, c_prev, c_new, dh, dc_next, dgates, dc_prev, b, units, forget_bias=1.0):
    check(lib().vp_lstm_cell_bwd(ptr(gates), ptr(c_prev), ptr(c_new), ptr(dh), ptr(dc_next), ptr(dgates), ptr(dc_prev), b, units,
                                 _f(forget_bias), stream_ptr()))


def colsum(x_addr, x_cs, out, n, positions, c, scale=1.0, out_stride=None):
    if 'colsum' in _SKIP:
        return
    check(lib().vp_colsum(addr(x_addr), x_cs, ptr(out), c if out_stride is None else out_stride, n, C.c_longlong(positions), c,
                          _f(scale), stream_ptr()))


def axpy_channels(src_addr, src_cs, dst_addr, dst_cs, rows, c, scale=1.0, row_mask=None, rows_per_mask=1, accumulate=True):
    check(lib().vp_axpy_channels(addr(src_addr), src_cs, addr(dst_addr), dst_cs, C.c_longlong(rows), c, _f(scale), ptr(row_mask),
                                 C.c_longlong(rows_per_mask), int(accumulate), stream_ptr()))


def act_bwd(y_addr, y_cs, dya_addr, dya_cs, dyb_addr, dyb_cs, dx_addr, dx_cs, rows, c, act, alpha=0.0):
    check(lib().vp_act_bwd(addr(y_addr), y_cs, addr(dya_addr), dya_cs, addr(dyb_addr or 0), dyb_cs, addr(dx_addr), dx_cs,
                           C.c_longlong(rows), c, act, _f(alpha), stream_ptr()))


def avgpool_bwd(dy, dx, dx_cs, n, positions, c):
    check(lib().vp_avgpool_bwd(ptr(dy), ptr(dx), dx_cs, n, positions, c, stream_ptr()))


def sample_z_bwd(mu, lss, eps, dz, dmu, dlss, total, kl_scale_dev):
    check(lib().vp_sample_z_bwd(ptr(mu), ptr(lss), ptr(eps), ptr(dz), ptr(dmu), ptr(dlss), total, ptr(kl_scale_dev), stream_ptr()))


def pixel_loss(pred_addr, pred_cs, target_addr, target_cs, dpred_addr, dpred_cs, rows, c, mode, mean_count, grad_scale, out):
    check(lib().vp_pixel_loss(addr(pred_addr), pred_cs, addr(target_addr), target_cs, addr(dpred_addr or 0), dpred_cs,
                              C.c_longlong(rows), c, mode, C.c_longlong(mean_count), _f(grad_scale), ptr(out), stream_ptr()))


GAN_KINDS = {'LSGAN': 0, 'GAN': 1, 'SNGAN': 2}


def gan_loss(logits, label, n, grad_scale, kind, dlogits, out):
    check(lib().vp_gan_loss(ptr(logits), _f(label), n, _f(grad_scale), GAN_KINDS[kind], ptr(dlogits), ptr(out), stream_ptr()))


def kl_loss(mu, lss, rows, nz, out):
    check(lib().vp_kl_loss(ptr(mu), ptr(lss), rows, nz, ptr(out), stream_ptr()))


def cosine_distance(a, b, da, rows, c, grad_scale, out):
    if 'cosd' in _SKIP:
        return
    check(lib().vp_cosine_distance(ptr(a), ptr(b), ptr(da), C.c_longlong(rows), c, _f(grad_scale), ptr(out), stream_ptr()))


def adam(p, g, m, v, n, lr_t_dev, beta1, beta2, grad_scale=1.0, eps=1e-8):
    if 'adam' in _SKIP:
        return
    check(lib().vp_adam(ptr(p), ptr(g), ptr(m), ptr(v), C.c_longlong(n), ptr(lr_t_dev), _f(beta1), _f(beta2), _f(eps),
                        _f(grad_scale), stream_ptr()))


def launch_count():
    f = lib().vp_launch_count
    f.restype = C.c_longlong
    return int(f())


def spectral_norm_fwd(w, u, rows, cols, v, s, u_new, scal):
    if 'sn' in _SKIP:
        return
    check(lib().vp_spectral_norm_fwd(ptr(w), ptr(u), rows, cols, ptr(v), ptr(s), ptr(u_new), ptr(scal), stream_ptr()))


def spectral_norm_bwd(w, u, g_wbar, rows, cols, v, s, scal, gs, gt, dw):
    if 'sn' in _SKIP:
        return
    check(lib().vp_spectral_norm_bwd(ptr(w), ptr(u), ptr(g_wbar), rows, cols, ptr(v), ptr(s), ptr(scal), ptr(gs), ptr(gt), ptr(dw),
                                     stream_ptr()))


def gather_clip(video, t_start, clip, clips, clip_len, pixels, video_batch, batch_offset):
    check(lib().vp_gather_clip(ptr(video), ptr(t_start), ptr(clip), clips, clip_len, C.c_longlong(pixels), video_batch,
                               batch_offset, stream_ptr()))


def scatter_clip(dclip, t_start, dvideo, clips, clip_len, pixels, video_batch, batch_offset):
    check(lib().vp_scatter_clip(ptr(dclip), ptr(t_start), ptr(dvideo), clips, clip_len, C.c_longlong(pixels), video_batch,
                                batch_offset, stream_ptr()))


def conv3d_c4_fwd(x, w, inv_scale, bias, out, n, d, h, wd, ci, alpha):
    if 'c4fwd' in _SKIP:
        return
    check(lib().vp_conv3d_c4_fwd(ptr(x), ptr(w), ptr(inv_scale), ptr(bias), ptr(out), n, d, h, wd, ci, _f(alpha), stream_ptr()))


def conv3d_c4_fwd_tc_ok(h, wd):
    """Shapes vp_conv3d_c4_fwd_tc tiles: L in {16, 8, 4} lines with h % L == 0 and three (L+2) x (wd+2) float4 planes <= 90 KB."""
    return wd + 2 <= 256 and any(h % L == 0 and 3 * (L + 2) * (wd + 2) * 16 <= 90 * 1024 for L in (16, 8, 4))


def conv3d_c4_fwd_tc(x, w, inv_scale, bias, out, n, d, h, wd, ci, alpha):
    if 'c4fwd' in _SKIP:
        return
    check(lib().vp_conv3d_c4_fwd_tc(ptr(x), ptr(w), ptr(inv_scale), ptr(bias), ptr(out), n, d, h, wd, ci, _f(alpha), stream_ptr()))


def conv3d_c4_wgrad(x, dy, gw, n, d, h, wd, ci):
    if 'c4wgrad' in _SKIP:
        return
    # tensor cores unless the fp32-exact mode is on (the CUDA-core kernel is exact) or the width does not tile by 64
    if wd % 64 == 0 and not exact_mode() and os.environ.get('VP_D0_WGRAD_CUDA_CORE', '0') != '1':
        check(lib().vp_conv3d_c4_wgrad_tc(ptr(x), ptr(dy), ptr(gw), n, d, h, wd, ci, stream_ptr()))
        return
    check(lib().vp_conv3d_c4_wgrad(ptr(x), ptr(dy), ptr(gw), n, d, h, wd, ci, stream_ptr()))


def image_warp_fwd(im, im_cs, flow, out, out_cs, n, h, w, c):
    check(lib().vp_image_warp_fwd(ptr(im), im_cs, ptr(flow), ptr(out), out_cs, n, h, w, c, stream_ptr()))


def image_warp_bwd(im, im_cs, flow, dout, dout_cs, dim, dim_cs, dflow, n, h, w, c):
    check(lib().vp_image_warp_bwd(ptr(im), im_cs, ptr(flow), ptr(dout), dout_cs, ptr(dim), dim_cs, ptr(dflow), n, h, w, c, stream_ptr()))
