"""GPU parity tests (-m gpu) of the TRAINING step and of the full-length BASELINE configurations against the CPU oracle
in plain fp32 (the reference's arithmetic), in the two arithmetic modes of the CUDA path:

  * product mode: TF32 tensor-core operands (activations truncated by tcgen05, weights rounded when packed), fp32
    accumulation.  Generator outputs 1e-3 max-abs (BASELINE.json north_star); model-level gradients 5e-2 relative L2 per
    tensor (operand rounding through an 11-step BPTT and a 7-layer discriminator is 1-3 % on the largest tensors).
  * fp32-exact mode (VP_EXACT=1): every tensor-core convolution as three TF32 passes hi*hi + lo*hi + hi*lo.  Here every
    gradient tensor must agree to 2e-3 relative L2 (the fp32-vs-fp64 noise floor of the ORACLE ITSELF is 7e-4 on these
    tensors): kernel selection, split-K, time-batched weight gradients, fused epilogues, the BPTT schedule -- everything
    except operand rounding -- is held to fp32 noise.  This is what separates rounding from a bug.

Why not an oracle with TF32-quantised operands for the model-level gradients?  It exists (`O.set_tf32_emulation`, used by the
op-level tests in test_gpu_kernels.py at 1e-5) but operand truncation is discontinuous: fp32 summation-order noise upstream
flips quantisation decisions downstream, so two correct TF32 implementations differ by 0.5-1.5 % on these gradients
(measured: the emulating oracle with fp32 vs fp64 accumulation, profiles/r02_parity_noise_floor.md).
"""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import savp_oracle as O

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), 'golden')
sys.path.insert(0, GOLD)


@pytest.fixture(scope='module')
def Model():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from video_prediction_b200.models import get_model_class
    return get_model_class('savp')


_MODE = {}


def tf32_mode():
    """Which quantisation the tensor cores apply to fp32 operands of kind::tf32: measured, not assumed."""
    if 'mode' in _MODE:
        return _MODE['mode']
    from video_prediction_b200 import lib as L
    g = torch.Generator().manual_seed(0)
    x = (torch.rand(2, 8, 16, 32, generator=g) + 0.5).cuda()
    w = (torch.rand(1, 1, 32, 16, generator=g) + 0.5).cuda()
    wp, n_pad, kc = L.pack_weights(w.contiguous(), (1, 1, 1), 32, 16, L.WKIND_PLAIN, L.WLAYOUT_FWD)
    out = torch.zeros(2, 8, 16, 16, device='cuda')
    L.conv_igemm(L.tensor_view(x, 32), L.geom((1, 1, 1)), wp, n_pad, kc, L.tensor_view(out, 16))
    torch.cuda.synchronize()
    errs = {}
    for mode in ('trunc', 'rna'):
        # weights are rounded (rna) when they are packed (csrc/pack.cu); activations are read raw by the tensor core
        xq, wq = O.tf32_quantize(x.cpu(), mode).double(), O.tf32_quantize(w.cpu(), 'rna').double()
        ref = (xq.reshape(-1, 32) @ wq.reshape(32, 16)).reshape(2, 8, 16, 16)
        errs[mode] = (out.cpu().double() - ref).abs().max().item()
    best = min(errs, key=errs.get)
    other = 'rna' if best == 'trunc' else 'trunc'
    assert errs[best] < 2e-5 and errs[other] > 10 * errs[best], errs     # all-positive operands: the two modes differ by ~5e-4 relative
    _MODE['mode'], _MODE['errs'] = best, errs
    return best


def test_tensor_core_operand_quantisation_is_identified():
    mode = tf32_mode()
    print('tcgen05 kind::tf32 operand quantisation:', mode, _MODE['errs'])
    assert mode in ('trunc', 'rna')


def _rel(a, b):
    a, b = a.detach().double().reshape(-1).cpu(), b.detach().double().reshape(-1).cpu()
    return ((a - b).norm() / (b.norm() + 1e-300)).item(), b.norm().item()


def _exempt(model):
    """Layers the CUDA path runs on fp32 CUDA cores would stay exact in the emulating oracle; since round 2 every
    convolution's forward / dgrad is on the TF32 engine (only the first discriminator layer's weight gradient is fp32)."""
    return ()


def _oracle_step(hp, params, inputs, noise, step, sampling, mode, exempt):
    O.set_tf32_emulation(mode, exempt)
    try:
        opt = dict(m={k: torch.zeros_like(v) for k, v in params.items()}, v={k: torch.zeros_like(v) for k, v in params.items()}, t=0)
        return O.train_step(params, opt, hp, inputs, noise, step=step, sampling=sampling)
    finally:
        O.set_tf32_emulation(None)


def _gpu_step(Model, hk, params, inputs, noise, step, sampling, A=0):
    model = Model(mode='train', hparams_dict=hk)
    model.set_params(params)
    binp = {'images': inputs['images'].permute(1, 0, 2, 3, 4)}
    if A:
        binp['actions'] = inputs['actions'].permute(1, 0, 2)
    model.build_graph(binp)
    model.global_step = step
    samp = sampling if sampling is not None else torch.zeros(model.S - model.hparams.context_frames, model.B, dtype=torch.bool)
    model.train_step(binp, noise, sampling=samp)
    torch.cuda.synchronize()
    return model


def _check_grads(model, res, tol, floor, what):
    worst = []
    for kind in ('g_grads', 'd_grads'):
        if kind not in res:
            continue
        items = [(k, g) for k, g in res[kind].items() if g is not None]
        gmax = max(g.double().norm().item() for _, g in items)
        for k, g in items:
            r, n = _rel(model.grads[k], g)
            if n < floor * gmax:
                continue        # e.g. conv biases in front of an instance norm: exactly zero in exact arithmetic
            worst.append((r, k, n))
    worst.sort(reverse=True)
    print('%s: worst relative L2 gradient errors: %s' % (what, ['%.2e %s' % (r, k.split('/', 1)[1]) for r, k, _ in worst[:4]]))
    bad = [(r, k) for r, k, _ in worst if r > tol]
    assert not bad, (what, bad[:5])
    return worst


CASES = {
    'deterministic_l1': dict(context_frames=2, sequence_length=12, nz=0, l1_weight=1.0, lr=1e-3),
    'vae_l1': dict(context_frames=2, sequence_length=12, nz=8, l1_weight=1.0, kl_weight=1e-3, kl_anneal_steps=(0, 10), lr=1e-3),
    'savp': dict(context_frames=2, sequence_length=12, lr=2e-4, beta1=0.5, l1_weight=100., kl_weight=1.0,
                 video_sn_vae_gan_weight=0.1, video_sn_gan_weight=0.1, vae_gan_feature_cdist_weight=10.0, kl_anneal_steps=(0, 10)),
    # transformation='flow' (savp_model.py:522-530, flow_ops.image_warp) instead of CDNA kernels
    'vae_flow': dict(context_frames=2, sequence_length=8, nz=8, l1_weight=1.0, kl_weight=1e-3, kl_anneal_steps=(0, 10), lr=1e-3,
                     transformation='flow'),
    # image_sn discriminators (networks.py:35-69; one sampled frame per video) next to a video_sn one whose encoder/ copy gets
    # no loss (video_sn_vae_gan_weight = 0), both feature-matching terms
    'image_video_gan': dict(context_frames=2, sequence_length=8, clip_length=6, lr=2e-4, beta1=0.5, l1_weight=100., kl_weight=1.0,
                            image_sn_gan_weight=0.1, image_sn_vae_gan_weight=0.1, video_sn_gan_weight=0.1,
                            vae_gan_feature_cdist_weight=10.0, gan_feature_cdist_weight=1.0, kl_anneal_steps=(0, 10)),
    'savp_gan_l2': dict(context_frames=2, sequence_length=8, clip_length=6, lr=2e-4, beta1=0.5, l1_weight=10., l2_weight=5.0,
                        kl_weight=1.0, video_sn_vae_gan_weight=0.1, video_sn_gan_weight=0.1, gan_feature_cdist_weight=1.0,
                        gan_loss_type='GAN', kl_anneal_steps=(0, 10)),
}
# arithmetic mode -> (env VP_EXACT, loss rtol, ignore gradient tensors below this fraction of the largest, output atol)
MODES = {'tf32': ('0', 1e-2, 1e-3, 1e-3), 'exact': ('1', 2e-3, 1e-4, 1e-4)}   # (post-update D features follow +-lr Adam steps)
# fp32-exact mode: relative-L2 bound per gradient tensor.  Generator-only cases: 2e-3 (3x the oracle's own fp32-vs-fp64 noise).
# With the discriminators the gradient is a near-cancellation of the real and the fake clip's contributions and the tensor
# core's fp32 accumulator is ~10x less accurate than a CPU fp32 convolution (profiles/r02_exact_mode_accumulator.log: error
# proportional to K, 1.4e-5 at K = 6400): 1e-2 for the shipped LSGAN configuration (measured 4.7e-3 ... 7.5e-3 depending on the
# engines' summation order; 3.3e-3 at B=16).  'savp_gan_l2' starts with logits ~ 0
# under the sigmoid-CE loss, where the real/fake terms cancel to 1 % (the CPU fp32 oracle itself is 5e-3 from fp64 there).
EXACT_GTOL = {'deterministic_l1': 2e-3, 'vae_l1': 2e-3, 'vae_flow': 3e-3, 'savp': 1e-2, 'image_video_gan': 1e-2, 'savp_gan_l2': 5e-2}


class arithmetic(object):
    def __init__(self, mode):
        self.v = MODES[mode][0]

    def __enter__(self):
        self.old = os.environ.get('VP_EXACT')
        os.environ['VP_EXACT'] = self.v

    def __exit__(self, *a):
        if self.old is None:
            os.environ.pop('VP_EXACT', None)
        else:
            os.environ['VP_EXACT'] = self.old


@pytest.mark.parametrize('mode', ['tf32', 'exact'])
@pytest.mark.parametrize('case', sorted(CASES))
def test_training_step_matches_fp32_oracle(Model, case, mode):
    """The three cases of tests/gpu_probe_train.py (deterministic / VAE / SAVP) + one with the GAN (sigmoid-CE) loss, l1 AND
    l2 and the non-VAE feature term, at B=2 with a random scheduled-sampling mask, in both arithmetic modes."""
    hk = CASES[case]
    hp = O.make_hparams(**hk)
    B, step, shape = 2, 5, (64, 64, 3)
    params, _ = O.init_params(hp, shape, seed=0)
    if hk.get('transformation') == 'flow':
        # freshly initialised flows are ~0, right on the floor() discontinuity of image_warp's gradient: move them to
        # non-integer displacements (x flows 0.37, 1.27, -0.53, 2.17; y flows 0.61, ...) so that rounding cannot flip cells
        k = 'generator/rnn/savp_cell/flows/conv2d/bias'
        params[k] = torch.tensor([0.37, 1.27, -0.53, 2.17, 0.61, -1.43, 0.29, 1.71])
    inputs, noise = O.make_synthetic_inputs(hp, B, shape)
    g = torch.Generator().manual_seed(7)
    sampling = torch.rand(hp.sequence_length - 1 - hp.context_frames, B, generator=g) < 0.5
    _, ltol, floor, otol = MODES[mode]
    with arithmetic(mode):
        model = _gpu_step(Model, hk, params, inputs, noise, step, sampling)
    lv = model.losses()
    res = _oracle_step(hp, params, inputs, noise, step, sampling, None, ())
    ref_l = dict(res['g_losses'])
    ref_l.update(res.get('d_losses', {}))
    for k, v in ref_l.items():
        assert abs(lv[k] - v) <= ltol * abs(v) + 1e-6, (k, lv[k], v)
    # the totals the reference exposes (base_model.py:461): sum(loss * weight)
    assert abs(model.g_loss - res['g_loss']) <= ltol * abs(res['g_loss']) + 1e-6, (model.g_loss, res['g_loss'])
    if 'd_loss' in res:
        assert abs(model.d_loss - res['d_loss']) <= ltol * abs(res['d_loss']) + 1e-6
    if mode == 'exact':
        _check_grads(model, res, EXACT_GTOL[case], floor, '%s [exact] vs fp32 oracle' % case)
    else:
        # product mode: the deviation from the fp32 oracle must be what TF32 OPERAND ROUNDING explains -- per tensor at most
        # max(5e-2, 2 x the error of the CPU oracle run with the same operand quantisation (activations truncated,
        # weights rounded, fp32 accumulation; `O.set_tf32_emulation`)).  Measured on the SAVP cases the two agree to ~5 %.
        emu = _oracle_step(hp, params, inputs, noise, step, sampling, tf32_mode(), _exempt(model))
        worst, bad = [], []
        for kind in ('g_grads', 'd_grads'):
            if kind not in res:
                continue
            items = [(k, g) for k, g in res[kind].items() if g is not None]
            gmax = max(g.double().norm().item() for _, g in items)
            for k, g in items:
                r, n = _rel(model.grads[k], g)
                if n < floor * gmax:
                    continue
                e, _ = _rel(emu[kind][k], g)
                worst.append((r, e, k))
                if r > max(5e-2, 2.0 * e):
                    bad.append((r, e, k))
        worst.sort(reverse=True)
        print('%s [tf32]: worst gradient errors (CUDA path | operand-rounding emulation on the CPU): %s'
              % (case, ['%.2e | %.2e %s' % (r, e, k.split('/', 1)[1]) for r, e, k in worst[:4]]))
        assert not bad, bad[:5]
    for k in ('gen_images',) + (('gen_images_enc',) if hp.nz else ()):
        err = (model.outputs_time_major(k).cpu() - res['outputs'][k]).abs().max().item()
        assert err <= otol, (k, err)
    if 'd_grads' in res:
        for k in [k for k in res['params'] if k.endswith('/u')]:        # u <- u' of every tower that has a loss term
            assert (model.params[k].cpu() - res['params'][k]).abs().max() <= 1e-4, k
    assert model.global_step == step + 1


@pytest.mark.parametrize('mode', ['tf32', 'exact'])
def test_benchmarked_configuration_b16_training_step_matches_golden(Model, mode):
    """BASELINE configs[1] at the size bench.py times (B=16): losses, outputs and every gradient tensor against the fp32 oracle
    outputs cached by tests/golden/make_golden_b16.py (count sketches; see there), in both arithmetic modes."""
    import make_golden_b16 as G
    gold = np.load(os.path.join(GOLD, 'savp_b16_step.npz'))
    hp, params, inputs, noise = G.case()
    _, ltol, floor, otol = MODES[mode]
    gtol = 5e-2 if mode == 'tf32' else EXACT_GTOL['savp']
    with arithmetic(mode):
        model = _gpu_step(Model, G.HK, params, inputs, noise, G.STEP, G.sampling_mask())
    lv = model.losses()
    lv.update(g_loss=model.g_loss, d_loss=model.d_loss)
    key = 'fp32'
    names = [k.split('/sketch/', 1)[1] for k in gold.files if k.startswith(key + '/sketch/')]
    assert len(names) > 100
    for k in [f for f in gold.files if f.startswith(key + '/loss/')]:
        nm, v = k.split('/loss/', 1)[1], float(gold[k])
        assert abs(lv[nm] - v) <= ltol * abs(v) + 1e-6, (nm, lv[nm], v)
    worst = []
    for kind in ('generator/', 'discriminator/'):
        sub = [n for n in names if n.startswith(kind)]
        gmax = max(float(gold['%s/norm/%s' % (key, n)]) for n in sub)
        for n in sub:
            ref_n = float(gold['%s/norm/%s' % (key, n)])
            if ref_n < floor * gmax:
                continue
            sk = G.sketch(n, model.grads[n].cpu()).numpy()
            ref = gold['%s/sketch/%s' % (key, n)]
            # |sketch(a) - sketch(b)| estimates |a - b| (6 % relative standard deviation with 512 buckets)
            worst.append((float(np.linalg.norm(sk - ref) / ref_n), n))
    worst.sort(reverse=True)
    print('B=16 [%s] vs fp32 oracle: worst gradient errors %s' % (mode, ['%.2e %s' % w for w in worst[:4]]))
    assert worst[0][0] <= 1.25 * gtol, worst[:5]
    for k in ('gen_images', 'gen_images_enc', 'zs_mu_enc'):
        got = model.outputs_time_major(k).cpu().reshape(-1)[::G.SAMPLE_STRIDE].numpy()
        assert np.abs(got - gold['%s/out/%s' % (key, k)]).max() <= otol, k
    for f in [f for f in gold.files if f.startswith(key + '/u/')]:
        assert np.abs(model.params[f.split('/u/', 1)[1]].cpu().numpy() - gold[f]).max() <= 1e-4


# ---------------------------------------------------------------------------------------------- full-length configs
def _forward(Model, hk, B, shape, A=0, seed=0, mode=None):
    hp = O.make_hparams(**hk)
    params, _ = O.init_params(hp, shape, action_dim=A, seed=seed)
    inputs, noise = O.make_synthetic_inputs(hp, B, shape, action_dim=A, seed=seed)
    model = Model(mode='test', hparams_dict=hk)
    model.set_params(params)
    binp = {'images': inputs['images'].permute(1, 0, 2, 3, 4)}
    if A:
        binp['actions'] = inputs['actions'].permute(1, 0, 2)
    model.build_graph(binp)
    model.set_inputs(binp, noise)
    model.generator_forward()
    torch.cuda.synchronize()
    out = {}
    for m in (None, mode):
        O.set_tf32_emulation(m)
        try:
            with torch.no_grad():
                out[m] = O.generator(O.Vars(params), hp, inputs, noise, O.ground_truth_mask(hp, B))
        finally:
            O.set_tf32_emulation(None)
    return model, out


@pytest.mark.parametrize('name,hk,B,shape,A', [
    # BASELINE configs[2]: action-conditioned SAVP, 64x64x3 + 4-dim actions, 2 context + 28 predicted
    ('cfg3', dict(context_frames=2, sequence_length=30, nz=8), 4, (64, 64, 3), 4),
    # BASELINE configs[4]: KTH shape 64x64x1, 10 context + 20 predicted, nz=32 (hparams/kth/ours_vae_l1)
    ('cfg5', dict(context_frames=10, sequence_length=30, nz=32), 4, (64, 64, 1), 0),
    # BASELINE configs[3]: 128x128x3, 4 context + 12 predicted (4 encoder / 4 decoder levels)
    ('cfg4', dict(context_frames=4, sequence_length=16, nz=8), 2, (128, 128, 3), 0),
])
def test_full_length_generator_matches_oracle(Model, name, hk, B, shape, A):
    """Full sequence lengths of BASELINE configs[2..4] (forward): TF32 error growth over up to 29 recurrent steps.  64x64
    configurations stay within the north-star's 1e-3 of the fp32 oracle in product mode; the 128x128 / 16-step configuration
    sits AT 1e-3 (0.95 - 1.03e-3 depending on the summation order of the chosen engines) and is held to 1.5e-3 there and to
    1e-4 in the fp32-exact mode.  Against the oracle with the same operand rounding the product mode is within 5e-4."""
    mode = tf32_mode()
    model, refs = _forward(Model, hk, B, shape, A, seed=1, mode=mode)
    tol32 = 1.5e-3 if name == 'cfg4' else 1e-3
    for k in ('gen_images', 'gen_images_enc'):
        got = model.outputs[k].cpu()
        e32 = (got - refs[None][k].permute(1, 0, 2, 3, 4)).abs().max().item()
        eq = (got - refs[mode][k].permute(1, 0, 2, 3, 4)).abs().max().item()
        print('%s %s: max-abs vs fp32 oracle %.2e, vs tf32-emulating oracle %.2e (T=%d)' % (name, k, e32, eq, hk['sequence_length']))
        assert e32 <= tol32, (name, k, e32)
        assert eq <= 5e-4, (name, k, eq)
    if name == 'cfg4':
        with arithmetic('exact'):
            model, refs = _forward(Model, hk, B, shape, A, seed=1, mode=None)
        for k in ('gen_images', 'gen_images_enc'):
            e = (model.outputs[k].cpu() - refs[None][k].permute(1, 0, 2, 3, 4)).abs().max().item()
            print('%s %s [exact]: max-abs vs fp32 oracle %.2e' % (name, k, e))
            assert e <= 1e-4, (name, k, e)


# ---------------------------------------------------------------------------------------------- graph replay vs eager
def test_captured_step_reproduces_the_eager_step(Model, tmp_path):
    """The step bench.py times is ONE captured CUDA graph with parallel branches (discriminator towers, spectral norm + packing
    under the generator forward).  From the same checkpoint and batch: the eager step, a captured replay and a second replay
    must produce the same losses and gradients up to what summation-order noise becomes in TF32 arithmetic (atomics in split-K
    and the weight gradients reorder fp32 sums; downstream truncations to TF32 flip, profiles/r02_parity_noise_floor.md):
    measured on a B200 6e-4 / 1e-3 between two replays and 5e-4 / 7e-4 between the graph and the eager step (G / D
    gradients), 1.4e-4 on the losses.  A step
    that is not executed at capture time (the bug this test found), a stale buffer or a race between branches shows as O(1)."""
    import make_golden_b16 as G
    hp, params, inputs, noise = G.case()
    binp = {'images': inputs['images'].permute(1, 0, 2, 3, 4)}
    grads, ck = {}, None
    for how in ('eager', 'graph'):
        model = Model(mode='train', hparams_dict=G.HK)
        model.set_params(params)
        model.build_graph(binp)
        model.use_cuda_graph = how == 'graph'
        model.train_step(binp)                                   # step 0 (always eager; the graph is captured afterwards)
        if ck is None:
            # both models continue from the SAME step-0 state: Adam's first update turns summation-order noise into +-lr
            # steps, so two step-0 runs end 5e-4 apart and step 1 from them differs by ~4e-3 in the losses (measured)
            ck = model.save(str(tmp_path))
        runs = []
        for rep in range(2 if how == 'graph' else 1):
            model.restore(None, ck)
            assert model.global_step == 1
            model.train_step(binp)
            torch.cuda.synchronize()
            assert (model._graph is not None) == (how == 'graph')
            runs.append((model.g_grad.clone(), model.d_grad.clone(), model.loss_vals.clone()))
        grads[how] = runs

    def rel(a, b):
        return ((a - b).double().norm() / b.double().norm()).item()
    (g0, d0, l0), (g1, d1, l1) = grads['graph']
    ge, de, le = grads['eager'][0]
    errs = dict(replay_vs_replay=(rel(g0, g1), rel(d0, d1), rel(l0, l1)), graph_vs_eager=(rel(g0, ge), rel(d0, de), rel(l0, le)))
    print('captured-step reproducibility (relative L2 of the flat G / D gradients, loss vector):', errs)
    assert max(errs['replay_vs_replay'][:2]) < 5e-3 and errs['replay_vs_replay'][2] < 1e-3, errs
    assert max(errs['graph_vs_eager'][:2]) < 3e-2 and errs['graph_vs_eager'][2] < 1e-3, errs
