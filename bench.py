#!/usr/bin/env python
"""bench.py -- SAVP training hot path on B200 (frames/sec, BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run, one rank per GPU)
  python bench.py --impl reference ...                      (the CPU arm: the oracle port on the host cores)
  python bench.py ... --dump-outputs DIR                    (also writes what the last timed step computed, DIR/<name>.npy)

Every timed loop of training steps (`e2e`, `value`, the step without the engine in `roofline`, the CPU arm) runs exactly K
steps.  Inputs, initial variables and per-step noise are seeded.  With --dump-outputs the last timed step starts from the
initial variables and optimizer state (restored outside the timed window), so what it computes depends on the arguments
alone and two runs, or two builds, can be compared output for output.

A "step" is one full optimisation step of --config (default cfg2 = configs[1] of BASELINE.json: SAVP, bair_action_free/ours_savp
hparams: VAE+GAN, 64x64x3, 2 context + 10 predicted, batch 16 per GPU): generator forward (posterior + prior unrolls),
4 discriminator towers, D backward + Adam(D), post-update D forward, G backward (BPTT) + Adam(G).
frames/sec = global_batch * (T-1) generated frames per step / step time.

`value`   : inputs resident in HBM, the whole step replayed from a CUDA graph, timed with CUDA events, max over ranks.
`e2e`     : the public API call (model.train_step(inputs)) with HOST inputs: pinned H2D of the batch + D2H of the losses
            inside the timed region.
`roofline`: the ConvLSTM gate convolutions (rnn_ops.py:121; the north-star kernel) timed alone with CUDA events, and
            `roofline.whole_engine`: every tensor-core call of one step (forward + dgrad + wgrad).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SAVP = dict(lr=0.0002, beta1=0.5, beta2=0.999, l1_weight=100.0, l2_weight=0.0, kl_weight=1.0, video_sn_vae_gan_weight=0.1,
            video_sn_gan_weight=0.1, vae_gan_feature_cdist_weight=10.0, gan_feature_cdist_weight=0.0, state_weight=0.0)
# BASELINE.json `configs` (SURVEY.md 8d): name -> hparams (shipped hparams files of the reference), image shape, action dim,
# per-GPU batch.  cfg2 is the configuration the metric is quoted on; the others are parity-test cases that can be timed too.
CONFIGS = {
    'cfg1': dict(what='BASELINE configs[0]: deterministic generator (hparams/bair_action_free/ours_deterministic_l1: no VAE, no GAN, '
                      'L1), synthetic 64x64x3, 2 context + 10 predicted',
                 hparams=dict(context_frames=2, sequence_length=12, batch_size=4, lr=0.001, beta1=0.9, beta2=0.999, l1_weight=1.0,
                              l2_weight=0.0, kl_weight=0.0, video_sn_vae_gan_weight=0.0, video_sn_gan_weight=0.0, state_weight=0.0, nz=0),
                 image=(64, 64, 3), actions=0, batch=4),
    'cfg2': dict(what='BASELINE configs[1]: SAVP (VAE+GAN) bair_action_free/ours_savp hparams, synthetic 64x64x3, 2 context + 10 '
                      'predicted',
                 hparams=dict(SAVP, context_frames=2, sequence_length=12, batch_size=16), image=(64, 64, 3), actions=0, batch=16),
    'cfg3': dict(what='BASELINE configs[2]: action-conditioned SAVP (ours_savp weights; the reference ships no hparams/bair), synthetic '
                      '64x64x3 + 4-dim actions, 2 context + 28 predicted',
                 hparams=dict(SAVP, context_frames=2, sequence_length=30, batch_size=32), image=(64, 64, 3), actions=4, batch=32),
    'cfg4': dict(what='BASELINE configs[3]: SAVP synthetic 128x128x3, 4 context + 12 predicted (CDNA warp stress)',
                 hparams=dict(SAVP, context_frames=4, sequence_length=16, batch_size=8), image=(128, 128, 3), actions=0, batch=8),
    'cfg5': dict(what='BASELINE configs[4]: VAE-only (hparams/kth/ours_vae_l1: nz=32, L1 + KL 1e-5, no GAN), KTH-shape synthetic '
                      '64x64x1, 10 context + 20 predicted',
                 hparams=dict(context_frames=10, sequence_length=30, batch_size=32, lr=0.001, beta1=0.9, beta2=0.999, l1_weight=1.0,
                              l2_weight=0.0, kl_weight=1e-05, video_sn_vae_gan_weight=0.0, video_sn_gan_weight=0.0, state_weight=0.0,
                              nz=32),
                 image=(64, 64, 1), actions=0, batch=32),
}
CFG = CONFIGS['cfg2']
SAVP_HPARAMS = CFG['hparams']          # kept for tests/profile_step.py
IMAGE = CFG['image']
PER_GPU_BATCH = CFG['batch']


def select_config(name):
    global CFG, SAVP_HPARAMS, IMAGE, PER_GPU_BATCH
    CFG = CONFIGS[name]
    SAVP_HPARAMS, IMAGE, PER_GPU_BATCH = CFG['hparams'], CFG['image'], CFG['batch']


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d['hbm_gbs'], bf16=d['bf16_tflops'], bf16_sustained=d.get('bf16_tflops_sustained'), src='measured')
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, src='fallback')


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        while not self.stop_flag:
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q, '--format=csv,noheader,nounits'],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(',')])
            except Exception:
                pass
            time.sleep(0.15)

    def summary(self):
        if not self.rows:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['unavailable'])
        sm = sorted(int(float(r[0])) for r in self.rows if r[0].replace('.', '').isdigit())
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith('active') for r in self.rows if len(r) > 2 + i)]
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=int(float(self.rows[0][1])), reasons=reasons,
                    samples=len(self.rows))


def synthetic_batch(batch, seed):
    """U[0,1) images (dataset contract base_dataset.py:189), one fresh batch per step, as pinned host tensors."""
    import torch
    g = torch.Generator().manual_seed(seed)
    T = SAVP_HPARAMS['sequence_length']
    imgs = torch.rand(batch, T, *IMAGE, generator=g)
    out = {'images': imgs}
    if CFG['actions']:
        out['actions'] = torch.randn(batch, T - 1, CFG['actions'], generator=g)
    return {k: (v.pin_memory() if torch.cuda.is_available() else v) for k, v in out.items()}


CPU_THREADS = 32      # the CPU arm is pinned to a fixed intra-op thread count (<= the box's cores) so that runs are comparable


def oracle_step_time(batch, steps, threads=None):
    """Times full training steps of the CPU oracle (the port of the reference's TF1 graph) of the selected config at batch
    `batch`.  One untimed warm-up step (allocator / oneDNN primitive cache), then `steps` timed ones.
    Returns (list of seconds per step, threads used)."""
    import torch
    from oracle import savp_oracle as O
    torch.set_num_threads(max(1, min(threads or CPU_THREADS, os.cpu_count() or 1)))
    hk = {k: v for k, v in SAVP_HPARAMS.items() if k != 'batch_size'}
    hp = O.make_hparams(**hk)
    params, _ = O.init_params(hp, IMAGE, action_dim=CFG['actions'], seed=0)
    opt = dict(m={k: torch.zeros_like(v) for k, v in params.items()}, v={k: torch.zeros_like(v) for k, v in params.items()}, t=0)
    times = []
    for s in range(steps + 1):
        inputs, noise = O.make_synthetic_inputs(hp, batch, IMAGE, action_dim=CFG['actions'], seed=s, smooth=False)
        t0 = time.time()
        res = O.train_step(params, opt, hp, inputs, noise, step=s)
        times.append(time.time() - t0)
        params = res['params']
    return times[1:], torch.get_num_threads()


def cpu_baseline_subprocess(config, batch, steps, timeout_s=240):
    """Runs the oracle timing in a fresh interpreter (no CUDA context) so that the GPU process's threads cannot interfere;
    bounded by a timeout."""
    code = ('import sys, json; sys.path.insert(0, %r); import bench; bench.select_config(%r); '
            't, n = bench.oracle_step_time(%d, %d); print(json.dumps(dict(sec=t, threads=n)))' % (ROOT, config, batch, steps))
    env = dict(os.environ, CUDA_VISIBLE_DEVICES='')
    try:
        r = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, timeout=timeout_s, env=env)
        line = [l for l in r.stdout.splitlines() if l.startswith('{')]
        return json.loads(line[-1]) if line else None
    except subprocess.TimeoutExpired:
        return None


def cpu_sample_batch():
    """The CPU arm runs a bounded sample of the workload: full training steps at a small batch (cost is linear in the batch)."""
    return 1 if IMAGE[0] >= 128 or SAVP_HPARAMS['sequence_length'] > 16 else 2


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    sample_b = cpu_sample_batch()
    S = SAVP_HPARAMS['sequence_length'] - 1
    k = args.steps
    times, cores = oracle_step_time(sample_b, k)
    med = sorted(times)[len(times) // 2]
    fps = sample_b * S / med
    sample = ('%d full training steps (+1 warm-up) at batch %d (of %d) on the host, torch/oneDNN fp32, %d intra-op threads: median %.2f s, '
              'min %.2f s, max %.2f s per step' % (k, sample_b, PER_GPU_BATCH, cores, med, min(times), max(times)))
    line = dict(metric='frames/sec SAVP 64x64 2+10 (training)', value=fps, unit='frames/s', n_gpus=args.gpus, steps=k,
                warmup=1, ms_per_step=med * 1e3, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32',
                data='synthetic', impl='reference',
                config=dict(workload='%s; CPU sample batch %d' % (CFG['what'], sample_b), name=args.config,
                            note='the TF1 reference cannot run here (needs tensorflow 1.x); this is its line-by-line CPU port (oracle/)'),
                cpu_baseline=dict(value=fps, unit='frames/s', cores=cores, kind='port', sample=sample,
                                  frames_per_s_min=sample_b * S / max(times), frames_per_s_max=sample_b * S / min(times)),
                e2e=dict(value=fps, unit='frames/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))


def ncu_traffic():
    """DRAM traffic of the dominant kernel per launch (dram__bytes_read.sum + dram__bytes_write.sum) from the committed
    `ncu --set full` capture of the lstm_h0 gate convolution (profiles/r02_ncu_full_summary.json, tests/ncu_capture_r02.sh),
    next to the algorithmic bytes of that launch (input + packed weights read, gate pre-activations written)."""
    out = dict(traffic=None)
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'profiles', 'r02_ncu_full_summary.json')

    def mb(v):
        num, unit = v.split()[:2]
        return float(num) * {'byte': 1.0, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}[unit]
    try:
        with open(path) as f:
            caps = json.load(f)['captures']['r02_engine_kernels.ncu-rep']
        c = [x for x in caps if 'igemm_halo' in x['kernel'] and x['grid'].startswith('(128,')][0]   # lstm_h0: 128 M = 256 tiles
        out['traffic'] = mb(c['dram_bytes_read']) + mb(c['dram_bytes_write'])
        out['traffic_unit'] = 'bytes per launch (lstm_h0 gate conv, halo mode, ncu --set full)'
        out['traffic_algorithmic'] = 32 * 1024 * 72 * 4 + 25 * 128 * 96 * 4 + 32 * 1024 * 128 * 4
        out['traffic_note'] = ('reads = input + weights once (no re-reads from HBM); the 16.8 MB of gate pre-activations stay in the '
                               '126 MB L2 for the gate kernel that follows, so almost nothing is written back')
        out['tensor_pipe_active_pct'] = float(c['tensor_pipe_active_pct_of_active'].split()[0])
        out['l2_to_sm_bytes'] = mb(c['l1tex__m_xbar2l1tex_read_bytes.sum'])
    except Exception:       # noqa: BLE001  (profile summary absent: leave traffic null)
        pass
    return out


def time_gate_kernels(model, iters=3):
    """CUDA-event timing of the five ConvLSTM gate convolutions (one launch per timestep buffer, cycling through all
    T-1 timesteps so consecutive launches touch different HBM lines; working set > L2), replayed from a CUDA graph."""
    import torch
    flops, ms = 0.0, 0.0
    per_layer = []
    for d in model.gl:
        if not d['use']:
            continue
        li = d['li']
        conv = d['rconv']
        rin, gpre = model.Bf['rin%d' % li], model.Bf['gpre%d' % li]
        S = model.S
        for t in range(S):
            conv.fwd(rin[t], gpre[t])
        torch.cuda.synchronize()
        # the S launches are replayed from a CUDA graph: a 16 us kernel launched eagerly through ctypes is host-bound
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for t in range(S):
                conv.fwd(rin[t], gpre[t])
        g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        t_ms = e0.elapsed_time(e1) / (iters * S)
        del g
        M = model.NB * d['h'] * d['w']
        fl = 2.0 * M * (4 * d['oc']) * (25 * conv.ci_ref)        # algorithmic: reference channel count, no padding
        per_layer.append(dict(layer='lstm_h%d' % li, M=M, N=4 * d['oc'], K=25 * conv.ci_ref, ms=t_ms, tflops=fl / t_ms / 1e9))
        flops += fl
        ms += t_ms
    return flops, ms, per_layer


def engine_in_graph_ms(model, one_step, steps):
    """The engine's cost INSIDE the captured step: the step is re-captured without the tensor-core engine calls
    (results are garbage by design) and timed; full step - this = what the engine costs on the critical path, with the
    overlap of the parallel graph branches and warm caches that the per-call timings cannot see."""
    import torch
    from video_prediction_b200 import lib as L
    saved = set(L._SKIP)
    try:
        L._SKIP.update(('igemm', 'wgrad'))
        model._graph, model._eager_steps = None, 0
        for _ in range(4):
            one_step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            one_step()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps
    finally:
        L._SKIP.clear()
        L._SKIP.update(saved)
        model._graph, model._eager_steps = None, 0


def engine_profile(model, batch):
    """Whole-engine roofline: ONE eager training step with every tensor-core engine call (forward + dgrad = `igemm`, weight
    gradients = `wgrad`) bracketed by CUDA events on its launching stream; algorithmic FLOPs as SURVEY.md 8(d) counts them
    (internal channel counts: the image's 3 channels are stored as 4).  The discriminator towers run sequentially here
    (VP_CONCURRENT_D=0) so that the event pairs do not time overlapping kernels."""
    import torch
    from video_prediction_b200 import lib as L
    old = os.environ.get('VP_CONCURRENT_D')
    os.environ['VP_CONCURRENT_D'] = '0'
    try:
        model.stage_step()
        torch.cuda.synchronize()
        # replay=True: every call is re-captured into a CUDA graph and the replay is timed -- an eager event pair around a
        # kernel of a few microseconds measures the host's launch path (ctypes + tensor-map encoding), not the GPU
        L.profile_engine(True, replay=True)
        model._step_device(getattr(model, '_allreduce', None))
        model.global_step += 1
        return L.profile_engine(False)
    finally:
        if old is None:
            os.environ.pop('VP_CONCURRENT_D', None)
        else:
            os.environ['VP_CONCURRENT_D'] = old


DUMP_CAP = 1 << 22     # elements per dumped array (16 MB of float32): at most two arrays reach it, so a dump stays < 64 MB


def dump_outputs(model, losses, out_dir):
    """Writes what the last timed step computed, as a caller of train_step() + losses() receives it, to out_dir/<name>.npy:
    every loss term (float64 scalars) and the step's generated frames and posterior statistics (float32, batch-major as
    `model.outputs` holds them).  An array of more than DUMP_CAP
    elements is written as <name>_sample.npy: its flattened elements at DUMP_CAP positions drawn with a fixed seed, in
    ascending order."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for k, v in losses.items():
        np.save(os.path.join(out_dir, k + '.npy'), np.float64(v))
    keys = ('gen_images', 'gen_images_enc', 'zs_mu_enc', 'zs_log_sigma_sq_enc') if model.hparams.nz else ('gen_images',)
    arrays = {k: model.outputs_time_major(k).transpose(0, 1) for k in keys}
    for name, v in arrays.items():
        if v.numel() > DUMP_CAP:
            idx = np.sort(np.random.default_rng(0).choice(v.numel(), DUMP_CAP, replace=False))
            v, name = v.reshape(-1)[torch.from_numpy(idx).to(v.device)], name + '_sample'
        np.save(os.path.join(out_dir, name + '.npy'), v.detach().float().contiguous().cpu().numpy())


def run_ours(args):
    import torch
    import torch.distributed as dist
    from video_prediction_b200 import lib as L
    from video_prediction_b200.models import get_model_class
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    torch.cuda.set_device(local)
    B = PER_GPU_BATCH
    # data parallelism lives in the model: build_graph reads torchrun's env (dp.init_from_env), broadcasts rank 0's variables
    # and train_step all-reduces the two flat gradient buffers (weak scaling: num_gpus=1 -> every rank feeds its own batch)
    model = get_model_class('savp')(mode='train', hparams_dict=dict(SAVP_HPARAMS), num_gpus=1)
    batch0 = synthetic_batch(B, seed=1000 * rank)
    log('building model %s (batch %d per GPU)' % (args.config, B))
    model.build_graph(batch0)
    assert model.world_size == world
    initial = None
    if args.dump_outputs:
        # every step adds summation-order noise (atomics) that Adam and the GAN game amplify (two runs end ~30 % apart after
        # 50 steps), so the last timed step of a dump run starts again from these seeded initial variables and optimizer state
        initial = tempfile.TemporaryDirectory()
        model.save(initial.name)
    log('built; warming up the eager path')
    S = model.S
    frames_per_step = world * B * S

    # ---------------- e2e: public API with host inputs (H2D + D2H inside the timed region)
    batches = [synthetic_batch(B, seed=1000 * rank + i) for i in range(4)]
    h2d = sum(v.numel() * 4 for v in batches[0].values())
    model.use_cuda_graph = not args.no_graph
    for i in range(max(3, args.warmup) + 1):
        model.train_step(batches[i % 4])
        model.losses()
    torch.cuda.synchronize()
    log('timing e2e')
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k_e2e = args.steps
    t0 = time.time()
    e0.record()
    for i in range(k_e2e):
        model.train_step(batches[i % 4])
        lv = model.losses()              # D2H of the step's losses (mean over replicas)
    e1.record()
    torch.cuda.synchronize()
    e2e_ms = max(e0.elapsed_time(e1), (time.time() - t0) * 1e3) / k_e2e
    d2h = model.loss_vals.numel() * 4
    log('e2e %.2f ms/step (cuda graph inside train_step: %s)' % (e2e_ms, model._graph is not None))

    # ---------------- value: HBM-resident inputs, whole step as one CUDA graph
    graph = model._graph
    model.set_inputs(batches[0])
    if graph is None:
        model.use_cuda_graph = False

    def one_step():
        model.train_step()       # inputs already resident; replays the captured graph
    # launches per step: counted on one eager execution of the same device step
    c0 = L.launch_count()
    model.stage_step()
    model._step_device(getattr(model, '_allreduce', None))
    model.global_step += 1
    launches_per_step = L.launch_count() - c0
    log('graph=%s launches/step=%s; warm-up' % (graph is not None, launches_per_step))
    for _ in range(max(3, args.warmup)):
        one_step()
    torch.cuda.synchronize()
    log('timing %d steps' % args.steps)
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1, e2, e3 = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    torch.cuda.synchronize()
    e0.record()
    for _ in range(args.steps - (initial is not None)):
        one_step()
    e1.record()
    if initial is not None:
        # the last timed step of a dump run starts from the seeded initial state, restored outside the timed window; its
        # host-side staging runs before its start event too, as it does under the GPU work of the step before in the loop
        model.restore(None, initial.name)     # copies into the buffers the captured graph reads
        initial.cleanup()
        model.redraw_step_randomness()
        model.stage_step()
        e2.record()
        if graph is not None:
            graph.replay()                    # what one_step() runs after the same staging
        else:
            model._step_device(getattr(model, '_allreduce', None))
        model.global_step += 1
        e3.record()
    torch.cuda.synchronize()
    ms = (e0.elapsed_time(e1) + (e2.elapsed_time(e3) if initial is not None else 0.0)) / args.steps
    sampler.stop_flag = True
    log('%.2f ms/step' % ms)
    if world > 1:
        t = torch.tensor([ms, e2e_ms], device='cuda')
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms = t[0].item(), t[1].item()
        dist.barrier()
    losses = model.losses()
    finite = all(v == v for v in losses.values())
    if args.dump_outputs and rank == 0:      # before the roofline legs, which run steps whose results are garbage by design
        dump_outputs(model, losses, args.dump_outputs)
        log('outputs of the last timed step written to %s' % args.dump_outputs)

    # ---------------- rooflines + CPU baseline (rank 0; the CPU leg at N = 1 only)
    no_engine_ms = None
    if not args.no_roofline and world == 1 and graph is not None:
        no_engine_ms = engine_in_graph_ms(model, one_step, args.steps)
        log('step without the engine: %.2f ms' % no_engine_ms)
    prof = None if args.no_roofline else engine_profile(model, batches[0])     # every rank runs the same (collective-bearing) step
    if rank == 0:
        peaks = load_peaks()
        roof = None
        if not args.no_roofline:
            flops, gate_ms, per_layer = time_gate_kernels(model)
            log('gate kernels timed; cpu baseline leg')
            achieved = flops / gate_ms / 1e9     # TFLOP/s over the gate convolutions of one timestep
            roof = dict(bound='tensor', kernel='ConvLSTM gate convolutions (rnn_ops.py:121) on the tcgen05 kind::tf32 engine, forward',
                        achieved=achieved, peak=peaks['bf16'], unit='TFLOP/s', frac=achieved / peaks['bf16'],
                        peak_source=peaks['src'] + ' cuBLAS bf16 (burst); the tf32 MMA rate is half of bf16',
                        peak_tf32_equiv=peaks['bf16'] / 2, frac_of_tf32_peak=achieved / (peaks['bf16'] / 2),
                        per_layer=per_layer, **ncu_traffic())
            tot_f = sum(d['flops'] for d in prof.values())
            tot_ms = sum(d['ms'] for d in prof.values())
            sustained = (peaks.get('bf16_sustained') or peaks['bf16']) / 2
            roof['whole_engine'] = dict(
                what='every tensor-core engine call of ONE training step (forward + dgrad + wgrad of all convolutions), '
                     'algorithmic FLOPs / summed GPU time of the calls, each call timed as a CUDA-graph replay of 4 repeats '
                     '(CUDA events; eager event pairs around kernels of a few microseconds time the host launch path)',
                tflop_per_step=tot_f / 1e12, engine_ms_per_step=tot_ms, achieved=tot_f / tot_ms / 1e9, unit='TFLOP/s',
                peak_tf32_equiv_sustained=sustained, frac_of_tf32_peak_sustained=tot_f / tot_ms / 1e9 / sustained,
                frac_of_bf16_peak_sustained=tot_f / tot_ms / 1e9 / (2 * sustained),
                by_kind={k: dict(calls=d['calls'], tflop=d['flops'] / 1e12, ms=d['ms'], tflops=d['flops'] / d['ms'] / 1e9)
                         for k, d in prof.items()},
                whole_step_tflops=tot_f / ms / 1e9)
            if no_engine_ms is not None:
                roof['whole_engine']['in_graph'] = dict(
                    what='captured step re-timed without the engine calls: full - without = the engine on the critical path',
                    step_ms=ms, step_without_engine_ms=no_engine_ms, engine_ms=ms - no_engine_ms,
                    achieved=tot_f / (ms - no_engine_ms) / 1e9, frac_of_tf32_peak_sustained=tot_f / (ms - no_engine_ms) / 1e9 / sustained)
        cpu = None
        if world == 1 and not args.no_cpu:
            sb = cpu_sample_batch()
            r = cpu_baseline_subprocess(args.config, sb, 3)
            if r is not None:
                med = sorted(r['sec'])[len(r['sec']) // 2]
                cpu = dict(value=sb * S / med, unit='frames/s', cores=r['threads'], kind='port',
                           sample='3 full training steps (+1 warm-up) at batch %d (of %d) with the CPU oracle (torch/oneDNN fp32, %d '
                                  'intra-op threads of %d logical CPUs): median %.2f s, min %.2f s, max %.2f s per step'
                                  % (sb, B, r['threads'], os.cpu_count() or 0, med, min(r['sec']), max(r['sec'])))
            else:
                cpu = dict(value=None, unit='frames/s', cores=os.cpu_count(), kind='port', sample='timed out')
        clocks = sampler.summary()
        line = dict(metric='frames/sec SAVP 64x64 2+10 (training)', value=frames_per_step / ms * 1e3, unit='frames/s',
                    n_gpus=world, steps=args.steps, warmup=max(3, args.warmup), ms_per_step=ms, higher_is_better=True,
                    scaling='weak', vs_baseline=None, dtype='tf32 tensor-core convolutions, fp32 accumulate / state / optimizer',
                    sequences_per_s=world * B / ms * 1e3,     # the reference's own `image/sec` print (train.py:331)
                    data='synthetic',
                    config=dict(workload='%s, batch %d per GPU; full step = G fwd (posterior + prior unrolls) + D towers + Adam(D) + '
                                         'post-update D fwd + G BPTT + Adam(G)' % (CFG['what'], B), name=args.config,
                                global_batch=world * B, per_gpu_batch=B, sequence_length=SAVP_HPARAMS['sequence_length'],
                                parallelism='dp%d' % world, cuda_graph=graph is not None,
                                l2='working set of one step (GBs of activations) is far larger than the 126 MB L2'),
                    e2e=dict(value=frames_per_step / e2e_ms * 1e3, unit='frames/s', ms_per_step=e2e_ms, h2d_bytes_per_step=h2d,
                             d2h_bytes_per_step=d2h, api='get_model_class("savp")(...).train_step(host inputs) + .losses()'),
                    gpu_launches=int(launches_per_step) * args.steps, gpu_launches_per_step=int(launches_per_step),
                    roofline=roof, cpu_baseline=cpu, clocks=clocks, losses_finite=finite,
                    losses={k: round(v, 6) for k, v in losses.items() if v})
        print(json.dumps(line))
        sys.stdout.flush()
    if world > 1:
        # NCCL teardown with a captured graph alive can block; every rank is done, so synchronise and leave
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def log(msg):
    sys.stderr.write('[bench %.1fs] %s\n' % (time.time() - T0, msg))
    sys.stderr.flush()


T0 = time.time()


def main():
    import faulthandler
    faulthandler.enable()
    faulthandler.dump_traceback_later(int(os.environ.get('BENCH_WATCHDOG_S', '420')), exit=True)   # a hang dumps all stacks and exits
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--no-roofline', action='store_true', help='skip the roofline legs (gate kernels, whole-engine profile)')
    ap.add_argument('--config', default='cfg2', choices=sorted(CONFIGS), help='BASELINE.json configs[i-1]; the metric is quoted on cfg2')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write what the last timed step computed to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs applies to --impl ours')
    select_config(args.config)
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)
    faulthandler.cancel_dump_traceback_later()


if __name__ == '__main__':
    main()
