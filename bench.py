#!/usr/bin/env python
"""bench.py — frame-pairs/s of the per-video test-time optimisation step (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--pairs B] [--impl b200|reference] [--dump-outputs DIR]

One "step" = one joint-phase optimisation step (depth net + scene-flow MLP trainable, flags of
experiments/davis/train_sequence.sh) over B synthetic frame pairs per GPU (default 384x224, 80 frames =
BASELINE.json configs[2]: the full sm_100a path - tcgen05 depth CNN + tcgen05 scene-flow MLP + fused re-projection
kernels; --height/--width/--frames/--gaps select the other configs). Gaps cycle step by step (all pairs of one
step share the gap). Prints ONE JSON line (rank 0). See the repository README / DESIGN.md for the field meanings.

--impl reference : the reference's CPU PyTorch computation, restated by oracle/step.py (kind "port" — the
Python reference tree cannot travel to the GPU box), on the host cores; same workload and gap schedule, each step a
bounded sample of it (one pair).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

H, W, N_FRAMES = 224, 384, 80
GAPS = (8, 6, 4, 2, 1)   # experiments' gap set; largest first so that the >= 3 warm-up steps size the caching allocator
METRIC = 'frame-pairs/sec per step (384x224)'
UNIT = 'frame-pairs/s'


def configure(args):
    """--height/--width/--frames/--gaps -> module-level workload (BASELINE.json configs[2..4])."""
    global H, W, N_FRAMES, GAPS, METRIC
    H, W, N_FRAMES = args.height, args.width, args.frames
    GAPS = tuple(int(g) for g in args.gaps.split(','))
    METRIC = 'frame-pairs/sec per step (%dx%d)' % (W, H)


def workload_name():
    if (W, H, N_FRAMES) == (384, 224, 80):
        base = "synthetic 80-frame sequence 384x224 (BASELINE.json configs[2]: full sm_100a path)"
    elif (W, H, N_FRAMES) == (768, 448, 80):
        base = "synthetic 80-frame sequence 768x448 (BASELINE.json configs[3])"
    elif (W, H, N_FRAMES) == (512, 288, 200):
        base = "ShutterStock-shape sequence 512x288, 200 frames, mixed-gap flow pairs (BASELINE.json configs[4], fp32/TF32 I/O)"
    else:
        base = "synthetic %d-frame sequence %dx%d" % (N_FRAMES, W, H)
    return base + ("; joint phase (--midas --use_disp --time_dependent --acc_mul 1): tcgen05 TF32 MiDaS depth CNN fwd+bwd, "
                   "tcgen05 bf16x3 scene-flow MLP, fused re-projection kernels, flat Adam; gaps cycle %s" % ','.join(map(str, GAPS)))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--pairs', type=int, default=8, help='frame pairs per step per GPU')
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--height', type=int, default=224)
    ap.add_argument('--width', type=int, default=384)
    ap.add_argument('--frames', type=int, default=80)
    ap.add_argument('--gaps', type=str, default='8,6,4,2,1')
    ap.add_argument('--no-extras', action='store_true', help='skip the B=1 line, the eager-GPU reference and the kernel rooflines')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--roofline-pairs', type=int, default=64)
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs)')
    args = ap.parse_args()
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs needs --impl b200')
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    return args


# ---------------------------------------------------------------------------------------------------
def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d['hbm_gbs']), float(d.get('bf16_tflops', 1590.0)), 'measured'   # burst: kernels timed alone
    return 6650.0, 1590.0, 'fallback'


class ClockSampler:
    """nvidia-smi sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '200'], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(',')]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])), mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[4:8]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def step_pairs(step, rank, world, B):
    """Pairs of one step on one rank: all share the gap (uniform Euler-step count across ranks); the global batch of the
    step is a run of world*B consecutive start frames (wrapping), of which rank r takes its B - disjoint across ranks
    whenever world*B <= n_frames-1-gap. The product sampler is dvd_b200.datasets.resident.GapBucketSampler
    (DistributedSampler-style partition of the pair list, train.py:301-305, bucketed by gap)."""
    gap = GAPS[step % len(GAPS)]
    n = N_FRAMES - 1 - gap
    out = []
    for j in range(B):
        f = (step * 7 + rank * B + j) % n
        out.append((f, f + gap))
    return gap, out


# ---------------------------------------------------------------------------------------------------
def _pick_cpu_threads(depth_sd):
    """torch's CPU convolutions slow down when heavily over-threaded (128 threads on this box: 90 s/step vs
    ~10 s on 8). Short sweep on one depth-net forward; the fastest count is what 'all the host threads it can
    use' means in practice."""
    import torch
    from oracle import depth_nets
    cores = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, cores) if c <= cores})
    x = torch.rand(1, 3, H, W)
    best, best_t = cands[0], float('inf')
    for c in cands:
        torch.set_num_threads(c)
        with torch.no_grad():
            depth_nets.midas_forward(depth_sd, x[:, :, :64, :96])     # warm the pool
            t0 = time.perf_counter()
            depth_nets.midas_forward(depth_sd, x)
            dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best, cores


def _seeded_state():
    from dvd_b200 import synthetic
    from dvd_b200.networks.sceneflow_field import SceneFlowFieldNet
    from dvd_b200.third_party.MiDaS import MidasNet
    depth = synthetic.seed_net_(MidasNet(non_negative=True, normalize_input=True), 0, 2000.0).state_dict()
    mlp = synthetic.seed_net_(SceneFlowFieldNet(net_width=256, n_layers=4, time_dependent=True, N_freq_xyz=16, N_freq_t=16), 1).state_dict()
    return depth, mlp


def cpu_reference_steps(n_steps, warmup, quiet=True):
    """The reference's CPU path (oracle port): joint-phase step on the host cores, ONE pair per step (a bounded sample of
    the GPU arm's step), gaps cycling through the same schedule as the GPU arm."""
    import torch
    from dvd_b200 import synthetic
    from oracle import step as ostep
    opt = synthetic.default_opt()
    depth, mlp = _seeded_state()
    threads, cores = _pick_cpu_threads(depth)
    ad, am = {}, {}
    times = []
    log = None
    # one untimed tiny step (64x96) so that lazy initialisation is not billed to the first timed step
    tiny = synthetic.make_batch([(3, 5)], H=64, W=96, n_frames=N_FRAMES, seed=99, leading_dim=False)
    ostep.train_step(depth, mlp, tiny, opt, epoch=6)
    for i in range(warmup + n_steps):
        gap = GAPS[i % len(GAPS)]
        f = (10 + i) % (N_FRAMES - 1 - gap)
        batch = synthetic.make_batch([(f, f + gap)], H=H, W=W, n_frames=N_FRAMES, seed=i, leading_dim=False)
        t0 = time.perf_counter()
        log, depth, mlp, _ = ostep.train_step(depth, mlp, batch, opt, epoch=6, adam_depth=ad, adam_mlp=am)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    total = sum(times)
    return {'value': len(times) / total, 'unit': UNIT, 'cores': threads, 'host_cores': cores, 'kind': 'port',
            'sample': '%d joint-phase step(s) x 1 pair at %dx%d, gaps cycling %s (the GPU arm\'s schedule), oracle/step.py on torch CPU, '
                      '%d threads (fastest of a sweep over 8..%d), %d warm-up' % (len(times), W, H, ','.join(map(str, GAPS)), threads,
                                                                                  cores, warmup),
            'seconds': total, 'last_loss': log['loss']}


def run_reference_arm(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cb = cpu_reference_steps(args.steps, args.warmup)
    line = {'metric': METRIC, 'value': cb['value'], 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': 1e3 * cb['seconds'] / max(args.steps, 1), 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'impl': 'reference',
            'config': {'workload': workload_name(), 'pairs_per_step_per_gpu': args.pairs,
                       'sampled_as': 'one pair per CPU step of the same gap schedule (bounded sample); CPU PyTorch path of the '
                                     'reference restated by oracle/step.py'},
            'cpu_baseline': cb,
            'e2e': {'value': cb['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line), flush=True)


def gpu_eager_reference(dev, B, n_steps=8, warmup=3):
    """Denominator of the >=10x target (BASELINE.md 4 step 2): the reference-equivalent step in EAGER PyTorch on the same
    GPU - oracle/step.py (the restatement of Model._train_on_batch the parity tests pin to the reference) with every tensor
    on cuda:0 and torch's defaults (cuDNN TF32 convolutions on, as the reference would run today). Two workloads: the
    reference's own schedule (1 pair per step, train_sequence.sh:29-34) and this bench's B pairs per step; same gap cycle."""
    import torch
    from dvd_b200 import synthetic
    from oracle import step as ostep
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cudnn.benchmark = False
    opt = synthetic.default_opt()
    depth, mlp = _seeded_state()
    sd_d = {k: v.to(dev) for k, v in depth.items()}
    sd_m = {k: v.to(dev) for k, v in mlp.items()}

    stats = {}

    def run(pairs_per_step):
        bs = []
        for i in range(warmup + n_steps):
            gap = GAPS[i % len(GAPS)]
            n = N_FRAMES - 1 - gap
            pr = [((5 * i + j) % n, (5 * i + j) % n + gap) for j in range(pairs_per_step)]
            b = synthetic.make_batch(pr, H=H, W=W, n_frames=N_FRAMES, seed=200 + i, leading_dim=False)
            bs.append({k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in b.items()})
        ad, am = {}, {}
        d, m = sd_d, sd_m
        for i in range(warmup):
            _, d, m, _ = ostep.train_step(d, m, bs[i], opt, 6, ad, am)
        torch.cuda.synchronize()
        # per-step wall times (each step ends in the reference's own host read-backs), MEDIAN step: one stray slow step (allocator
        # growth, cuDNN heuristics on a new gap) must not decide the denominator of the speed-up
        ts = []
        for b in bs[warmup:]:
            t0 = time.perf_counter()
            _, d, m, _ = ostep.train_step(d, m, b, opt, 6, ad, am)
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        ts.sort()
        stats['steps_s_%d' % pairs_per_step] = [round(t, 4) for t in ts]
        # the gap schedule mixes cheap and expensive steps: mean over the schedule, with the slowest step replaced by the median
        ts[-1] = ts[len(ts) // 2]
        return n_steps * pairs_per_step / sum(ts)

    out = {'what': 'oracle/step.py (reference-equivalent eager PyTorch step) on cuda:0, cuDNN TF32 (torch default), inputs resident, '
                   '%d timed steps after %d warm-up, gaps cycling %s; slowest step replaced by the median step' % (
                       n_steps, warmup, ','.join(map(str, GAPS))), 'unit': UNIT}
    try:
        out['pairs_per_step_1'] = run(1)
        out['pairs_per_step_%d' % B] = run(B) if B > 1 else out['pairs_per_step_1']
    except Exception as e:   # noqa: BLE001
        out['error'] = repr(e)[:300]
    out.update(stats)
    torch.cuda.empty_cache()
    return out


# ---------------------------------------------------------------------------------------------------
DUMP_LOSSES = ('loss', 'flow_loss_1_2', 'disp_loss_1_2', 'sf_loss', 'acc_reg')
DUMP_DEPTH_SAMPLE = 1 << 20    # depth-net values kept per array (of ~105 M); the MLP's ~0.3 M are kept whole


def dump_outputs(out_dir, log, model):
    """What the last timed step hands its caller, as out_dir/<name>.npy: its loss terms (float64 scalars, the batch log), and
    the model state it leaves behind, which is what a checkpoint of the run would hold - parameters and both Adam moments of
    the scene-flow MLP in full, and of the depth net a fixed sample (the same DUMP_DEPTH_SAMPLE positions, drawn with seed 0,
    for every array and run), float32, in state-dict order. With the same arguments the inputs are identical from run to run,
    so two builds can be compared array by array."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for k in DUMP_LOSSES:
        np.save(os.path.join(out_dir, k + '.npy'), np.float64(log[k]))
    for tag, net, opt_ in (('depth_net', model.net_depth, model.optimizer_depth),
                           ('sceneflow_mlp', model.net_sceneflow, model.optimizer_scene)):
        params = [p for _, p in net.named_parameters()]
        st = opt_.state_dict()['state']
        moments = {key: [st[i][key] if i in st else torch.zeros_like(p) for i, p in enumerate(params)]
                   for key in ('exp_avg', 'exp_avg_sq')}
        arrays = {'params': params, 'adam_exp_avg': moments['exp_avg'], 'adam_exp_avg_sq': moments['exp_avg_sq']}
        n = sum(p.numel() for p in params)
        idx = None
        if n > DUMP_DEPTH_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(n, DUMP_DEPTH_SAMPLE, replace=False))
            idx = torch.from_numpy(idx).to(params[0].device)
        for name, ts in arrays.items():
            v = torch.cat([t.detach().reshape(-1).float() for t in ts])
            if idx is not None:
                v = v[idx]
            np.save(os.path.join(out_dir, '%s_%s.npy' % (tag, name)), v.cpu().numpy())


def roofline_reproject(pairs, hbm_peak, peak_kind):
    """Fused re-projection kernels on a batch >> L2 (pairs x 344 KB x 8 tensors), L2 flushed between launches,
    CUDA events on the launching (current) stream."""
    import torch
    from dvd_b200 import ops, synthetic
    dev = torch.device('cuda', torch.cuda.current_device())
    one = synthetic.make_batch([(4, 8)], H=H, W=W, seed=0, leading_dim=False)
    rep = lambda t: t.to(dev).repeat(pairs, *([1] * (t.dim() - 1))).contiguous()  # noqa: E731
    flow, mask = rep(one['flow_1_2']), rep(one['mask_2'].reshape(1, H, W))
    poses = rep(ops.pack_poses_from_batch({k: v for k, v in one.items() if torch.is_tensor(v)}))
    d1, d2 = rep(synthetic.make_depths(1, H, W, seed=1)), rep(synthetic.make_depths(1, H, W, seed=2))
    sf = torch.randn(pairs, 3, H, W, device=dev) * 0.05
    cfg = ops.make_loss_cfg()
    flush = torch.zeros(64 << 20, dtype=torch.int32, device=dev)   # 256 MB, flushed by READING it (clean L2 lines)
    px = pairs * H * W
    scal = ops.reproject_loss_fwd(d1, d2, flow, mask, sf, poses, cfg)
    P = ops.unproject_fwd(d1, poses, 1)
    cases = [('unproject_fwd_kernel', lambda: ops.unproject_fwd(d1, poses, 1), 16),
             ('reproject_loss_fwd_kernel', lambda: ops.reproject_loss_fwd(d1, d2, flow, mask, sf, poses, cfg), 32),
             ('reproject_loss_bwd_kernel', lambda: ops.reproject_loss_bwd(d1, d2, flow, mask, sf, poses, cfg, scal), 48),
             ('unproject_bwd_kernel', lambda: ops.unproject_bwd(P, poses, 1), 16)]
    out = []
    for name, fn, bpp in cases:
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        # every iteration is enqueued behind a ~20 ms spin kernel before the one synchronisation, so the host side of
        # the call (ctypes + output allocation, ~50 us) runs ahead of the GPU and the event pair brackets device work only
        torch.cuda._sleep(40_000_000)
        evs = []
        for _ in range(10):
            flush_sink = flush.sum()   # read 256 MB: evicts L2 without leaving dirty lines behind
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        ts = [a.elapsed_time(b) * 1e-3 for a, b in evs]
        t = sum(ts) / len(ts)
        out.append({'kernel': name, 'bytes_per_px': bpp, 'us': t * 1e6, 'achieved': px * bpp / t / 1e9,
                    'frac': px * bpp / t / 1e9 / hbm_peak})
    # DRAM traffic per pixel from the committed ncu pass (profiles/r1_ncu_reproject_variants.txt: dram__bytes_read.sum +
    # dram__bytes_write.sum of one 64-pair launch / 5 505 024 px): no re-reads.
    ncu_bpp = {'reproject_loss_fwd_kernel': 32.7, 'reproject_loss_bwd_kernel': 46.3}
    tot_t = sum(k['us'] for k in out) * 1e-6
    dom = max(out[1:3], key=lambda k: k['us'])
    return {'bound': 'hbm', 'kernel': dom['kernel'], 'achieved': dom['achieved'], 'peak': hbm_peak, 'unit': 'GB/s',
            'frac': dom['frac'], 'traffic': ncu_bpp[dom['kernel']] * px, 'traffic_unit': 'bytes/launch (ncu DRAM read+write)',
            'algorithmic_bytes': dom['bytes_per_px'] * px, 'peak_kind': peak_kind,
            'note': 'whole C-ABI call between the events (memset of g_depth_2 + pose staging + kernel); kernel alone under ncu: bwd 105 us, fwd 52 us '
                    '(profiles/r1_ncu_reproject_variants.txt); the scatter-add of g_depth_2 (4 reductions / px) is ~1/3 of the backward (DESIGN.md 4.1)',
            'how': 'CUDA events in bench.py, %d pairs per launch (%.0f MB algorithmic traffic), 256 MB L2 flush between launches'
                   % (pairs, px * dom['bytes_per_px'] / 1e6),
            'chain_112B_per_px': {'achieved': px * 112 / tot_t / 1e9, 'frac': px * 112 / tot_t / 1e9 / hbm_peak},
            'kernels': out}


def roofline_mlp(tflops_peak, peak_kind, pairs=2, n_eval=2):
    """tcgen05 scene-flow MLP kernels, CUDA events. Useful work = 593 408 FLOP per pixel and evaluation
    (SURVEY.md 8(d)) for the forward, the same again for dgrad and for wgrad; the bf16x3 split issues 3x as many
    tensor-core MACs (reported as `issued`)."""
    import torch
    from dvd_b200 import ops
    from oracle import sf_mlp
    dev = torch.device('cuda', torch.cuda.current_device())
    layers = sf_mlp.init_layers(seed=1)
    ws = [w.to(dev).contiguous() for w, _ in layers]
    bs = [b.to(dev).contiguous() for _, b in layers]
    cfg = ops.make_mlp_cfg()
    pk = ops.PackedMlp(cfg, dev).refresh(ws, bs)
    p = (torch.randn(pairs, 3, H, W) * 3).to(dev)
    t = torch.full((pairs, 1, H, W), 0.25, device=dev)
    flops = 593408.0 * pairs * H * W * n_eval

    def ev(fn, iters=5):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) * 1e-3 / iters
    t_inf = ev(lambda: ops.mlp_chain_fwd(pk, p, t, 1 / 80, n_eval, n_eval, save=False, want_steps=False))
    f = ops.mlp_chain_fwd(pk, p, t, 1 / 80, n_eval, n_eval, save=True)
    gw = [torch.zeros_like(w) for w in ws]
    gb = [torch.zeros_like(b) for b in bs]
    g = torch.randn_like(p)
    t_bwd = ev(lambda: ops.mlp_chain_bwd(pk, f, t, 1 / 80, n_eval, g, None, gw, gb))
    t_trn = ev(lambda: ops.mlp_chain_fwd(pk, p, t, 1 / 80, n_eval, n_eval, save=True))
    useful = flops / t_inf / 1e12
    return {'bound': 'tensor', 'kernel': 'mlp_chain_fwd_kernel (inference variant)', 'achieved': useful, 'unit': 'TFLOP/s',
            'achieved_kind': 'useful fp32-equivalent FLOPs', 'issued_bf16_tflops': 3 * useful, 'peak': tflops_peak,
            'peak_kind': peak_kind + ' dense bf16 (cuBLAS)', 'frac': 3 * useful / tflops_peak,
            'how': 'CUDA events, %d pairs x %d Euler steps at %dx%d' % (pairs, n_eval, W, H),
            'train_fwd_tflops': flops / t_trn / 1e12, 'bwd_dgrad_plus_wgrad_tflops': 2 * flops / t_bwd / 1e12}


def roofline_depth_convs(model, batch, epoch, tflops_peak, peak_kind):
    """Live roofline of the tensor-core convolution kernels of the step (the kernels that dominate it): one more optimisation
    step with every conv2d_tc / conv_wgrad launch bracketed by CUDA events on the launching stream (dvd_b200.conv_ops.PROFILE);
    achieved = sum of algorithmic FLOPs / sum of launch durations per kernel; TF32 dense peak = measured bf16 peak / 2."""
    import torch
    from dvd_b200 import conv_ops
    conv_ops.PROFILE = []
    graph_flag = getattr(model.opt, 'cuda_graph', True)
    model.opt.cuda_graph = False          # the probe brackets individual launches: run this one step eagerly,
    world_flag = model._world             # on this rank alone (the other ranks have left: no gradient exchange),
    model._world = 1
    overlap_flag = os.environ.get('DVD_BWD_OVERLAP')
    os.environ['DVD_BWD_OVERLAP'] = '0'   # and on one stream (concurrent launches would be billed each other's time)
    try:
        model._train_on_batch(epoch, 0, batch)
        torch.cuda.synchronize()
        rec = conv_ops.PROFILE
    finally:
        conv_ops.PROFILE = None
        model.opt.cuda_graph = graph_flag
        model._world = world_flag
        if overlap_flag is None:
            del os.environ['DVD_BWD_OVERLAP']
        else:
            os.environ['DVD_BWD_OVERLAP'] = overlap_flag
    agg = {}
    for kind, flops, e0, e1, _info in rec:
        a = agg.setdefault(kind, [0.0, 0.0, 0])
        a[0] += flops
        a[1] += e0.elapsed_time(e1) * 1e-3
        a[2] += 1
    peak = tflops_peak / 2
    kern = {'fwd': 'conv2d_tc_kernel (forward)', 'dgrad': 'conv2d_tc_kernel (data gradient)', 'wgrad': 'conv_wgrad_kernel'}
    parts = []
    for k in ('fwd', 'dgrad', 'wgrad'):
        if k in agg and agg[k][1] > 0:
            f, t, n = agg[k]
            parts.append({'kernel': kern[k], 'launches': n, 'gflop': f / 1e9, 'ms': t * 1e3, 'achieved': f / t / 1e12, 'frac': f / t / 1e12 / peak})
    tot_f = sum(a[0] for a in agg.values())
    tot_t = sum(a[1] for a in agg.values())
    dom = max(parts, key=lambda q: q['ms']) if parts else None
    return {'bound': 'tensor', 'kernel': dom['kernel'] if dom else None, 'achieved': dom['achieved'] if dom else None, 'peak': peak,
            'unit': 'TFLOP/s', 'frac': dom['frac'] if dom else None, 'traffic': None, 'peak_kind': peak_kind + ' dense bf16 (cuBLAS) / 2 = TF32',
            'how': 'CUDA events around every tensor-core convolution launch of one %d-pair step (MiDaS, %dx%d): algorithmic FLOPs '
                   '(2*N*OH*OW*Cout*Cin/groups*k*k per pass) / event time, summed per kernel' % (batch['img_1'].shape[-4], W, H),
            'all_conv_kernels': {'achieved': tot_f / tot_t / 1e12 if tot_t else None, 'frac': tot_f / tot_t / 1e12 / peak if tot_t else None,
                                 'ms_per_step': tot_t * 1e3, 'gflop_per_step': tot_f / 1e9},
            'kernels': parts}


def run_b200_arm(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise RuntimeError('bench.py --impl b200 needs a GPU: dvd_b200 has no CPU fallback')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    from dvd_b200 import ops, synthetic
    from dvd_b200.models import get_model
    opt = synthetic.default_opt(batch_size=1, multiprocess_distributed=world > 1, global_rank=rank)
    model = get_model('scene_flow_motion_field')(opt, None)
    synthetic.seed_net_(model.net_depth, 0, 2000.0)
    synthetic.seed_net_(model.net_sceneflow, 1)
    model.to(dev)
    if world > 1:
        model.sync_parameters(0)
    B, K, Wm = args.pairs, args.steps, args.warmup
    EPOCH = opt.warm_sf + 1   # joint phase

    def make_batches(Bp, total_steps):
        host = []
        for s_ in range(total_steps):
            gap, pairs = step_pairs(s_, rank, world, Bp)
            b = synthetic.make_batch(pairs, H=H, W=W, n_frames=N_FRAMES, seed=1000 * rank + s_)
            host.append({k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in b.items()})
        resident = [{k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in hb.items()} for hb in host]
        for rb, hb in zip(resident, host):   # keep the scalar metadata readable on the host without a sync
            rb['time_step'] = hb['time_step']
            rb['steps_hint'] = int(round(float(hb['frame_id_2'].reshape(-1)[0] - hb['frame_id_1'].reshape(-1)[0])))
        return host, resident

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(batches, n_warm, n_steps, sampler=None):
        # untimed preparation before the W warm-up steps: every step signature (pairs x gap) of the region is run often enough for
        # its CUDA graph to exist (Model._graph_step: 2 eager steps, then capture), so that no capture falls into the timed region
        sigs = {}
        for s_ in range(n_warm + n_steps):
            sigs.setdefault(GAPS[s_ % len(GAPS)], s_)
        for _rep in range(3):
            for s_ in sigs.values():
                model._train_on_batch(EPOCH, s_, batches[s_])
        for s_ in range(n_warm):
            model._train_on_batch(EPOCH, s_, batches[s_])
        barrier()
        if sampler:
            sampler.start()
        ops.LAUNCHES['n'] = 0
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        torch.cuda.profiler.start()      # cudaProfilerStart: `ncu --profile-from-start off` lists exactly the timed launches
        logs = [model._train_on_batch(EPOCH, n_warm + s_, batches[n_warm + s_]) for s_ in range(n_steps)]
        torch.cuda.profiler.stop()
        b.record()
        barrier()
        clocks = sampler.stop() if sampler else None
        t = a.elapsed_time(b) * 1e-3
        if world > 1:
            tt = torch.tensor([t], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t = float(tt)
        return t, logs, clocks, ops.LAUNCHES['n']

    host, resident = make_batches(B, Wm + K)
    # (1) device-resident inputs: the headline `value`
    t_dev, logs, clocks, launches = timed(resident, Wm, K, ClockSampler(local))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, logs[-1], model)
    # (2) end to end through the plug-in call with HOST (pinned) batches: H2D + D2H inside the timed region
    t_e2e, logs2, _, _ = timed(host, Wm, K)
    h2d = sum(v.numel() * v.element_size() for v in host[Wm].values() if torch.is_tensor(v))
    d2h = 9 * 4
    # (3) the reference's own schedule: ONE pair per step (train_sequence.sh:29-34), same gap cycle
    b1 = None
    if not args.no_extras and B != 1:
        host1, res1 = make_batches(1, Wm + K)
        t1_dev, _, _, l1 = timed(res1, Wm, K)
        t1_e2e, _, _, _ = timed(host1, Wm, K)
        b1 = {'value': K * world / t1_dev, 'unit': UNIT, 'ms_per_step': 1e3 * t1_dev / K, 'steps': K,
              'e2e': K * world / t1_e2e, 'gpu_launches_per_step': l1 / K,
              'what': 'this arm at 1 pair per step per GPU (the batch the reference DataLoader delivers), same gap cycle'}
        del host1, res1
    if rank != 0:
        if world > 1:
            model.release_graphs()      # NCCL cannot destroy a communicator while graphs that captured its collectives are alive
            dist.destroy_process_group()
        return
    hbm_peak, tflops_peak, peak_kind = measured_peaks()
    pairs_total = K * B * world
    value = pairs_total / t_dev
    roof_conv = roof = roof_mlp = gref = None
    if not args.no_extras:
        roof_conv = roofline_depth_convs(model, resident[Wm], EPOCH, tflops_peak, peak_kind)
        roof = roofline_reproject(args.roofline_pairs, hbm_peak, peak_kind)
        roof_mlp = roofline_mlp(tflops_peak, peak_kind)
        del host, resident
        torch.cuda.empty_cache()
        if world == 1:
            gref = gpu_eager_reference(dev, B, n_steps=K)
            if 'pairs_per_step_%d' % B in gref:
                gref['speedup_value_vs_eager_same_batch'] = value / gref['pairs_per_step_%d' % B]
                gref['speedup_value_vs_eager_1_pair_per_step'] = value / gref['pairs_per_step_1']
                if b1:
                    gref['speedup_b1_vs_eager_1_pair_per_step'] = b1['value'] / gref['pairs_per_step_1']
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference_steps(len(GAPS), 0)   # bounded sample: one step per gap of the schedule, ~20-30 s of CPU work
    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': K, 'warmup': Wm,
        'ms_per_step': 1e3 * t_dev / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32 storage; depth-CNN convolutions TF32 on tcgen05 (operands RN-rounded, fp32 accumulate = the reference\'s GPU default); '
                 'MLP GEMMs bf16x3-split on tcgen05 (fp32-grade, err ~2e-5); re-projection, stem, head, Adam fp32',
        'data': 'synthetic',
        'config': {'workload': workload_name(), 'height': H, 'width': W, 'frames': N_FRAMES, 'gaps': list(GAPS),
                   'pairs_per_step_per_gpu': B, 'global_pairs_per_step': B * world, 'parallelism': 'dp%d' % world,
                   'l2': 'per-step working set (depth-net activations of %d images + saved MLP activations, several GB) >> 126 MB L2; '
                         'no explicit flush' % (2 * B)},
        'clocks': clocks,
        'e2e': {'value': pairs_total / t_e2e, 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                'ms_per_step': 1e3 * t_e2e / K, 'api': 'Model._train_on_batch(epoch, i, pinned-host batch dict)'},
        'gpu_launches': launches,
        'b1': b1,
        'gpu_reference': gref,
        'roofline': roof_conv,
        'roofline_reproject': roof,
        'roofline_mlp': roof_mlp,
        'cpu_baseline': cpu,
        'last_batch_log': {k: v for k, v in logs[-1].items() if isinstance(v, (int, float))},
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        model.release_graphs()
        dist.destroy_process_group()


def main():
    args = parse()
    configure(args)
    if args.impl == 'reference':
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == '__main__':
    main()
