"""TEST INFRASTRUCTURE — generates tests/golden/*.pt by executing the UNMODIFIED reference
(/root/reference, imported through oracle/ref_harness.py) on seeded synthetic inputs.

Run where the reference tree is available:   python -m oracle.gen_golden [reproject|mlp|modules|step|all]
The fixtures are small (tens of KB .. a few MB) and committed; the GPU box never sees /root/reference.
Tensors are stored channel-planar ([B,C,H,W]) to match the C ABI layout.
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import ref_harness  # noqa: E402

GOLD = os.path.join(ROOT, 'tests', 'golden')


def _cf(x):  # [B,H,W,1,C] -> [B,C,H,W]
    return x.squeeze(3).permute(0, 3, 1, 2).contiguous()


def reproject_inputs(B=2, H=24, W=32, seed=0, dtype=torch.float32):
    from dvd_b200 import synthetic
    pairs = [(3, 5), (10, 18), (40, 41), (7, 13)][:B]
    batch = synthetic.make_batch(pairs, H=H, W=W, seed=seed, dtype=dtype, leading_dim=False, flow_sigma=4.0)
    d1 = synthetic.make_depths(B, H, W, seed=seed + 1, dtype=dtype)
    d2 = synthetic.make_depths(B, H, W, seed=seed + 2, dtype=dtype)
    # exercise every branch: depth >= 100 (mask), warped z >= 100, projected z < 1e-3, clamp(1e-3)
    d1[0, 0, :3, :5] = 150.0
    d2[B - 1, 0, 5:9, 5:11] = 250.0
    d1[B - 1, 0, 10:12, :] = -1.0
    d2[0, 0, 14:16, 3:9] = 5e-4
    g = torch.Generator().manual_seed(seed + 3)
    sf = (torch.randn(B, 3, H, W, generator=g, dtype=torch.float64) * 0.05).to(dtype)
    return batch, d1, d2, sf


def run_reference_reproject(ns, model, batch, d1, d2, sf, *, warm, use_disp, use_disp_ratio, midas,
                            flow_mul=1.0, disp_mul=1.0):
    """flow_by_depth + scene_flow_projection_slack + Model._calc_loss, exactly as
    Model._predict_on_batch / _calc_loss chain them (smf.py:240-264,285-324)."""
    d1 = d1.clone().requires_grad_()
    d2 = d2.clone().requires_grad_()
    sf = sf.clone().requires_grad_()
    fb, sl = ns.sfp.flow_by_depth(), ns.sfp.scene_flow_projection_slack()
    if d1.dtype == torch.float64:
        H, W = d1.shape[-2:]
        yy, xx = torch.meshgrid(torch.arange(H).double(), torch.arange(W).double(), indexing='ij')
        coord = torch.ones([1, H, W, 1, 3], dtype=torch.float64)
        coord[0, ..., 0, 0] = xx
        coord[0, ..., 0, 1] = yy
        fb.coord = coord
        sl.coord = coord.clone()
    pose = {k: batch[k] for k in ('R_1', 'R_2', 'R_1_T', 'R_2_T', 't_1', 't_2', 'K', 'K_inv')}
    dflow = fb(depth_1=d1, depth_2=d2, flow_1_2=batch['flow_1_2'], **pose)
    sfl = sf.permute(0, 2, 3, 1)[..., None, :]
    res = sl(depth_1=d1, depth_2=d2, flow_1_2=batch['flow_1_2'], flow_2_1=batch['flow_2_1'],
             sflow_1_2=sfl, sflow_2_1=sfl, **pose)
    res['sf_1_2'] = sf
    res['sf_by_dep_1_2'] = dflow['sf_by_depth']
    model.opt.use_disp, model.opt.use_disp_ratio, model.opt.midas = use_disp, use_disp_ratio, midas
    model.opt.flow_mul, model.opt.disp_mul = flow_mul, disp_mul
    model.warm = warm
    model._input.mask_2 = batch['mask_2']
    model._input.flow_1_2 = batch['flow_1_2']
    loss, loss_data = model._calc_loss(res)
    gd1, gd2, gsf = torch.autograd.grad(loss, [d1, d2, sf], allow_unused=True)
    tensors = {
        'global_p1': _cf(dflow['global_p1']), 'sf_by_depth': _cf(dflow['sf_by_depth']),
        'warped_global_p2': _cf(dflow['warped_global_p2']),
        'warped_p2_camera_2': _cf(res['warped_p2_camera_2']), 'p1_camera_2': _cf(res['p1_camera_2']),
        'dflow_1_2': res['dflow_1_2'].permute(0, 3, 1, 2).contiguous(),
        'staticflow_1_2': res['staticflow_1_2'].permute(0, 3, 1, 2).contiguous(),
        'depth_image_1_2': res['depth_image_1_2'].contiguous(), 'depth_warp_1_2': res['depth_warp_1_2'].contiguous(),
    }
    tensors = {k: v.detach() for k, v in tensors.items()}
    zero = lambda g, like: torch.zeros_like(like) if g is None else g  # noqa: E731
    return {'tensors': tensors, 'loss': float(loss), 'loss_data': {k: float(v) for k, v in loss_data.items()},
            'g_d1': zero(gd1, d1).detach(), 'g_d2': zero(gd2, d2).detach(), 'g_sf': zero(gsf, sf).detach()}


LOSS_MODES = {
    'joint_disp': dict(warm=False, use_disp=True, use_disp_ratio=False, midas=True),
    'warm_disp': dict(warm=True, use_disp=True, use_disp_ratio=False, midas=True, flow_mul=2.0, disp_mul=0.5),
    'joint_sf': dict(warm=False, use_disp=False, use_disp_ratio=False, midas=True),
    'joint_ratio_nomidas': dict(warm=False, use_disp=False, use_disp_ratio=True, midas=False),
}


def _light_model(ns):
    """A reference Model shell good enough for _calc_loss (no networks needed)."""
    m = ns.smf.Model.__new__(ns.smf.Model)
    m.opt = ref_harness.default_opt()
    m._input = lambda: None
    from functools import partial
    import torch.nn.functional as F
    m.L1_crit = partial(F.l1_loss, reduction='none')
    m.L2_crit = partial(F.mse_loss, reduction='none')
    return m


def gen_reproject():
    ns = ref_harness.import_reference()
    model = _light_model(ns)
    batch, d1, d2, sf = reproject_inputs()
    out = {'inputs': {'batch': {k: v for k, v in batch.items() if torch.is_tensor(v)}, 'd1': d1, 'd2': d2, 'sf': sf},
           'modes': {}}
    for name, kw in LOSS_MODES.items():
        out['modes'][name] = run_reference_reproject(ns, model, batch, d1, d2, sf, **kw)
        out['modes'][name]['kw'] = kw
    # tensors are mode-independent; keep one copy
    out['tensors'] = out['modes']['joint_disp']['tensors']
    for m in out['modes'].values():
        del m['tensors']
    torch.save(out, os.path.join(GOLD, 'reproject_golden.pt'))
    print('wrote reproject_golden.pt', {k: v['loss'] for k, v in out['modes'].items()})


def mlp_inputs(B=2, H=16, W=24, seed=5, dtype=torch.float32):
    from dvd_b200 import synthetic
    from oracle import geometry
    batch = synthetic.make_batch([(3, 5), (20, 28)][:B], H=H, W=W, seed=seed, dtype=dtype, leading_dim=False)
    d1 = synthetic.make_depths(B, H, W, seed=seed + 1, dtype=dtype)
    R1, R2, t1, t2, K, Kinv = geometry._poses(batch)
    P1 = geometry.unproject(d1, R1, t1, Kinv)
    return P1.contiguous(), batch['time_stamp_1'].contiguous(), float(batch['time_step'])


def gen_mlp():
    ns = ref_harness.import_reference()
    torch.manual_seed(11)
    net = ns.sff.SceneFlowFieldNet(net_width=256, n_layers=4, time_dependent=True, N_freq_xyz=16, N_freq_t=16)
    # reference init: kaiming_normal_(a=0.2), bias 0 (smf.py:123, netinterface.py:55-84); biases are then
    # perturbed so that the bias path is exercised by the parity test.
    ns.smf.Model.init_weight(None, net, 'kaiming', 0.01, a=0.2)
    with torch.no_grad():
        for p in net.parameters():
            if p.dim() == 1:
                p.normal_(0, 0.05)
    P1, ts, dt = mlp_inputs()
    model = ns.smf.Model.__new__(ns.smf.Model)
    model.opt = ref_harness.default_opt()
    model.net_sceneflow = net
    out = {'state_dict': {k: v.clone() for k, v in net.state_dict().items()}, 'P1': P1, 'ts': ts, 'dt': dt}
    # single eval (raw network output)
    p = P1.clone().requires_grad_()
    raw = net(p, ts)
    out['raw'] = raw.detach()
    # multi-step, steps=3, with gradients w.r.t. p and all weights for a fixed cotangent
    g = torch.Generator().manual_seed(3)
    cot = torch.randn(P1.shape, generator=g)
    # zero the cotangent on pixels that sit on a LeakyReLU kink (see oracle/sf_mlp.py: kink_band)
    from oracle import sf_mlp
    band = sf_mlp.kink_band(P1, ts, dt, 3, sf_mlp.layers_from_state_dict(net.state_dict()))
    cot = cot * (~band).unsqueeze(1).float()
    out['kink_band_pixels'] = int(band.sum())
    for steps in (1, 3):
        net.zero_grad()
        p = P1.clone().requires_grad_()
        sf = model.forward_sf_net_multi_step(p, ts, time_step=dt, steps=steps)
        (sf * cot).sum().backward()
        out['multi_%d' % steps] = {'sf': sf.detach(), 'g_p': p.grad.clone(),
                                   'g_w': {k: v.grad.clone() for k, v in net.named_parameters()}}
    out['cot'] = cot
    # acceleration regulariser (smf.py:326-344)
    net.zero_grad()
    p = P1.clone().requires_grad_()
    model._input = lambda: None
    model._input.time_stamp_1 = ts
    model._input.time_step = torch.tensor(dt)
    model.opt.acc_mul = 1.0
    val = model._opt_reg({'global_p1': p}, steps=5)
    out['acc_reg'] = {'value': val, 'g_p': p.grad.clone(), 'g_w': {k: v.grad.clone() for k, v in net.named_parameters()}}
    # the same regulariser restricted to the pixels off the kink band (what the gradient parity test uses):
    net.zero_grad()
    p = P1.clone().requires_grad_()
    keep = (~band).unsqueeze(1).float()
    s0 = model.forward_sf_net(p, ts)
    s1 = model.forward_sf_net(p + s0, ts + dt)
    val_k = (keep * (s1 - s0).abs()).sum() / (s0.numel() + 1e-6)
    val_k.backward()
    out['acc_reg_keep'] = {'keep': keep, 'value': float(val_k), 'g_p': p.grad.clone(),
                           'g_w': {k: v.grad.clone() for k, v in net.named_parameters()}}
    torch.save(out, os.path.join(GOLD, 'mlp_golden.pt'))
    print('wrote mlp_golden.pt acc_reg=%g |sf|max=%g' % (val, out['multi_3']['sf'].abs().max()))


def geometry_inputs(dtype):
    """Inputs of the module-level geometry comparison (tests/test_oracle_vs_reference.py), all from seeds; the float32 set is
    the float64 set rounded."""
    from dvd_b200 import synthetic
    B, H, W = 2, 40, 56
    b = synthetic.make_batch([(3, 5), (10, 18)], H=H, W=W, dtype=dtype, leading_dim=False, flow_sigma=6.0)
    d1 = synthetic.make_depths(B, H, W, seed=1, dtype=dtype)
    d2 = synthetic.make_depths(B, H, W, seed=2, dtype=dtype)
    d1[0, 0, :3, :5] = 150.0
    d1[1, 0, 10:12, :] = -1.0
    sf = (torch.randn(B, 3, H, W, generator=torch.Generator().manual_seed(3), dtype=torch.float64) * 0.05).to(dtype)
    return b, d1, d2, sf


def depth_net_input():
    return torch.rand(2, 3, 64, 96, generator=torch.Generator().manual_seed(4))


def mlp_inputs_small():
    g = torch.Generator().manual_seed(5)
    return torch.randn(1, 3, 9, 11, generator=g) * 3, torch.full((1, 1, 9, 11), 0.4)


# checkpoint skeleton: tensors above this size are stored as (shape, dtype) and refilled from a seed by the test
SKELETON_MAX_NUMEL = 16


def checkpoint_skeleton(obj):
    """Everything of a checkpoint except the values of its large tensors: containers, keys, order, small tensors verbatim."""
    if torch.is_tensor(obj):
        if obj.numel() > SKELETON_MAX_NUMEL:
            return ('seeded_tensor', tuple(obj.shape), str(obj.dtype).replace('torch.', ''))
        return obj.clone()
    if isinstance(obj, dict):
        return {k: checkpoint_skeleton(v) for k, v in obj.items()}
    if isinstance(obj, (list, tuple)):
        return type(obj)(checkpoint_skeleton(v) for v in obj)
    return obj


def checkpoint_from_skeleton(obj, g):
    """Inverse of checkpoint_skeleton: large tensors refilled, in traversal order, from generator `g` (second moments >= 0)."""
    if isinstance(obj, tuple) and len(obj) == 3 and obj[0] == 'seeded_tensor':
        t = torch.randn(obj[1], generator=g, dtype=torch.float64)
        return t.to(getattr(torch, obj[2]))
    if isinstance(obj, dict):
        return {k: (checkpoint_from_skeleton(v, g).abs() if k == 'exp_avg_sq' else checkpoint_from_skeleton(v, g))
                for k, v in obj.items()}
    if isinstance(obj, (list, tuple)):
        return type(obj)(checkpoint_from_skeleton(v, g) for v in obj)
    return obj


def gen_reference_modules():
    """Outputs of the reference's own modules that tests/test_oracle_vs_reference.py compares the oracle and the mirrors with."""
    import tempfile
    from dvd_b200 import synthetic
    ns = ref_harness.import_reference()
    # geometry modules: flow_by_depth + scene_flow_projection_slack, float32 and float64
    for dtype in (torch.float32, torch.float64):
        b, d1, d2, sf = geometry_inputs(dtype)
        H, W = d1.shape[-2:]
        fb, sl = ns.sfp.flow_by_depth(), ns.sfp.scene_flow_projection_slack()
        if dtype == torch.float64:
            yy, xx = torch.meshgrid(torch.arange(H).double(), torch.arange(W).double(), indexing='ij')
            coord = torch.ones([1, H, W, 1, 3], dtype=dtype)
            coord[0, ..., 0, 0], coord[0, ..., 0, 1] = xx, yy
            fb.coord, sl.coord = coord, coord.clone()
        pose = {k: b[k] for k in ('R_1', 'R_2', 'R_1_T', 'R_2_T', 't_1', 't_2', 'K', 'K_inv')}
        r1 = fb(depth_1=d1, depth_2=d2, flow_1_2=b['flow_1_2'], **pose)
        sfl = sf.permute(0, 2, 3, 1)[..., None, :]
        r2 = sl(depth_1=d1, depth_2=d2, flow_1_2=b['flow_1_2'], flow_2_1=b['flow_2_1'], sflow_1_2=sfl, sflow_2_1=sfl, **pose)
        ref = {'global_p1': _cf(r1['global_p1']), 'sf_by_depth': _cf(r1['sf_by_depth']),
               'warped_p2_camera_2': _cf(r2['warped_p2_camera_2']), 'p1_camera_2': _cf(r2['p1_camera_2']),
               'dflow_1_2': r2['dflow_1_2'].permute(0, 3, 1, 2).contiguous(),
               'staticflow_1_2': r2['staticflow_1_2'].permute(0, 3, 1, 2).contiguous(),
               'depth_image_1_2': r2['depth_image_1_2'].contiguous(), 'depth_warp_1_2': r2['depth_warp_1_2'].contiguous()}
        name = 'ref_geometry_%s.pt' % str(dtype).replace('torch.', '')
        torch.save({k: v.detach().clone() for k, v in ref.items()}, os.path.join(GOLD, name))
        print('wrote', name)
    out = {}
    # depth nets with name-seeded weights: parameter names / shapes and outputs
    x = depth_net_input()
    midas = synthetic.seed_net_(ns.midas.MidasNet(path=None, non_negative=True, normalize_input=True), 0, 2000.0).eval()
    hg = synthetic.seed_net_(ns.hourglass.HourglassModel_Embed(noexp=False), 0)
    hg.defrost()
    with torch.no_grad():
        out['midas'] = {'keys': [(k, tuple(v.shape)) for k, v in midas.state_dict().items()], 'out': midas(x.clone())}
        out['hourglass'] = {'keys': [(k, tuple(v.shape)) for k, v in hg.state_dict().items()], 'out': hg(x.clone())}
    # scene-flow MLP with name-seeded weights
    net = synthetic.seed_net_(ns.sff.SceneFlowFieldNet(net_width=256, n_layers=4, time_dependent=True, N_freq_xyz=16,
                                                       N_freq_t=16), 3)
    p, t = mlp_inputs_small()
    with torch.no_grad():
        out['mlp'] = {'keys': [(k, tuple(v.shape)) for k, v in net.state_dict().items()], 'out': net(p, t)}
    # a checkpoint written by the reference's NetInterface.save_state_dict after one optimisation step (hourglass variant)
    opt = ref_harness.default_opt(midas=False, lr=1e-4)
    ref_model, _ = ref_harness.build_reference_model(opt, seed=0)
    batch = synthetic.make_batch([(3, 5)], H=32, W=48, seed=1, smooth_flow=True)
    ref_model._train_on_batch(6, 0, {k: (v.clone() if torch.is_tensor(v) else v) for k, v in batch.items()})
    with tempfile.TemporaryDirectory() as d:
        f = os.path.join(d, 'ref.pt')
        ref_model.save_state_dict(f, save_optimizer=True, additional_values={'epoch': 6})
        out['checkpoint'] = checkpoint_skeleton(torch.load(f, map_location='cpu', weights_only=False))
    torch.save(out, os.path.join(GOLD, 'ref_modules.pt'))
    print('wrote ref_modules.pt')


if __name__ == '__main__':
    what = sys.argv[1] if len(sys.argv) > 1 else 'all'
    os.makedirs(GOLD, exist_ok=True)
    if what in ('reproject', 'all'):
        gen_reproject()
    if what in ('mlp', 'all'):
        gen_mlp()
    if what in ('modules', 'all'):
        gen_reference_modules()
    if what in ('step', 'all'):
        from oracle import gen_golden_step
        gen_golden_step.main()
