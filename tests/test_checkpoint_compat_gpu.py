"""Checkpoint hand-over with the reference (models/netinterface.py:528-574): a file in the reference's layout - net state dicts
under the reference's parameter names plus `torch.optim.Adam.state_dict()`s, exactly what `NetInterface.save_state_dict` writes -
is loaded into the dvd_b200 Model; the next Adam step on the flat buffers then equals torch.optim.Adam's on the same gradient, and
the state written back is loadable by torch.optim.Adam again. (The file is produced here with torch itself;
tests/test_oracle_vs_reference.py::test_reference_written_checkpoint_loads does the same with the layout of a file written by the
reference's own NetInterface.)"""
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.timeout(600)
def test_reference_layout_checkpoint_loads_and_steps_like_torch_adam(tmp_path):
    from dvd_b200 import synthetic
    from dvd_b200.models import get_model
    from dvd_b200.networks.sceneflow_field import SceneFlowFieldNet
    from dvd_b200.third_party.MiDaS import MidasNet
    lr, betas = 1e-4, (0.5, 0.9)
    nets = [synthetic.seed_net_(MidasNet(non_negative=True, normalize_input=True), 3, 2000.0),
            synthetic.seed_net_(SceneFlowFieldNet(net_width=256, n_layers=4, time_dependent=True, N_freq_xyz=16, N_freq_t=16), 4)]
    opts = [torch.optim.Adam(n.parameters(), lr=lr * (1 if i == 0 else 1000), betas=betas) for i, n in enumerate(nets)]
    g = torch.Generator().manual_seed(0)
    for _ in range(2):                        # two reference-side steps so that exp_avg / exp_avg_sq / step are non-trivial
        for n, o in zip(nets, opts):
            for p in n.parameters():
                p.grad = torch.randn(p.shape, generator=g) * 1e-3
            o.step()
    f = str(tmp_path / 'ref_layout.pt')
    torch.save({'nets': [n.state_dict() for n in nets], 'optimizers': [o.state_dict() for o in opts], 'epoch': 7}, f)

    model = get_model('scene_flow_motion_field')(synthetic.default_opt(lr=lr), None)
    extra = model.load_state_dict(f)
    assert extra == {'epoch': 7}
    model.to(torch.device('cuda:0'))
    for mine, ref in zip(model._nets, nets):
        for (k, a), (k2, b) in zip(mine.state_dict().items(), ref.state_dict().items()):
            assert k == k2 and torch.equal(a.cpu(), b), k
    assert model.optimizer_depth.adam.step_count == 2 and model.optimizer_scene.adam.step_count == 2
    # one more step on both sides with the same gradient
    for n, o, mo in zip(nets, opts, model._optimizers):
        grads = [torch.randn(p.shape, generator=g) * 1e-3 for p in n.parameters()]
        for p, gr in zip(n.parameters(), grads):
            p.grad = gr
        o.step()
        mo.zero_grad()
        for p, gr in zip(mo.flat.params, grads):
            p.grad.copy_(gr)
        mo.step()
    torch.cuda.synchronize()
    for mine, ref in zip(model._nets, nets):
        for (k, a), (_, b) in zip(mine.named_parameters(), ref.named_parameters()):
            err = float((a.detach().cpu() - b.detach()).abs().max())
            assert err <= 2e-7 + 1e-6 * float(b.detach().abs().max()), (k, err)
    # and back: the optimiser state this Model writes loads into torch.optim.Adam
    f2 = str(tmp_path / 'back.pt')
    model.save_state_dict(f2, save_optimizer=True, additional_values={'epoch': 8})
    sd = torch.load(f2, map_location='cpu', weights_only=False)
    for n, o, s in zip(nets, opts, sd['optimizers']):
        ref_state = o.state_dict()['state']
        for i in ref_state:
            assert int(float(s['state'][i]['step'])) == 3
            for key in ('exp_avg', 'exp_avg_sq'):
                a, b = s['state'][i][key], ref_state[i][key]
                assert a.shape == b.shape and float((a - b).abs().max()) <= 1e-9 + 1e-5 * float(b.abs().max()), (i, key)
        o2 = torch.optim.Adam(n.parameters(), lr=lr, betas=betas)
        s2 = dict(s)
        s2['param_groups'] = o.state_dict()['param_groups']
        o2.load_state_dict(s2)
