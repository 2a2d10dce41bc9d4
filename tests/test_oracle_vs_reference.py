"""CPU: the oracle restatement and the host-side mirrors against outputs of the UNMODIFIED reference code, stored in
tests/golden/ref_*.pt by oracle/gen_golden.py (`python -m oracle.gen_golden modules`, which imports the reference through
oracle/ref_harness.py). Inputs and name-seeded weights are rebuilt here from the same seeds."""
import os

import pytest
import torch

from conftest import GOLDEN, rel_err
from oracle import gen_golden


def _load(name):
    return torch.load(os.path.join(GOLDEN, name), weights_only=False)


@pytest.fixture(scope='module')
def ref_modules():
    return _load('ref_modules.pt')


def _keys(sd):
    return [(k, tuple(v.shape)) for k, v in sd.items()]


@pytest.mark.parametrize('dtype', [torch.float32, torch.float64])
def test_geometry_matches_reference_modules(dtype):
    from oracle import geometry
    b, d1, d2, sf = gen_golden.geometry_inputs(dtype)
    ref = _load('ref_geometry_%s.pt' % str(dtype).replace('torch.', ''))
    o = geometry.reproject(d1, d2, sf, b)
    tol = 5e-6 if dtype == torch.float32 else 1e-12
    for k, v in ref.items():
        assert v.dtype == dtype
        assert rel_err(o[k], v) < tol, k


def test_depth_net_mirrors_and_functional_oracle_match_reference(ref_modules):
    from dvd_b200 import synthetic
    from dvd_b200.third_party import MiDaS as M, hourglass as HG
    from oracle import depth_nets
    x = gen_golden.depth_net_input()
    # name-seeded weights: the same parameter names and shapes as the reference's nets mean the same values
    mine = synthetic.seed_net_(M.MidasNet(non_negative=True, normalize_input=True), 0, 2000.0).eval()
    assert _keys(mine.state_dict()) == ref_modules['midas']['keys']
    a = ref_modules['midas']['out']
    with torch.no_grad():
        # the MiDaS mirror only holds parameters (all of its arithmetic is CUDA: depth_engine.py); on the CPU its state dict
        # drives the functional oracle, and it refuses to run itself
        assert rel_err(depth_nets.midas_forward(mine.state_dict(), x), a) < 1e-5
        with pytest.raises(RuntimeError):
            mine(x)
    mh = synthetic.seed_net_(HG.HourglassModel_Embed(noexp=False), 0)
    assert _keys(mh.state_dict()) == ref_modules['hourglass']['keys']
    mh.defrost()
    a = ref_modules['hourglass']['out']
    with torch.no_grad():
        assert rel_err(mh(x), a) < 1e-6
        assert rel_err(depth_nets.hourglass_forward(mh.state_dict(), x), a) < 1e-5


def test_mlp_oracle_matches_reference_module(ref_modules):
    from dvd_b200 import synthetic
    from dvd_b200.networks.sceneflow_field import SceneFlowFieldNet
    from oracle import sf_mlp
    net = synthetic.seed_net_(SceneFlowFieldNet(net_width=256, n_layers=4, time_dependent=True, N_freq_xyz=16, N_freq_t=16), 3)
    assert _keys(net.state_dict()) == ref_modules['mlp']['keys']
    p, t = gen_golden.mlp_inputs_small()
    with torch.no_grad():
        assert rel_err(sf_mlp.mlp_forward(p, t, sf_mlp.layers_from_state_dict(net.state_dict())), ref_modules['mlp']['out']) < 1e-5


def test_reference_written_checkpoint_loads(ref_modules, tmp_path):
    """A checkpoint in the layout the REFERENCE's own `NetInterface.save_state_dict` (models/netinterface.py:528-536) wrote after
    one of its optimisation steps loads into the dvd_b200 Model: same net keys / values, and its two torch.optim.Adam state dicts
    map onto the flat Adam buffers (exp_avg, exp_avg_sq, step) and come back out identical. Hourglass variant. The fixture keeps
    the file's whole structure (containers, keys, order, which parameters have optimiser state, small tensors); the values of
    the large tensors are refilled from a seed."""
    from dvd_b200 import synthetic
    from dvd_b200.flat import FlatAdam, FlatParams
    from dvd_b200.models import get_model
    ref_sd = gen_golden.checkpoint_from_skeleton(ref_modules['checkpoint'], torch.Generator().manual_seed(0))
    f = str(tmp_path / 'ref.pt')
    torch.save(ref_sd, f)
    mine = get_model('scene_flow_motion_field')(synthetic.default_opt(midas=False, lr=1e-4), None)
    extra = mine.load_state_dict(f)
    assert extra.get('epoch') == 6
    for net, rsd in zip(mine._nets, ref_sd['nets']):
        msd = net.state_dict()
        assert list(msd) == list(rsd)
        for k in rsd:
            assert torch.equal(msd[k], rsd[k]), k
    # optimiser state: reference dict -> flat buffers -> dict (FlatParams / FlatAdam hold plain tensors: works on the CPU too)
    for net, osd in zip(mine._nets, ref_sd['optimizers']):
        adam = FlatAdam(FlatParams(net), 1e-4, (0.5, 0.9))
        adam.load_state_dict(osd)
        back = adam.state_dict()
        # torch.optim.Adam keeps state only for parameters that ever received a gradient (the hourglass has unused layers);
        # the flat optimiser writes (all-zero) moments for the others as well
        assert set(osd['state']) <= set(back['state'])
        for i in set(back['state']) - set(osd['state']):
            assert float(back['state'][i]['exp_avg'].abs().max()) == 0.0 and float(back['state'][i]['exp_avg_sq'].abs().max()) == 0.0
        for i, st in osd['state'].items():
            assert int(float(back['state'][i]['step'])) == int(float(st['step']))
            assert torch.equal(back['state'][i]['exp_avg'], st['exp_avg']) and torch.equal(back['state'][i]['exp_avg_sq'], st['exp_avg_sq'])
