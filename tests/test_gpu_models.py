"""GPU parity of the CALLERS (SURVEY 8(a) rows a8-a10): our KernelNN / KernelInduced / MKGN / MGKN modules,
loaded with the reference modules' parameters, against golden outputs produced by the reference's own model
classes (oracle/gen_golden.py).  pytest -m gpu."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.helpers import GOLDEN, TOL, cfg1_weights, ei64, rel_err, t, vcycle_weights

pytestmark = [pytest.mark.gpu, pytest.mark.usefixtures('edge_kernel_mode')]
DEV = 'cuda:0'


class _Data(object):
    pass


def _load(model, state):
    model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in state.items()})
    return model.to(DEV).eval()


@pytest.mark.parametrize('precision', ['f16', 'fp32'])
def test_kernelnn_full_forward_cfg1(precision):
    from graph_pde_b200.models import KernelNN
    g = np.load(os.path.join(GOLDEN, 'g2_cfg1_ball16.npz'))
    fc1, ws, bs, root, bias = cfg1_weights(g)
    model = KernelNN(32, 1024, 4, 6, in_width=6, precision=precision)
    st = model.state_dict()
    st['fc1.weight'], st['fc1.bias'] = fc1.weight.detach(), fc1.bias.detach()
    for i, l in enumerate((0, 2, 4)):
        st['conv1.nn.layers.%d.weight' % l], st['conv1.nn.layers.%d.bias' % l] = ws[i], bs[i]
    st['conv1.root'], st['conv1.bias'] = root, bias
    st['fc2.weight'], st['fc2.bias'] = t(g['w/fc2.weight']), t(g['w/fc2.bias'])
    model.load_state_dict(st)
    model = model.to(DEV).eval()
    d = _Data()
    d.x, d.edge_index, d.edge_attr = t(g['node_x']).to(DEV), ei64(g['edge_index']).to(DEV), t(g['edge_attr']).to(DEV)
    with torch.no_grad():
        out = model(d)
    assert rel_err(out, t(g['model_out'])) < TOL[precision]


@pytest.mark.parametrize('steps', ['fused', 'plain'])
@pytest.mark.parametrize('variant', ['neurips1', 'general'])
@pytest.mark.parametrize('precision', ['f16', 'fp32'])
def test_mgkn_vcycle(variant, precision, steps, monkeypatch):
    """`steps`: KernelInduced inference chains `residual_step` on pre-activations ('fused', the default) or runs the
    reference's conv / add / ReLU sequence ('plain', NNCONV_B200_FUSED_STEPS=0); both against the reference's output."""
    from graph_pde_b200 import models
    from graph_pde_b200.models import KernelInduced, MKGN
    if steps == 'plain' and variant != 'neurips1':
        pytest.skip('only KernelInduced has the fused step chain')
    monkeypatch.setattr(models, '_FUSED_STEPS', steps == 'fused')
    g = np.load(os.path.join(GOLDEN, 'g4_mgkn_vcycle.npz'))
    pts = [int(p) for p in g['points']]
    cls = KernelInduced if variant == 'neurips1' else MKGN
    model = cls(width=32, ker_width=64, depth=2, ker_in=6, points=pts, level=len(pts), in_width=6,
                precision=precision)
    model = _load(model, vcycle_weights(g, variant))
    d = _Data()
    d.x = t(g['node_x']).to(DEV)
    for nm in ('mid', 'down', 'up'):
        setattr(d, 'edge_index_' + nm, ei64(g['edge_index_' + nm]).to(DEV))
        setattr(d, 'edge_attr_' + nm, t(g['edge_attr_' + nm]).to(DEV))
    d.edge_index_range = torch.from_numpy(g['range_mid']).to(DEV)
    d.edge_index_down_range = torch.from_numpy(g['range_down']).to(DEV)
    d.edge_index_up_range = torch.from_numpy(g['range_up']).to(DEV)
    with torch.no_grad():
        out = model(d)
        out2 = model(d)                       # second call: plans / edge features come from the caches
    assert rel_err(out, t(g[variant + '/out'])) < TOL[precision]
    assert rel_err(out2, t(g[variant + '/out'])) < TOL[precision]


@pytest.mark.parametrize('precision', ['f16', 'fp32'])
def test_mgkn_orthogonal_burgers1d(precision):
    from graph_pde_b200.models import MGKN
    g = np.load(os.path.join(GOLDEN, 'g5_mgkn_burgers1d.npz'))
    model = MGKN(width=32, ker_width=64, depth=2, ker_in=4, in_width=2, s=int(g['s']), precision=precision)
    model = _load(model, {k[2:]: g[k] for k in g.files if k.startswith('w/')})
    n = int(g['n_edge_sets'])
    X = [t(g['X/%d' % l]).to(DEV) for l in range(int(g['n_levels']))]
    eis = [ei64(g['edge_index/%d' % i]).to(DEV) for i in range(n)]
    eas = [t(g['edge_attr/%d' % i]).to(DEV) for i in range(n)]
    with torch.no_grad():
        out = model((X, None, eis, eas))
    assert rel_err(out, t(g['out'])) < TOL[precision]


def test_cuda_graph_replay_of_kernelnn_and_vcycle():
    """SURVEY 8(f2): the whole forward replayed from a CUDA graph gives the eager result; refreshed static inputs
    are picked up."""
    from graph_pde_b200 import GraphedForward
    from graph_pde_b200.models import KernelInduced, KernelNN
    g = np.load(os.path.join(GOLDEN, 'g2_cfg1_ball16.npz'))
    torch.manual_seed(0)
    model = KernelNN(32, 64, 3, 6, in_width=6).to(DEV).eval()
    d = _Data()
    d.x, d.edge_index, d.edge_attr = t(g['node_x']).to(DEV), ei64(g['edge_index']).to(DEV), t(g['edge_attr']).to(DEV)
    with torch.no_grad():
        eager = model(d).clone()
    gf = GraphedForward(model, d)
    assert rel_err(gf.replay(), eager) < 1e-4      # fp32 atomics: summation order differs run to run
    x2 = torch.randn_like(d.x)
    with torch.no_grad():
        d.x.copy_(x2)
        eager2 = model(d).clone()
    assert rel_err(gf.replay(), eager2) < 1e-4
    assert rel_err(eager2, eager) > 1e-2

    g4 = np.load(os.path.join(GOLDEN, 'g4_mgkn_vcycle.npz'))
    pts = [int(p) for p in g4['points']]
    vm = KernelInduced(width=32, ker_width=64, depth=2, ker_in=6, points=pts, level=len(pts), in_width=6)
    vm = _load(vm, vcycle_weights(g4, 'neurips1'))
    dv = _Data()
    dv.x = t(g4['node_x']).to(DEV)
    for nm in ('mid', 'down', 'up'):
        setattr(dv, 'edge_index_' + nm, ei64(g4['edge_index_' + nm]).to(DEV))
        setattr(dv, 'edge_attr_' + nm, t(g4['edge_attr_' + nm]).to(DEV))
    dv.edge_index_range = torch.from_numpy(g4['range_mid']).to(DEV)
    dv.edge_index_down_range = torch.from_numpy(g4['range_down']).to(DEV)
    dv.edge_index_up_range = torch.from_numpy(g4['range_up']).to(DEV)
    gv = GraphedForward(vm, dv)
    assert rel_err(gv.replay(), t(g4['neurips1/out'])) < TOL['f16']


def test_fused_loss_epilogue_matches_reference_formulas():
    """f4: one pass for mse_loss, the differentiated L1 norm and LpLoss.rel of the decoded fields
    (UAI1_full_resolution.py:262-268; utilities.py:87-99, 184-199) -- against the formulas written with torch ops."""
    from graph_pde_b200.losses import fused_losses
    dev = torch.device('cuda:0')
    g = torch.Generator().manual_seed(0)
    B, n = 4, 3000
    out = torch.randn(B * n, 1, generator=g).to(dev).requires_grad_(True)
    y = torch.randn(B * n, generator=g).to(dev)

    class Norm(object):                      # UnitGaussianNormalizer's fields (utilities.py:70-78)
        mean = torch.randn(n, generator=g)
        std = torch.rand(n, generator=g) + 0.5
        eps = 1e-5
    loss, st = fused_losses(out, y, batch_size=B, normalizer=Norm)
    loss.backward()
    o2 = out.detach().clone().requires_grad_(True)
    ref_l1 = torch.norm(o2.view(-1) - y.view(-1), 1)
    ref_l1.backward()
    mean, std = Norm.mean.to(dev), Norm.std.to(dev)
    dec = lambda v: v.view(B, -1) * (std + Norm.eps) + mean      # noqa: E731
    diff = torch.norm(dec(o2.detach()) - dec(y), 2, 1)
    rel = diff / torch.norm(dec(y), 2, 1)
    ref = torch.stack([F.mse_loss(o2.detach().view(-1, 1), y.view(-1, 1)), ref_l1.detach(), rel.sum(), rel.mean()])
    assert float((st - ref).abs().max() / ref.abs().max()) < 1e-5
    assert abs(float(loss) - float(ref_l1)) / float(ref_l1) < 1e-5
    assert torch.equal(out.grad, o2.grad)
