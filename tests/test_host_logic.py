"""CPU-only tests of the host-side mirror of the reference interface (no kernels run)."""
import math
import os
import pickle

import numpy as np
import pytest
import torch

from graph_pde_b200 import graphs
from graph_pde_b200.models import DenseNet, KernelInduced, KernelNN, MGKN, MKGN
from graph_pde_b200.nn_conv import NNConv, NNConv_old, _linear_chain
from oracle import nnconv_oracle as O
from tests.helpers import GOLDEN, vcycle_weights


def test_signature_attributes_repr_and_state_dict_keys():
    mlp = DenseNet([6, 16, 16, 64], torch.nn.ReLU)
    conv = NNConv_old(8, 8, mlp, aggr='mean')
    assert repr(conv) == 'NNConv_old(8, 8)'                  # nn_conv.py:284-286
    assert (conv.in_channels, conv.out_channels, conv.aggr) == (8, 8, 'mean')
    assert sorted(conv.state_dict().keys()) == sorted(
        ['root', 'bias'] + ['nn.layers.%d.%s' % (i, n) for i in (0, 2, 4) for n in ('weight', 'bias')])
    conv2 = NNConv(8, 8, DenseNet([6, 16, 64], torch.nn.ReLU), aggr='mean', root_weight=False, bias=False)
    assert conv2.root is None and conv2.bias is None
    assert repr(conv2) == 'NNConv(8, 8)'
    with pytest.raises(ValueError):
        NNConv_old(8, 8, mlp, aggr='median')


def test_reset_parameters_matches_reference_stream():
    """Same RNG consumption order as DenseNet ctor + NNConv_old.reset_parameters (nn_conv.py:261-265)."""
    torch.manual_seed(0)
    conv = NNConv_old(32, 32, DenseNet([6, 64, 64, 1024], torch.nn.ReLU), aggr='mean')
    ws, bs, root, bias = O.reference_init(32, 32, [6, 64, 64, 1024], seed=0)
    lin = _linear_chain(conv.nn)
    for l, w, b in zip(lin, ws, bs):
        assert torch.equal(l.weight.detach(), w) and torch.equal(l.bias.detach(), b)
    assert torch.equal(conv.root.detach(), root) and torch.equal(conv.bias.detach(), bias)
    assert float(conv.root.detach().abs().max()) <= 1 / math.sqrt(32)


def test_whole_module_pickle_roundtrip(tmp_path):
    """The reference saves whole modules with torch.save(model) (UAI1_full_resolution.py:317)."""
    model = KernelNN(8, 16, 2, 6, in_width=6)
    p = tmp_path / 'm.pt'
    torch.save(model, p)
    back = torch.load(p, weights_only=False)
    assert isinstance(back.conv1, NNConv_old) and back.depth == 2
    for a, b in zip(model.state_dict().values(), back.state_dict().values()):
        assert torch.equal(a, b)


def test_checkpoint_state_dict_loads_into_our_kernelnn():
    g = np.load(os.path.join(GOLDEN, 'g3_checkpoint_grain_new.npz'))
    st = {k[2:]: torch.from_numpy(g[k]) for k in g.files if k.startswith('w/')}
    mlp = DenseNet([6, 64, 32, 4096], torch.nn.ReLU)
    conv = NNConv_old(64, 64, mlp, aggr='mean')
    conv.load_state_dict({k[len('conv1.'):]: v for k, v in st.items() if k.startswith('conv1.')})
    assert torch.equal(conv.nn.layers[4].weight.detach(), st['conv1.nn.layers.4.weight'])


def test_cpu_tensors_are_rejected_loudly():
    conv = NNConv_old(8, 8, DenseNet([6, 16, 64], torch.nn.ReLU), aggr='mean')
    x = torch.randn(10, 8)
    ei = torch.randint(0, 10, (2, 30))
    ea = torch.randn(30, 6)
    with torch.no_grad(), pytest.raises(RuntimeError, match='no CPU path'):
        conv(x, ei, ea)


def test_unsupported_edge_network_is_rejected():
    bad = torch.nn.Sequential(torch.nn.Linear(6, 16), torch.nn.Tanh(), torch.nn.Linear(16, 64))
    with pytest.raises(NotImplementedError):
        _linear_chain(bad)
    with pytest.raises(NotImplementedError):
        _linear_chain(torch.nn.Sequential(torch.nn.Linear(6, 16), torch.nn.ReLU()))


def test_model_constructors_match_reference_layouts():
    g = np.load(os.path.join(GOLDEN, 'g4_mgkn_vcycle.npz'))
    pts = [int(p) for p in g['points']]
    ki = KernelInduced(width=32, ker_width=64, depth=2, ker_in=6, points=pts, level=len(pts), in_width=6)
    ref_keys = sorted(k[len('neurips1/shape/'):] for k in g.files if k.startswith('neurips1/shape/'))
    assert sorted(ki.state_dict().keys()) == ref_keys
    for k in ref_keys:
        assert tuple(ki.state_dict()[k].shape) == tuple(g['neurips1/shape/' + k]), k
    mk = MKGN(width=32, ker_width=64, depth=2, ker_in=6, points=pts, level=len(pts), in_width=6)
    ref_keys = sorted(k[len('general/shape/'):] for k in g.files if k.startswith('general/shape/'))
    assert sorted(mk.state_dict().keys()) == ref_keys
    for k in ref_keys:
        assert tuple(mk.state_dict()[k].shape) == tuple(g['general/shape/' + k]), k
    g5 = np.load(os.path.join(GOLDEN, 'g5_mgkn_burgers1d.npz'))
    mg = MGKN(width=32, ker_width=64, depth=2, ker_in=4, in_width=2, s=int(g5['s']))
    ref_keys = sorted(k[2:] for k in g5.files if k.startswith('w/'))
    assert sorted(mg.state_dict().keys()) == ref_keys
    for k in ref_keys:
        assert tuple(mg.state_dict()[k].shape) == g5['w/' + k].shape, k


def test_graph_builder_matches_oracle_and_sklearn_golden():
    g = np.load(os.path.join(GOLDEN, 'g6_ball_graphs.npz'))
    for key in [k for k in g.files if k.startswith('ei/')]:
        s, r = key[3:].split('_')
        s, r = int(s), float(r)
        ei = graphs.ball_connectivity(s, r)
        np.testing.assert_array_equal(ei.numpy(), g[key].astype(np.int64))
        th = torch.arange(s * s, dtype=torch.float64) * 0.01
        ea = graphs.ball_edge_attr(graphs.square_grid(s), ei, th)
        np.testing.assert_allclose(ea.numpy(), g['ea/' + key[3:]], atol=1e-6)
    part = graphs.ball_connectivity(31, 0.1, nodes=(100, 140))
    full = graphs.ball_connectivity(31, 0.1)
    sel = (full[0] >= 100) & (full[0] < 140)
    assert torch.equal(part, full[:, sel])
    assert full.size(1) == 25673                                # ties-in rule (SURVEY H3)


def test_multilevel_graph_builder_matches_reference_golden():
    """graphs.multi_level_ball_graph vs RandomMultiMeshGenerator (multipole-graph-neural-operator/
    utilities.py:546-712) on the seeded G7 fixture: same randperm stream, same edge order, ranges and attributes."""
    g7 = np.load(os.path.join(GOLDEN, 'g7_multilevel_graph.npz'))
    torch.manual_seed(0)
    g = graphs.multi_level_ball_graph(int(g7['s']), [int(v) for v in g7['m']], list(g7['ri']), list(g7['rx']),
                                      theta=torch.from_numpy(g7['theta']))
    for name, key in (('edge_index_mid', 'e_mid'), ('edge_index_down', 'e_down'), ('edge_index_up', 'e_up'),
                      ('edge_index_range', 'r_mid'), ('edge_index_down_range', 'r_down'),
                      ('edge_index_up_range', 'r_up')):
        assert np.array_equal(getattr(g, name).numpy(), g7[key].astype(np.int64)), name
    for name, key in (('edge_attr_mid', 'a_mid'), ('edge_attr_down', 'a_down'), ('edge_attr_up', 'a_up')):
        assert np.allclose(getattr(g, name).numpy(), g7[key], atol=1e-6), name


def test_multipole_grid1d_matches_reference_golden():
    """graphs.multi_pole_grid1d vs the reference's multi_pole_grid1d + get_edge_attr
    (multipole-graph-neural-operator/utilities.py:1702-1777) on the periodic s=64 hierarchy stored in G5."""
    g = np.load(os.path.join(GOLDEN, 'g5_mgkn_burgers1d.npz'))
    X, ei, ea = graphs.multi_pole_grid1d(g['X/0'][:, 1], int(g['s']), is_periodic=True)
    assert len(X) == int(g['n_levels']) and len(ei) == int(g['n_edge_sets'])
    for l in range(len(X)):
        assert np.allclose(X[l].numpy(), g['X/%d' % l], atol=1e-6)
    for i in range(len(ei)):
        assert np.array_equal(ei[i].numpy(), g['edge_index/%d' % i].astype(np.int64))
        assert np.allclose(ea[i].numpy(), g['edge_attr/%d' % i], atol=1e-6)
    # truncation (BASELINE config 5: "5 levels" of the 12 the shipped rule gives at s=8192) and edge counts of
    # SURVEY a10: nn = 2s, inter_l = 3 s_l - 6 without periodic wrap
    X5, ei5, _ = graphs.multi_pole_grid1d(torch.zeros(8192), 8192, is_periodic=False, levels=5)
    assert [x.shape[0] for x in X5] == [8192, 4096, 2048, 1024, 512]
    assert ei5[0].shape[1] == 2 * 8192 - 2
    assert [e.shape[1] for e in ei5[1:]] == [3 * n - 6 for n in (8192, 4096, 2048, 1024, 512)]


def test_dropin_modules_resolve_like_the_reference_imports(monkeypatch):
    import importlib
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    monkeypatch.syspath_prepend(os.path.join(root, 'dropin'))
    for m in ('nn_conv', 'torch_geometric', 'torch_geometric.nn', 'torch_geometric.data'):
        sys.modules.pop(m, None)
    nn_conv_mod = importlib.import_module('nn_conv')
    tg_nn = importlib.import_module('torch_geometric.nn')
    tg_data = importlib.import_module('torch_geometric.data')
    conv = nn_conv_mod.NNConv_old(8, 8, DenseNet([6, 16, 64], torch.nn.ReLU), aggr='mean')
    assert type(conv).__module__ == 'nn_conv' and repr(conv) == 'NNConv_old(8, 8)'
    assert issubclass(tg_nn.NNConv, NNConv_old)
    # block-diagonal batching rule (PyG Batch): 'index' keys are offset by the node count
    a = tg_data.Data(x=torch.zeros(3, 2), edge_index=torch.tensor([[0, 1], [1, 2]]), edge_attr=torch.zeros(2, 6))
    b = tg_data.Data(x=torch.ones(2, 2), edge_index=torch.tensor([[0], [1]]), edge_attr=torch.ones(1, 6))
    batch = next(iter(tg_data.DataLoader([a, b], batch_size=2)))
    assert batch.x.shape == (5, 2) and batch.edge_index.tolist() == [[0, 1, 3], [1, 2, 4]]
    for m in ('nn_conv', 'torch_geometric', 'torch_geometric.nn', 'torch_geometric.data'):
        sys.modules.pop(m, None)


def test_device_resident_loader_shares_the_mesh_and_caches_block_diagonal_index():
    """f3: DataLoader(device=...) moves the dataset once, keeps the shared edge_index shared, collates on that device
    and reuses ONE block-diagonal edge_index per batch size (so the conv's plan cache hits every step)."""
    import importlib.util
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'dropin', 'torch_geometric', 'data',
                        '__init__.py')
    spec = importlib.util.spec_from_file_location('dropin_pyg_data', path)
    D = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(D)
    ei = torch.tensor([[0, 1, 2], [1, 2, 0]])
    data = [D.Data(x=torch.randn(3, 2), y=torch.randn(3), edge_index=ei, edge_attr=torch.randn(3, 4)) for _ in range(6)]
    loader = D.DataLoader(data, batch_size=2, shuffle=True, device='cpu')
    assert all(it.edge_index is loader.dataset[0].edge_index for it in loader.dataset)      # still one mesh tensor
    batches = list(loader)
    assert len(batches) == 3
    assert all(b.edge_index is batches[0].edge_index for b in batches)                      # cached block diagonal
    assert batches[0].edge_index.tolist() == [[0, 1, 2, 3, 4, 5], [1, 2, 0, 4, 5, 3]]
    assert batches[0].x.shape == (6, 2) and batches[0].batch.tolist() == [0, 0, 0, 1, 1, 1]
    single = next(iter(D.DataLoader(data, batch_size=1)))
    assert single is not data[0] and single.x is data[0].x                                   # shallow copy of the item


def test_vcycle_step_chain_on_preactivations_equals_the_reference_op_sequence(monkeypatch):
    """`KernelInduced` inference chains `residual_step` (z' = relu(z) + conv(relu(z)), last ReLU applied once);
    with the CPU oracle standing in for the two conv entry points the chained forward must equal the reference's
    conv / add / ReLU sequence and the golden output of the reference's own class (G4)."""
    import numpy as np
    from graph_pde_b200 import models, nn_conv
    from tests.helpers import GOLDEN, ei64, t

    def lin(conv):
        ls = [m for m in conv.nn.layers if isinstance(m, torch.nn.Linear)]
        return [l.weight.detach() for l in ls], [l.bias.detach() for l in ls]

    def conv_forward(self, x, edge_index, edge_attr):
        ws, bs = lin(self)
        return O.nnconv_forward(x, edge_index, edge_attr, ws, bs, None if self.root is None else self.root.detach(),
                                None if self.bias is None else self.bias.detach(), self.aggr)

    calls = {'res': 0}

    def residual_step(self, z, edge_index, edge_attr, relu_in=True):
        calls['res'] += 1
        x = torch.relu(z) if relu_in else z
        return x + conv_forward(self, x, edge_index, edge_attr)

    monkeypatch.setattr(nn_conv.NNConv_old, 'forward', conv_forward)
    monkeypatch.setattr(nn_conv.NNConv_old, 'residual_step', residual_step)
    g = np.load(os.path.join(GOLDEN, 'g4_mgkn_vcycle.npz'))
    pts = [int(p) for p in g['points']]
    model = models.KernelInduced(width=32, ker_width=64, depth=2, ker_in=6, points=pts, level=len(pts), in_width=6)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in vcycle_weights(g, 'neurips1').items()})

    class D(object):
        pass
    d = D()
    d.x = t(g['node_x'])
    for nm in ('mid', 'down', 'up'):
        setattr(d, 'edge_index_' + nm, ei64(g['edge_index_' + nm]))
        setattr(d, 'edge_attr_' + nm, t(g['edge_attr_' + nm]))
    d.edge_index_range = torch.from_numpy(g['range_mid'])
    d.edge_index_down_range = torch.from_numpy(g['range_down'])
    d.edge_index_up_range = torch.from_numpy(g['range_up'])
    with torch.no_grad():
        monkeypatch.setattr(models, '_FUSED_STEPS', True)
        fused = model(d)
        n_res = calls['res']
        monkeypatch.setattr(models, '_FUSED_STEPS', False)
        plain = model(d)
    assert n_res == 2 * (3 * len(pts) - 2) and calls['res'] == n_res       # 13 steps per depth iteration at 5 levels
    ref = t(g['neurips1/out'])
    assert float((fused - ref).abs().max() / ref.abs().max()) < 1e-5
    assert float((fused - plain).abs().max() / ref.abs().max()) < 1e-5
    # with gradients required the model must stay on the autograd-capable op sequence
    monkeypatch.setattr(models, '_FUSED_STEPS', True)
    out = model(d)
    assert calls['res'] == n_res and out.requires_grad
