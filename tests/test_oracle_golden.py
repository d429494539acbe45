"""Pin the CPU oracle (oracle/nnconv_oracle.py) against golden vectors produced by the reference's own
nn_conv.py / utilities.py / model classes (oracle/gen_golden.py).  CPU only."""
import os

import numpy as np
import torch

from oracle import nnconv_oracle as O
from tests.helpers import vcycle_weights

TOL = dict(rtol=2e-5, atol=2e-5)     # fp32 vs fp32, summation order differs only by chunking


def _t(a):
    return torch.from_numpy(np.asarray(a))


def _ei(a):
    return torch.from_numpy(np.asarray(a).astype(np.int64))


def test_g1_tiny_multigraph_all_flags(golden_dir):
    g = np.load(os.path.join(golden_dir, 'g1_tiny_multigraph.npz'))
    ei, ea, x = _ei(g['edge_index']), _t(g['edge_attr']), _t(g['x'])
    for aggr in ('mean', 'add'):
        for rw in (1, 0):
            for bs in (1, 0):
                tag = '%s_r%d_b%d' % (aggr, rw, bs)
                ws = [_t(g[tag + '/nn.layers.0.weight']), _t(g[tag + '/nn.layers.2.weight'])]
                bsl = [_t(g[tag + '/nn.layers.0.bias']), _t(g[tag + '/nn.layers.2.bias'])]
                root = _t(g[tag + '/root']) if rw else None
                bias = _t(g[tag + '/bias']) if bs else None
                out = O.nnconv_forward(x, ei, ea, ws, bsl, root, bias, aggr, 5, 7)
                np.testing.assert_allclose(out.numpy(), g[tag + '/out'], **TOL)
                out_c = O.nnconv_forward(x, ei, ea, ws, bsl, root, bias, aggr, 5, 7, edge_chunk=37)
                np.testing.assert_allclose(out_c.numpy(), g[tag + '/out'], **TOL)
    ws = [_t(g['oned/nn.layers.0.weight']), _t(g['oned/nn.layers.2.weight'])]
    bsl = [_t(g['oned/nn.layers.0.bias']), _t(g['oned/nn.layers.2.bias'])]
    out = O.nnconv_forward(_t(g['oned/x']), ei, _t(g['oned/edge_attr']), ws, bsl, _t(g['oned/root']),
                           _t(g['oned/bias']), 'mean', 1, 4)
    np.testing.assert_allclose(out.numpy(), g['oned/out'], **TOL)


def test_g2_cfg1_seeded_weights_and_stack(golden_dir):
    """BASELINE config 1.  Weights are re-drawn from the seed with the restated init order and checked
    against the reference's checksums, then the T=4 conv stack is compared iteration by iteration."""
    g = np.load(os.path.join(golden_dir, 'g2_cfg1_ball16.npz'))
    w, kw, T = int(g['width']), int(g['ker_width']), int(g['depth'])
    torch.manual_seed(0)
    fc1 = torch.nn.Linear(6, w)                         # KernelNN.__init__ order: fc1, kernel, conv1, fc2
    st = {'fc1.weight': fc1.weight.detach(), 'fc1.bias': fc1.bias.detach()}
    # continue the SAME RNG stream: DenseNet ctor, NNConv_old.reset_parameters
    lins = [torch.nn.Linear(a, b) for a, b in zip([6, kw, kw], [kw, kw, w * w])]
    for lin in lins:
        lin.reset_parameters()
    root = torch.empty(w, w).uniform_(-1 / np.sqrt(w), 1 / np.sqrt(w))
    bias = torch.empty(w).uniform_(-1 / np.sqrt(w), 1 / np.sqrt(w))
    ws = [l.weight.detach() for l in lins]
    bs = [l.bias.detach() for l in lins]
    for i, l in enumerate((0, 2, 4)):
        assert abs(float(ws[i].double().sum()) - float(g['sum/conv1.nn.layers.%d.weight' % l])) < 1e-6
        assert abs(float(ws[i].double().abs().sum()) - float(g['abs/conv1.nn.layers.%d.weight' % l])) < 1e-4
    np.testing.assert_array_equal(root.numpy(), g['w/conv1.root'])
    np.testing.assert_array_equal(bias.numpy(), g['w/conv1.bias'])
    ei, ea = _ei(g['edge_index']), _t(g['edge_attr'])
    x = torch.nn.functional.linear(_t(g['node_x']), st['fc1.weight'], st['fc1.bias'])
    np.testing.assert_allclose(x.numpy(), g['x0'], **TOL)
    for k in range(T):
        x = torch.relu(O.nnconv_forward(x, ei, ea, ws, bs, root, bias, 'mean', edge_chunk=4096))
        np.testing.assert_allclose(x.numpy(), g['x_after'][k], rtol=1e-4, atol=1e-5)


def test_g3_checkpoint_weights_stack(golden_dir):
    g = np.load(os.path.join(golden_dir, 'g3_checkpoint_grain_new.npz'))
    st = {k[2:]: _t(g[k]) for k in g.files if k.startswith('w/')}
    ws, bs = O.mlp_params_from_state(st, 'conv1.nn.')
    assert [tuple(w.shape) for w in ws] == [(64, 6), (32, 64), (4096, 32)]
    ei, ea = _ei(g['edge_index']), _t(g['edge_attr'])
    x = _t(g['x0'])
    out = O.kernelnn_conv_stack(x, ei, ea, ws, bs, st['conv1.root'], st['conv1.bias'], 6)
    np.testing.assert_allclose(out.numpy(), g['x_after'][5], rtol=1e-4, atol=1e-5)
    x1 = torch.relu(O.nnconv_forward(x, ei, ea, ws, bs, st['conv1.root'], st['conv1.bias'], 'mean'))
    np.testing.assert_allclose(x1.numpy(), g['x_after'][0], rtol=1e-4, atol=1e-5)


def test_g4_mgkn_vcycle_both_variants(golden_dir):
    g = np.load(os.path.join(golden_dir, 'g4_mgkn_vcycle.npz'))
    data = dict(edge_index_mid=_ei(g['edge_index_mid']), edge_index_down=_ei(g['edge_index_down']),
                edge_index_up=_ei(g['edge_index_up']), edge_attr_mid=_t(g['edge_attr_mid']),
                edge_attr_down=_t(g['edge_attr_down']), edge_attr_up=_t(g['edge_attr_up']),
                range_mid=g['range_mid'], range_down=g['range_down'], range_up=g['range_up'])
    pts = [int(p) for p in g['points']]
    for variant in ('neurips1', 'general'):
        st = {k: _t(v) for k, v in vcycle_weights(g, variant).items()}
        out = O.mgkn_vcycle_forward(_t(g['node_x']), data, st, int(g['depth']), len(pts), pts, variant)
        np.testing.assert_allclose(out.numpy(), g[variant + '/out'], rtol=1e-4, atol=1e-5)


def test_g5_mgkn_orthogonal_burgers(golden_dir):
    g = np.load(os.path.join(golden_dir, 'g5_mgkn_burgers1d.npz'))
    st = {k[2:]: _t(g[k]) for k in g.files if k.startswith('w/')}
    n = int(g['n_edge_sets'])
    eis = [_ei(g['edge_index/%d' % i]) for i in range(n)]
    eas = [_t(g['edge_attr/%d' % i]) for i in range(n)]
    out = O.mgkn_orthogonal_forward(_t(g['X/0']), eis, eas, st, int(g['depth']), int(g['width']), int(g['s']))
    np.testing.assert_allclose(out.numpy(), g['out'], rtol=1e-4, atol=1e-5)


def test_g6_ball_graph_generator_matches_sklearn_path(golden_dir):
    g = np.load(os.path.join(golden_dir, 'g6_ball_graphs.npz'))
    for key in [k for k in g.files if k.startswith('ei/')]:
        s, r = key[3:].split('_')
        s, r = int(s), float(r)
        ei = O.ball_connectivity(s, r)
        np.testing.assert_array_equal(ei, g[key].astype(np.int64))
        th = np.arange(s * s, dtype=np.float64) * 0.01
        ea = O.ball_edge_attr(O.square_grid(s), ei, th)
        np.testing.assert_allclose(ea, g['ea/' + key[3:]], rtol=0, atol=1e-7)


def test_tie_rule_counts():
    """SURVEY H3: at 31^2 r=0.1 the exact rule gives 25,673 (ties in) / 22,201 (ties out)."""
    assert O.ball_connectivity(31, 0.1, ties_in=True).shape[1] == 25673
    assert O.ball_connectivity(31, 0.1, ties_in=False).shape[1] == 22201
    assert O.ball_connectivity(16, 0.25).shape[1] == 9324
