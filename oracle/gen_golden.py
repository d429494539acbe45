"""Generate tests/golden/*.npz by running the REFERENCE's own files, unmodified.

TEST INFRASTRUCTURE.  Needs a checkout of the reference (the tests only read the .npz files it writes):

    [GRAPH_PDE_REFERENCE=<reference checkout>] python oracle/gen_golden.py [g1 g2 ... g7]

(no names: all seven; the checkout defaults to /root/reference).  What runs:
graph-neural-operator/{nn_conv.py,utilities.py},
multipole-graph-neural-operator/utilities.py and the model classes KernelNN /
KernelInduced / MKGN / MGKN extracted (by `ast`, not copied) from the reference scripts, over
oracle/pyg_stub (the restated third-party boundary, see its docstring).  The outputs are the golden
vectors that pin oracle/nnconv_oracle.py and, through it, the CUDA path.  Every file stays under 1 MB.
"""
import ast
import hashlib
import os
import sys
import warnings

import numpy as np
import torch

warnings.filterwarnings('ignore')
HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get('GRAPH_PDE_REFERENCE') or '/root/reference'      # the reference checkout
GNO = os.path.join(REF, 'graph-neural-operator')
MGNO = os.path.join(REF, 'multipole-graph-neural-operator')
OUT = os.path.join(HERE, '..', 'tests', 'golden')
WANT = set(a[:2] for a in sys.argv[1:]) or None    # e.g. g3 g4


def _import_reference():
    sys.path[:0] = [os.path.join(HERE, 'pyg_stub'), GNO]
    import nn_conv            # GNO/nn_conv.py, unmodified
    import utilities as gno_utilities
    import importlib.util
    spec = importlib.util.spec_from_file_location('mgno_utilities', os.path.join(MGNO, 'utilities.py'))
    mgno_utilities = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mgno_utilities)
    return nn_conv, gno_utilities, mgno_utilities


def _class_from_script(path, name, namespace):
    """Compile ONE class definition out of a reference script (the scripts run training at import)."""
    tree = ast.parse(open(path).read())
    node = [n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == name][0]
    mod = ast.Module(body=[node], type_ignores=[])
    exec(compile(mod, path, 'exec'), namespace)
    return namespace[name]


def _np_state(module):
    return {k: v.detach().numpy().copy() for k, v in module.state_dict().items()}


def _save(name, **rec):
    if WANT is None or name[:2] in WANT:
        np.savez_compressed(os.path.join(OUT, name), **rec)


def main():
    assert os.path.isdir(GNO) and os.path.isdir(MGNO), 'no reference checkout at %s (set GRAPH_PDE_REFERENCE)' % REF
    os.makedirs(OUT, exist_ok=True)
    nn_conv, U, MU = _import_reference()
    import torch.nn.functional as F
    ns_gno = dict(torch=torch, np=np, F=F, DenseNet=U.DenseNet, NNConv_old=nn_conv.NNConv_old)
    # MGKN scripts import upstream torch_geometric.nn.NNConv == same math as NNConv_old (SURVEY 0.3)
    ns_mgno = dict(torch=torch, np=np, F=F, DenseNet=MU.DenseNet, NNConv=nn_conv.NNConv_old)

    # ---------------- G1: tiny multigraph, every flag combination, everything stored -------------
    g = torch.Generator().manual_seed(1234)
    N, E, cin, cout, kin = 40, 300, 5, 7, 3
    src = torch.randint(0, N - 6, (E,), generator=g)      # last 6 nodes: no out-edges
    dst = torch.randint(3, N, (E,), generator=g)          # first 3 nodes: no in-edges (mean of empty set)
    src[10:20] = src[0]
    dst[10:20] = dst[0]                                   # duplicate edges
    ei = torch.stack([src, dst])
    ea = torch.randn(E, kin, generator=g)
    x = torch.randn(N, cin, generator=g)
    rec = dict(edge_index=ei.numpy().astype(np.int32), edge_attr=ea.numpy(), x=x.numpy())
    for aggr in ('mean', 'add'):
        for rw in (True, False):
            for bs in (True, False):
                torch.manual_seed(7)
                mlp = U.DenseNet([kin, 10, cin * cout], torch.nn.ReLU)
                conv = nn_conv.NNConv_old(cin, cout, mlp, aggr=aggr, root_weight=rw, bias=bs)
                tag = '%s_r%d_b%d' % (aggr, rw, bs)
                for k, v in _np_state(conv).items():
                    rec['%s/%s' % (tag, k)] = v
                rec['%s/out' % tag] = conv(x, ei, ea).detach().numpy()
    # 1-D x / 1-D edge_attr unsqueeze path (nn_conv.py:269-270)
    torch.manual_seed(8)
    mlp = U.DenseNet([1, 6, 1 * 4], torch.nn.ReLU)
    conv = nn_conv.NNConv_old(1, 4, mlp, aggr='mean')
    x1 = torch.randn(N, generator=g)
    ea1 = torch.randn(E, generator=g)
    for k, v in _np_state(conv).items():
        rec['oned/%s' % k] = v
    rec['oned/x'] = x1.numpy()
    rec['oned/edge_attr'] = ea1.numpy()
    rec['oned/out'] = conv(x1, ei, ea1).detach().numpy()
    _save('g1_tiny_multigraph.npz', **rec)

    # ---------------- G2: BASELINE config 1 (16x16, r=.25, w=32, kw=1024, T=4), seeded weights ----
    torch.manual_seed(0)
    np.random.seed(0)
    s, r, w, kw, T = 16, 0.25, 32, 1024, 4
    mg = U.SquareMeshGenerator([[0, 1], [0, 1]], [s, s])
    ei = mg.ball_connectivity(r)
    theta = np.random.randn(s * s)
    ea = mg.attributes(theta=theta)
    KernelNN = _class_from_script(os.path.join(GNO, 'UAI1_full_resolution.py'), 'KernelNN', dict(ns_gno))
    torch.manual_seed(0)
    model = KernelNN(w, kw, T, 6, in_width=6)
    node_x = torch.cat([mg.get_grid(), torch.tensor(theta, dtype=torch.float).view(-1, 1),
                        torch.randn(s * s, 3)], dim=1)
    with torch.no_grad():
        xs = [model.fc1(node_x)]
        for k in range(T):
            xs.append(F.relu(model.conv1(xs[-1], ei, ea)))
        full = model(type('D', (), dict(x=node_x, edge_index=ei, edge_attr=ea))())
    st = _np_state(model)
    rec = dict(edge_index=ei.numpy().astype(np.int32), edge_attr=ea.numpy(), theta=theta,
               node_x=node_x.numpy(), x0=xs[0].numpy(), x_after=np.stack([t.numpy() for t in xs[1:]]),
               model_out=full.numpy(), s=s, r=r, width=w, ker_width=kw, depth=T)
    # weights are reproducible from the seed (oracle.reference_init); store checksums + small tensors
    for k, v in st.items():
        rec['sum/%s' % k] = np.float64(v.astype(np.float64).sum())
        rec['abs/%s' % k] = np.float64(np.abs(v.astype(np.float64)).sum())
        if v.size <= 8192:
            rec['w/%s' % k] = v
    _save('g2_cfg1_ball16.npz', **rec)

    # ---------------- G3: shipped checkpoint weights (the reference's only fixture) ---------------
    import __main__

    class KernelNNCkpt(torch.nn.Module):      # placeholder class for unpickling `__main__.KernelNN`
        pass
    __main__.KernelNN = KernelNNCkpt
    ck = torch.load(os.path.join(GNO, 'model', 'grain_new_r64_s64testm100'), map_location='cpu',
                    weights_only=False)
    # the trained 4096 x 128 output layer of the edge network alone is 2 MB: keep the first 32 of the 128 units of
    # the second hidden layer (edge network 6 -> 64 -> 32 -> 4096, still width 64), so that the file stays < 1 MB
    k3 = 32
    lay = ck.conv1.nn.layers
    with torch.no_grad():
        lay[2].weight = torch.nn.Parameter(lay[2].weight[:k3].clone())
        lay[2].bias = torch.nn.Parameter(lay[2].bias[:k3].clone())
        lay[4].weight = torch.nn.Parameter(lay[4].weight[:, :k3].clone())
    lay[2].out_features = lay[4].in_features = k3
    st = {k: v.detach().clone() for k, v in ck.state_dict().items()}
    torch.manual_seed(0)
    np.random.seed(0)
    s, r = 16, 0.25
    mg = U.SquareMeshGenerator([[0, 1], [0, 1]], [s, s])
    ei = mg.ball_connectivity(r)
    theta = np.random.randn(s * s)
    ea = mg.attributes(theta=theta)
    node_x = torch.cat([mg.get_grid(), torch.tensor(theta, dtype=torch.float).view(-1, 1),
                        torch.randn(s * s, 3)], dim=1)
    conv = ck.conv1                      # a real reference NNConv_old instance with trained weights
    with torch.no_grad():
        xs = [F.linear(node_x, st['fc1.weight'], st['fc1.bias'])]
        for k in range(6):
            xs.append(F.relu(conv(xs[-1], ei, ea)))
    rec = dict(edge_index=ei.numpy().astype(np.int32), edge_attr=ea.numpy(), node_x=node_x.numpy(),
               x0=xs[0].numpy(), x_after=np.stack([t.numpy() for t in xs[1:]]))
    for k, v in st.items():
        rec['w/%s' % k] = v.numpy()
    _save('g3_checkpoint_grain_new.npz', **rec)

    # ---------------- G4: MGKN V-cycle (both script variants) on a small multi-level graph ---------
    torch.manual_seed(0)
    np.random.seed(0)
    s = 31
    m = [200, 80, 30]
    level = len(m)
    mmg = MU.RandomMultiMeshGenerator([[0, 1], [0, 1]], [s, s], level=level, sample_sizes=m)
    idx, idx_all = mmg.sample()
    ei_mid, ei_down, ei_up = mmg.ball_connectivity([0.15, 0.3, 0.6], [0.2, 0.4])
    r_mid, r_down, r_up = mmg.get_edge_index_range()
    theta = np.random.randn(s * s)
    ea_mid, ea_down, ea_up = mmg.attributes(theta=theta)
    node_x = torch.cat([torch.tensor(mmg.grid_sample_all, dtype=torch.float),
                        torch.randn(sum(m), 4)], dim=1)
    data = type('D', (), dict(x=node_x, edge_index_mid=ei_mid, edge_index_down=ei_down, edge_index_up=ei_up,
                              edge_index_range=r_mid, edge_index_down_range=r_down, edge_index_up_range=r_up,
                              edge_attr_mid=ea_mid, edge_attr_down=ea_down, edge_attr_up=ea_up))()
    rec = dict(node_x=node_x.numpy(), points=np.array(m),
               edge_index_mid=ei_mid.numpy().astype(np.int32), edge_index_down=ei_down.numpy().astype(np.int32),
               edge_index_up=ei_up.numpy().astype(np.int32), range_mid=r_mid.numpy(), range_down=r_down.numpy(),
               range_up=r_up.numpy(), edge_attr_mid=ea_mid.numpy(), edge_attr_down=ea_down.numpy(),
               edge_attr_up=ea_up.numpy(), width=32, ker_width=64, depth=2)

    def seeded_state(variant, seed, model):
        # the untrained parameters are a seeded draw (1.7 MB): stored as seed, shapes and sha256 of their bytes,
        # the tests re-draw them with the project's constructors (same init stream) and check the hashes
        rec[variant + '/seed'] = seed
        for k, v in _np_state(model).items():
            rec['%s/shape/%s' % (variant, k)] = np.array(v.shape)
            rec['%s/sha256/%s' % (variant, k)] = np.array(hashlib.sha256(np.ascontiguousarray(v).tobytes()).hexdigest())
    KI = _class_from_script(os.path.join(MGNO, 'neurips1_MGKN.py'), 'KernelInduced', dict(ns_mgno))
    torch.manual_seed(1)
    model = KI(width=32, ker_width=64, depth=2, ker_in=6, points=m, level=level, in_width=6, out_width=1)
    with torch.no_grad():
        rec['neurips1/out'] = model(data).numpy()
    seeded_state('neurips1', 1, model)
    MK = _class_from_script(os.path.join(MGNO, 'MGKN_general_darcy2d.py'), 'MKGN', dict(ns_mgno))
    torch.manual_seed(2)
    import io
    import contextlib
    with contextlib.redirect_stdout(io.StringIO()):
        model = MK(width=32, ker_width=64, depth=2, ker_in=6, points=m, level=level, in_width=6, out_width=1)
    with torch.no_grad():
        rec['general/out'] = model(data).numpy()
    seeded_state('general', 2, model)
    _save('g4_mgkn_vcycle.npz', **rec)

    # ---------------- G5: orthogonal MGKN, Burgers 1-D multipole graph -----------------------------
    torch.Tensor.cuda = lambda self, *a, **k: self      # reference calls .cuda() (MGNO/utilities.py:1743)
    torch.manual_seed(0)
    np.random.seed(0)
    s, Nsamp = 64, 1
    theta = np.random.randn(Nsamp, s, 1)
    with contextlib.redirect_stdout(io.StringIO()):
        grid_list, theta_list, ei_list, _ = MU.multi_pole_grid1d(theta=theta, theta_d=1, s=s, N=Nsamp,
                                                                 is_periodic=True)
    X_list, ea_list = [], []
    for l in range(len(grid_list)):
        X_list.append(torch.cat([grid_list[l].reshape(-1, 1), theta_list[l][0].reshape(-1, 1)], dim=1))
    for i in range(len(ei_list)):
        l = 0 if i == 0 else i - 1
        ea_list.append(MU.get_edge_attr(grid_list[l], theta_list[l][0, :, 0], ei_list[i]))
    MG = _class_from_script(os.path.join(MGNO, 'MGKN_orthogonal_burgers1d.py'), 'MGKN', dict(ns_mgno))
    torch.manual_seed(3)
    model = MG(width=32, ker_width=64, depth=2, ker_in=4, in_width=2, s=s)
    with torch.no_grad():
        out = model((X_list, None, ei_list, ea_list))
    rec = dict(out=out.numpy(), s=s, width=32, ker_width=64, depth=2, n_levels=len(grid_list),
               n_edge_sets=len(ei_list))
    for l, X in enumerate(X_list):
        rec['X/%d' % l] = X.numpy()
    for i in range(len(ei_list)):
        rec['edge_index/%d' % i] = ei_list[i].numpy().astype(np.int32)
        rec['edge_attr/%d' % i] = ea_list[i].numpy()
    for k, v in _np_state(model).items():
        rec['w/%s' % k] = v
    _save('g5_mgkn_burgers1d.npz', **rec)

    # ---------------- G6: graph-generator restatement pins (edge lists from sklearn path) ----------
    rec = {}
    for (s, r) in [(16, 0.25), (21, 0.13), (9, 0.3)]:       # no lattice distance ties with r
        mg = U.SquareMeshGenerator([[0, 1], [0, 1]], [s, s])
        ei = mg.ball_connectivity(r)
        th = np.arange(s * s, dtype=np.float64) * 0.01
        rec['ei/%d_%g' % (s, r)] = ei.numpy().astype(np.int32)
        rec['ea/%d_%g' % (s, r)] = mg.attributes(theta=th).numpy()
    _save('g6_ball_graphs.npz', **rec)
    # ---------------- G7: multi-level (MGKN) graph generator pins, RandomMultiMeshGenerator, seeded ----------
    s, m, ri, rx = 31, [200, 80, 30], [0.155, 0.31, 0.62], [0.21, 0.41]    # radii without lattice ties
    torch.manual_seed(0)
    mmg = MU.RandomMultiMeshGenerator([[0, 1], [0, 1]], [s, s], level=3, sample_sizes=m)
    mmg.sample()
    e_mid, e_down, e_up = mmg.ball_connectivity(ri, rx)
    r_mid, r_down, r_up = mmg.get_edge_index_range()
    theta = np.random.RandomState(0).randn(s * s)
    a_mid, a_down, a_up = mmg.attributes(theta=theta)
    _save('g7_multilevel_graph.npz', s=s, m=np.array(m), ri=np.array(ri),
                        rx=np.array(rx), theta=theta, e_mid=e_mid.numpy().astype(np.int32),
                        e_down=e_down.numpy().astype(np.int32), e_up=e_up.numpy().astype(np.int32),
                        r_mid=r_mid.numpy(), r_down=r_down.numpy(), r_up=r_up.numpy(),
                        a_mid=a_mid.numpy(), a_down=a_down.numpy(), a_up=a_up.numpy())
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == '__main__':
    main()
