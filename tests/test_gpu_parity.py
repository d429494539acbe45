"""GPU parity: the CUDA path (through the C ABI of libnnconv_b200.so) vs golden vectors produced by the
reference's own files and vs the CPU oracle on seeded inputs.  Run on the B200 box: pytest -m gpu."""
import os

import numpy as np
import pytest
import torch

from oracle import nnconv_oracle as O
from tests.helpers import GOLDEN, TOL, DenseNetLike, cfg1_weights, ei64, make_conv, rel_err, t

pytestmark = [pytest.mark.gpu, pytest.mark.usefixtures('edge_kernel_mode')]


@pytest.fixture(scope='module')
def dev():
    assert torch.cuda.is_available()
    return torch.device('cuda:0')


def _conv_cls():
    from graph_pde_b200.nn_conv import NNConv_old
    return NNConv_old


def test_library_loaded_and_device_ok(dev):
    from graph_pde_b200 import _lib
    L = _lib.lib()
    assert L.nnconv_abi_version() == _lib.ABI_VERSION
    _lib.check(L.nnconv_init())


def test_g1_tiny_multigraph_all_flags_fp32(dev):
    """in=5/out=7 is not a tensor-core shape: exercises the CUDA-core fp32 path, duplicates, isolated nodes."""
    g = np.load(os.path.join(GOLDEN, 'g1_tiny_multigraph.npz'))
    ei, ea, x = ei64(g['edge_index']).to(dev), t(g['edge_attr']).to(dev), t(g['x']).to(dev)
    for aggr in ('mean', 'add'):
        for rw in (1, 0):
            for bs in (1, 0):
                tag = '%s_r%d_b%d' % (aggr, rw, bs)
                ws = [g[tag + '/nn.layers.0.weight'], g[tag + '/nn.layers.2.weight']]
                bsl = [g[tag + '/nn.layers.0.bias'], g[tag + '/nn.layers.2.bias']]
                conv = make_conv(_conv_cls(), ws, bsl, g[tag + '/root'] if rw else None,
                                 g[tag + '/bias'] if bs else None, aggr, 5, 7, 'fp32', dev)
                with torch.no_grad():
                    out = conv(x, ei, ea)
                assert rel_err(out, t(g[tag + '/out'])) < TOL['fp32'], tag
    ws = [g['oned/nn.layers.0.weight'], g['oned/nn.layers.2.weight']]
    bsl = [g['oned/nn.layers.0.bias'], g['oned/nn.layers.2.bias']]
    conv = make_conv(_conv_cls(), ws, bsl, g['oned/root'], g['oned/bias'], 'mean', 1, 4, 'fp32', dev)
    with torch.no_grad():
        out = conv(t(g['oned/x']).to(dev), ei, t(g['oned/edge_attr']).to(dev))     # 1-D x and edge_attr
    assert rel_err(out, t(g['oned/out'])) < TOL['fp32']


@pytest.mark.parametrize('precision', ['f16', 'bf16', 'f16x2', 'fp32'])
def test_g2_cfg1_conv_stack(dev, precision):
    """BASELINE config 1: 16x16, r=0.25, w=32, ker_width=1024, T=4 -- every iteration vs the reference."""
    g = np.load(os.path.join(GOLDEN, 'g2_cfg1_ball16.npz'))
    fc1, ws, bs, root, bias = cfg1_weights(g)
    conv = make_conv(_conv_cls(), ws, bs, root, bias, 'mean', 32, 32, precision, dev)
    ei, ea = ei64(g['edge_index']).to(dev), t(g['edge_attr']).to(dev)
    x = t(g['x0']).to(dev)
    with torch.no_grad():
        for k in range(int(g['depth'])):
            x = torch.relu(conv(x, ei, ea))
            assert rel_err(x, t(g['x_after'][k])) < TOL[precision], (precision, k)


@pytest.mark.parametrize('precision', ['f16', 'bf16', 'f16x2', 'fp32'])
def test_g3_checkpoint_weights(dev, precision):
    """Trained weights shipped by the reference (graph-neural-operator/model/grain_new_r64_s64testm100)."""
    g = np.load(os.path.join(GOLDEN, 'g3_checkpoint_grain_new.npz'))
    st = {k[2:]: g[k] for k in g.files if k.startswith('w/')}
    ws = [st['conv1.nn.layers.%d.weight' % i] for i in (0, 2, 4)]
    bs = [st['conv1.nn.layers.%d.bias' % i] for i in (0, 2, 4)]
    conv = make_conv(_conv_cls(), ws, bs, st['conv1.root'], st['conv1.bias'], 'mean', 64, 64, precision, dev)
    ei, ea = ei64(g['edge_index']).to(dev), t(g['edge_attr']).to(dev)
    x = t(g['x0']).to(dev)
    with torch.no_grad():
        for k in range(6):
            x = torch.relu(conv(x, ei, ea))
            assert rel_err(x, t(g['x_after'][k])) < TOL[precision], (precision, k)


@pytest.mark.parametrize('precision', ['f16', 'f16x2', 'fp32'])
@pytest.mark.parametrize('layers', [[6, 64, 4096], [4, 128, 64, 4096], [6, 32, 64, 48, 128, 4096], [3, 4096]])
def test_random_multigraph_unsorted_sources(dev, precision, layers):
    if precision == 'f16x2' and len(layers) == 2:
        pytest.skip('f16x2 needs >= 2 Linear layers (no reference call site has a single-Linear edge network)')
    """Edges NOT grouped by source (exercises the radix-sort plan), hub node with > 128 out-edges, isolated
    nodes, duplicate edges, nodes with no in-edges (mean of the empty set = 0), 1..5 layer edge MLPs."""
    gen = torch.Generator().manual_seed(5)
    N, E, w = 300, 5000, 64
    src = torch.randint(0, N - 20, (E,), generator=gen)
    dst = torch.randint(10, N, (E,), generator=gen)
    src[:700] = 7                                   # hub: several tiles for one source
    src[1000:1010] = src[1000]
    dst[1000:1010] = dst[1000]
    ei = torch.stack([src, dst])
    ea = torch.randn(E, layers[0], generator=gen)
    x = torch.randn(N, w, generator=gen)
    torch.manual_seed(11)
    mlp = DenseNetLike(layers)
    lin = [m for m in mlp.layers if isinstance(m, torch.nn.Linear)]
    ws, bs = [l.weight.detach() for l in lin], [l.bias.detach() for l in lin]
    for aggr in ('mean', 'add'):
        conv = make_conv(_conv_cls(), ws, bs, torch.randn(w, w) * 0.1, torch.randn(w) * 0.1, aggr, w, w,
                         precision, dev)
        ref = O.nnconv_forward(x, ei, ea, ws, bs, conv.root.detach().cpu(), conv.bias.detach().cpu(), aggr)
        with torch.no_grad():
            out = conv(x.to(dev), ei.to(dev), ea.to(dev))
        assert rel_err(out, ref) < TOL[precision], (aggr, layers)


def test_edge_subset_call_and_zero_edges(dev):
    """MGKN style: N >> touched nodes, column-sliced edge_index view, no root / no bias; and E = 0."""
    gen = torch.Generator().manual_seed(9)
    N, E, w = 500, 3000, 64
    ei_all = torch.stack([torch.randint(0, 60, (E,), generator=gen), torch.randint(100, 180, (E,), generator=gen)])
    ei_all = ei_all[:, torch.argsort(ei_all[0], stable=True)]
    ea_all = torch.randn(E, 6, generator=gen)
    x = torch.randn(N, w, generator=gen)
    torch.manual_seed(3)
    mlp = DenseNetLike([6, 64, w * w])
    lin = [m for m in mlp.layers if isinstance(m, torch.nn.Linear)]
    ws, bs = [l.weight.detach() for l in lin], [l.bias.detach() for l in lin]
    conv = make_conv(_conv_cls(), ws, bs, None, None, 'mean', w, w, 'f16', dev)
    ei_d, ea_d, x_d = ei_all.to(dev), ea_all.to(dev), x.to(dev)
    a, b = 500, 2100
    with torch.no_grad():
        out = conv(x_d, ei_d[:, a:b], ea_d[a:b, :])          # non-contiguous view, as neurips1_MGKN.py:75
        out0 = conv(x_d, ei_d[:, 0:0], ea_d[0:0, :])
    ref = O.nnconv_forward(x, ei_all[:, a:b], ea_all[a:b], ws, bs, None, None, 'mean')
    assert rel_err(out, ref) < TOL['f16']
    assert float(out0.abs().max()) == 0.0


def test_properties_at_config2_size(dev):
    """BASELINE config 2 size (85x85, r=0.10, w=64, ker_width=1024): oracle on a sample of target nodes plus
    size-independent properties (linearity in x, mean == add / in-degree, determinism of the cached features)."""
    s, r, w, kw = 85, 0.10, 64, 1024
    ei = torch.from_numpy(O.ball_connectivity(s, r))
    assert ei.size(1) == 1466497                       # SURVEY 8(d): exact, no lattice ties
    rs = np.random.RandomState(0)
    theta = rs.randn(s * s)
    ea = torch.from_numpy(O.ball_edge_attr(O.square_grid(s), ei.numpy(), theta))
    torch.manual_seed(0)
    x = torch.randn(s * s, w)
    ws, bs, root, bias = O.reference_init(w, w, [6, kw, kw, w * w], seed=0)
    conv = make_conv(_conv_cls(), ws, bs, root, bias, 'mean', w, w, 'f16', dev)
    conv_add = make_conv(_conv_cls(), ws, bs, None, None, 'add', w, w, 'f16', dev)
    conv_mean = make_conv(_conv_cls(), ws, bs, None, None, 'mean', w, w, 'f16', dev)
    ei_d, ea_d, x_d = ei.to(dev), ea.to(dev), x.to(dev)
    with torch.no_grad():
        out = conv(x_d, ei_d, ea_d)
        out2 = conv(2.5 * x_d, ei_d, ea_d)
        o_add = conv_add(x_d, ei_d, ea_d)
        o_mean = conv_mean(x_d, ei_d, ea_d)
    # oracle on the edges that end in 24 sampled target nodes
    nodes = torch.from_numpy(rs.choice(s * s, 24, replace=False))
    mask = torch.isin(ei[1], nodes)
    ref = O.nnconv_forward(x, ei[:, mask], ea[mask], ws, bs, root, bias, 'mean', edge_chunk=2048)
    assert rel_err(out.cpu()[nodes], ref[nodes]) < TOL['f16']
    # linearity in x (bias is the only affine part)
    lin_err = rel_err(out2 - bias.to(dev), 2.5 * (out - bias.to(dev)))
    assert lin_err < 2e-3
    deg = torch.zeros(s * s).index_add_(0, ei[1], torch.ones(ei.size(1))).clamp(min=1).to(dev)
    assert rel_err(o_mean, o_add / deg[:, None]) < 1e-5


@pytest.fixture
def lib_options():
    """Set library knobs (nnconv_set_option) for one test and restore the defaults afterwards."""
    from graph_pde_b200 import _lib
    touched = []

    def setter(name, value):
        touched.append(name)
        _lib.set_option(name, value)
    yield setter
    for name in touched:
        _lib.set_option(name, None)


@pytest.mark.parametrize('knob', ['no_fuse', 'no_pipe+no_fuse', 'ring=4', 'small_ring', 'no_coop', 'gemm_direct_store', 'scatter_mode=0',
                                  'apply_passes=2'])
def test_alternative_schedules_give_the_same_answer(dev, knob, monkeypatch, lib_options):
    """The fused persistent kernel (default, cooperative launch), the same kernel launched plainly (no_coop), the
    per-batch PDL-pipelined kernels (no_fuse) and the plain stream-ordered kernels (no_pipe) must agree; a tiny Y
    ring forces many batches through the flag protocol."""
    from graph_pde_b200 import nn_conv
    for kv in knob.split('+'):
        if kv == 'small_ring':
            monkeypatch.setattr(nn_conv, '_Y_BYTES', 64 * 64 * 2 * 64 * 3)      # G3: Kp = 64, out = 64 ... many batches
        elif '=' in kv:
            k, v = kv.split('=')
            lib_options(k, int(v))
        else:
            lib_options(kv, 1)
    g = np.load(os.path.join(GOLDEN, 'g3_checkpoint_grain_new.npz'))
    st = {k[2:]: g[k] for k in g.files if k.startswith('w/')}
    ws = [st['conv1.nn.layers.%d.weight' % i] for i in (0, 2, 4)]
    bs = [st['conv1.nn.layers.%d.bias' % i] for i in (0, 2, 4)]
    conv = make_conv(_conv_cls(), ws, bs, st['conv1.root'], st['conv1.bias'], 'mean', 64, 64, 'f16', dev)
    ei, ea = ei64(g['edge_index']).to(dev), t(g['edge_attr']).to(dev)
    x = t(g['x0']).to(dev)
    with torch.no_grad():
        for k in range(6):
            x = torch.relu(conv(x, ei, ea))
            assert rel_err(x, t(g['x_after'][k])) < TOL['f16'], (knob, k)


def test_block_diagonal_batch_equals_per_graph(dev):
    """PyG Batch collation (block-diagonal edge_index, node offset): batched conv == per-graph conv
    (UAI3_resolution.py:191 uses batch 10); also the drop-in DataLoader's collation rule."""
    gen = torch.Generator().manual_seed(21)
    w = 64
    torch.manual_seed(5)
    mlp = DenseNetLike([6, 64, w * w])
    lin = [m for m in mlp.layers if isinstance(m, torch.nn.Linear)]
    ws, bs = [l.weight.detach() for l in lin], [l.bias.detach() for l in lin]
    conv = make_conv(_conv_cls(), ws, bs, torch.randn(w, w) * 0.1, torch.randn(w) * 0.1, 'mean', w, w, 'f16', dev)
    graphs_ = []
    for n, e in ((50, 400), (80, 900), (33, 100)):
        ei = torch.stack([torch.randint(0, n, (e,), generator=gen), torch.randint(0, n, (e,), generator=gen)])
        graphs_.append((torch.randn(n, w, generator=gen), ei, torch.randn(e, 6, generator=gen)))
    with torch.no_grad():
        singles = [conv(x.to(dev), ei.to(dev), ea.to(dev)) for x, ei, ea in graphs_]
        off = np.cumsum([0] + [g[0].size(0) for g in graphs_])
        xb = torch.cat([g[0] for g in graphs_]).to(dev)
        eib = torch.cat([g[1] + int(o) for g, o in zip(graphs_, off)], dim=1).to(dev)
        eab = torch.cat([g[2] for g in graphs_]).to(dev)
        outb = conv(xb, eib, eab)
    assert rel_err(outb, torch.cat(singles)) < 5e-4


@pytest.mark.parametrize('precision', ['f16', 'bf16'])
@pytest.mark.parametrize('knob', ['', 'no_fuse'])
def test_node_features_beyond_fp16_range(dev, precision, knob, lib_options):
    """Node features far outside the fp16 range (an untrained MGKN V-cycle reaches 5e5 after four depth
    iterations), rows of very different magnitude and all-zero rows: the 16-bit operand rows are normalised by a
    power of two per source (k_src_prep) so the result stays within the stated tolerance of the fp32 reference."""
    if knob:
        lib_options(knob, 1)
    torch.manual_seed(11)
    s, r, w, kw = 12, 0.3, 32, 64
    ei = torch.as_tensor(np.asarray(O.ball_connectivity(s, r))).long()
    grid = torch.as_tensor(np.asarray(O.square_grid(s))).float()
    ea = torch.cat([grid[ei[0]], grid[ei[1]], torch.randn(ei.size(1), 2)], dim=1).float()
    ws, bs, root, bias = O.reference_init(w, w, [6, kw, kw, w * w], True, True, seed=5)
    n = s * s
    x = torch.randn(n, w)
    mag = torch.tensor([3e5, 1.0, 2e-6, 7e7])[torch.arange(n) % 4]
    x = x * mag[:, None]
    x[5] = 0.0
    x[17] = 0.0
    ref = O.nnconv_forward(x.double(), ei, ea.double(), [v.double() for v in ws], [v.double() for v in bs],
                           root.double(), bias.double(), 'mean', w, w)
    conv = make_conv(_conv_cls(), ws, bs, root, bias, 'mean', w, w, precision, dev)
    with torch.no_grad():
        out = conv(x.to(dev), ei.to(dev), ea.to(dev))
    assert bool(torch.isfinite(out).all())
    assert rel_err(out, ref) < TOL[precision]
    # per-row check on the small-magnitude destinations is meaningless (they receive from large sources); instead
    # check linearity in x, which the exact power-of-two scaling must preserve to rounding
    with torch.no_grad():
        out4 = conv((4.0 * x).to(dev), ei.to(dev), ea.to(dev))
    lin_ref = 4.0 * (out - bias.to(dev)) + bias.to(dev)
    assert rel_err(out4, lin_ref) < 1e-5


@pytest.mark.parametrize('precision', ['f16', 'bf16'])
def test_low_out_degree_graph_uses_per_edge_kernel_matrices(dev, precision, edge_kernel_mode):
    """The 1-D multipole stencils of MGKN_orthogonal_burgers1d.py give every node 2-4 out-edges: the conv switches
    to formulation B (K_e built once by the tcgen05 GEMM, one streaming pass per application) and must agree with
    the oracle and with formulation C on the same inputs."""
    from graph_pde_b200 import graphs, nn_conv
    if edge_kernel_mode == 'off':
        pytest.skip('this test switches the mode itself')
    s, w, kw = 512, 64, 128
    X, eis, eas = graphs.multi_pole_grid1d(torch.randn(s, generator=torch.Generator().manual_seed(0)), s, is_periodic=True,
                                           levels=3)
    ei, ea = eis[1], eas[1]                          # interactive neighbours of the finest level: 4 out-edges per node
    ws, bs, root, bias = O.reference_init(w, w, [4, kw, kw, w * w], True, True, seed=4)
    x = torch.randn(s, w, generator=torch.Generator().manual_seed(1))
    ref = O.nnconv_forward(x, ei, ea, ws, bs, root, bias, 'mean')
    conv = make_conv(_conv_cls(), ws, bs, root, bias, 'mean', w, w, precision, dev)
    n0 = nn_conv.stats.get('edge_kernel_passes', 0)
    xd, eid, ead = x.to(dev), ei.to(dev), ea.to(dev)
    with torch.no_grad():
        out_b = conv(xd, eid, ead)
        out_b2 = conv(2.0 * xd, eid, ead)                            # second application reuses K_e
    assert nn_conv.stats.get('edge_kernel_passes', 0) == n0 + 1
    assert rel_err(out_b, ref) < TOL[precision]
    assert rel_err(out_b2 - bias.to(dev), 2.0 * (out_b - bias.to(dev))) < 1e-5
    old = nn_conv._EDGE_KERNELS
    nn_conv._EDGE_KERNELS = 'off'
    try:
        conv_c = make_conv(_conv_cls(), ws, bs, root, bias, 'mean', w, w, precision, dev)
        with torch.no_grad():
            out_c = conv_c(xd, eid, ead)
    finally:
        nn_conv._EDGE_KERNELS = old
    assert rel_err(out_b, out_c) < 2 * TOL[precision]


@pytest.mark.gpu
@pytest.mark.parametrize('precision', ['f16', 'bf16', 'f16x2', 'fp32'])
@pytest.mark.parametrize('flags', ['', 'root', 'root+bias'])
def test_residual_step_equals_conv_add_on_preactivations(dev, precision, flags, edge_kernel_mode):
    """`residual_step` (nnconv_apply_ex / nnconv_apply_edge_ex with NNCONV_APPLY_RELU_IN | NNCONV_APPLY_RESIDUAL) against
    the reference's op sequence `relu(z) + conv(relu(z))` (neurips1_MGKN.py:76) -- oracle and this library's own plain
    application -- on a graph with a hub, isolated nodes and duplicate edges, and on a chain of three steps."""
    gen = torch.Generator().manual_seed(9)
    N, E, w, kw = 260, 3000, 64, 64
    src = torch.randint(0, N - 15, (E,), generator=gen)
    dst = torch.randint(5, N, (E,), generator=gen)
    src[:300] = 3
    src[400:406], dst[400:406] = src[400], dst[400]
    ei, ea = torch.stack([src, dst]), torch.rand(E, 6, generator=gen)
    z = torch.randn(N, w, generator=gen)
    ws, bs, root, bias = O.reference_init(w, w, [6, kw, kw, w * w], True, True, seed=3)
    root = root if 'root' in flags else None
    bias = bias if 'bias' in flags else None
    conv = make_conv(_conv_cls(), ws, bs, root, bias, 'mean', w, w, precision, dev)
    zd, eid, ead = z.to(dev), ei.to(dev), ea.to(dev)
    x = torch.relu(z)
    ref = x + O.nnconv_forward(x, ei, ea, ws, bs, root, bias, 'mean')
    with torch.no_grad():
        out = conv.residual_step(zd, eid, ead, relu_in=True)
        plain = torch.relu(zd) + conv(torch.relu(zd), eid, ead)
        out_lin = conv.residual_step(zd, eid, ead, relu_in=False)
        plain_lin = zd + conv(zd, eid, ead)
    assert rel_err(out, ref) < TOL[precision]
    assert rel_err(out, plain) < 2e-6             # same kernels, only the fp32 summation order differs
    assert rel_err(out_lin, plain_lin) < 2e-6
    with torch.no_grad():                         # chain: z3 = step(step(step(z))) vs the op-by-op sequence
        zc, pc = zd, zd
        for k in range(3):
            zc = conv.residual_step(zc, eid, ead, relu_in=k > 0)
            a = torch.relu(pc) if k > 0 else pc
            pc = a + conv(a, eid, ead)
        # a 1e-7 summation-order difference can flip a 16-bit operand rounding of the next step (bf16: 8x coarser)
        assert rel_err(zc, pc) < (1e-3 if precision == 'bf16' else 1e-4)
    with pytest.raises(RuntimeError):
        conv.residual_step(zd.clone().requires_grad_(True), eid, ead)


@pytest.mark.gpu
@pytest.mark.parametrize('ring_deep', [1, 0])
def test_deep_y_ring_for_narrow_edge_networks(dev, ring_deep, lib_options, edge_kernel_mode):
    """ker_width 128 -> 16 KB of Y per source, so the 48 MiB Y budget holds every one of the 1900 sources: the fused
    kernel runs 15 batches of 128 sources through a 14-deep ring (option `ring_deep`) instead of 3 batches of 640
    through a 3-deep one (default); both schedules against the oracle, T = 3 applications."""
    if edge_kernel_mode != 'off':
        pytest.skip('the persistent fused kernel is the subject')
    lib_options('ring_deep', ring_deep)
    gen = torch.Generator().manual_seed(21)
    N, S, w, kw = 2000, 1900, 64, 128
    deg = torch.randint(8, 40, (S,), generator=gen)
    src = torch.repeat_interleave(torch.arange(S), deg)
    E = int(src.numel())
    dst = torch.randint(0, N, (E,), generator=gen)
    ei, ea = torch.stack([src, dst]), torch.rand(E, 6, generator=gen)
    ws, bs, root, bias = O.reference_init(w, w, [6, kw, kw, w * w], True, True, seed=8)
    conv = make_conv(_conv_cls(), ws, bs, root, bias, 'mean', w, w, 'f16', dev)
    x = torch.randn(N, w, generator=gen)
    xd, eid, ead = x.to(dev), ei.to(dev), ea.to(dev)
    for _ in range(3):
        ref = O.nnconv_forward(x, ei, ea, ws, bs, root, bias, 'mean')
        with torch.no_grad():
            out = conv(xd, eid, ead)
        assert rel_err(out, ref) < TOL['f16']
        x = torch.relu(ref)
        xd = x.to(dev)


@pytest.mark.gpu
@pytest.mark.parametrize('w', [32, 64])
@pytest.mark.parametrize('precision', ['f16', 'bf16'])
def test_per_edge_kernels_warp_per_source_and_warp_per_edge(dev, precision, w):
    """Formulation B's two application kernels in their 16-byte-load form (in = out = 32 / 64): >= 2048 sources with 2-4
    out-edges each run one warp per source (`k_apply_edge_src_v`), fewer sources one warp per edge (`k_apply_edge_v`)."""
    from graph_pde_b200 import graphs, nn_conv
    old = nn_conv._EDGE_KERNELS
    nn_conv._EDGE_KERNELS = 'on'
    try:
        for s in (4096, 256):
            X, eis, eas = graphs.multi_pole_grid1d(torch.randn(s, generator=torch.Generator().manual_seed(2)), s,
                                                   is_periodic=True, levels=2)
            ei, ea = eis[1], eas[1]
            ws, bs, root, bias = O.reference_init(w, w, [4, 32, 32, w * w], True, True, seed=6)
            x = torch.randn(s, w, generator=torch.Generator().manual_seed(3))
            ref = O.nnconv_forward(x, ei, ea, ws, bs, root, bias, 'mean')
            conv = make_conv(_conv_cls(), ws, bs, root, bias, 'mean', w, w, precision, dev)
            with torch.no_grad():
                out = conv(x.to(dev), ei.to(dev), ea.to(dev))
                z = conv.residual_step(x.to(dev), ei.to(dev), ea.to(dev), relu_in=True)
            assert rel_err(out, ref) < TOL[precision], (s, w)
            xr = torch.relu(x)
            assert rel_err(z, xr + O.nnconv_forward(xr, ei, ea, ws, bs, root, bias, 'mean')) < TOL[precision], (s, w)
    finally:
        nn_conv._EDGE_KERNELS = old
