"""Shared helpers for the parity tests (CPU side: golden loaders; GPU side: module builders)."""
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')

# stated tolerances: max|out - ref| / max|ref| per tensor-core operand precision (DESIGN.md "Precision")
TOL = {'fp32': 2e-5, 'f16x2': 2e-5, 'f16': 2e-3, 'bf16': 2e-2}


def t(a):
    return torch.from_numpy(np.asarray(a))


def ei64(a):
    return torch.from_numpy(np.asarray(a).astype(np.int64))


def rel_err(out, ref):
    out = out.detach().double().cpu()
    ref = ref.detach().double().cpu()
    return float((out - ref).abs().max() / ref.abs().max().clamp(min=1e-30))


def cfg1_weights(g):
    """Re-draw the seeded KernelNN(w=32, kw=1024) parameters of golden G2 (same stream as the reference)."""
    w, kw = int(g['width']), int(g['ker_width'])
    torch.manual_seed(0)
    fc1 = torch.nn.Linear(6, w)
    lins = [torch.nn.Linear(a, b) for a, b in zip([6, kw, kw], [kw, kw, w * w])]
    for lin in lins:
        lin.reset_parameters()
    root = torch.empty(w, w).uniform_(-1 / np.sqrt(w), 1 / np.sqrt(w))
    bias = torch.empty(w).uniform_(-1 / np.sqrt(w), 1 / np.sqrt(w))
    return fc1, [l.weight.detach() for l in lins], [l.bias.detach() for l in lins], root, bias


def vcycle_weights(g, variant):
    """Parameters of the golden G4 model `variant` ('neurips1': KernelInduced, 'general': MKGN) as numpy arrays.
    G4 stores their seed, shapes and sha256 instead of the values: they are re-drawn here with this project's
    constructors, which draw the reference classes' init stream, and must hash to the reference's bytes."""
    import hashlib
    from graph_pde_b200.models import MKGN, KernelInduced
    pts = [int(p) for p in g['points']]
    cls = KernelInduced if variant == 'neurips1' else MKGN
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(int(g[variant + '/seed']))
        model = cls(width=int(g['width']), ker_width=int(g['ker_width']), depth=int(g['depth']), ker_in=6, points=pts,
                    level=len(pts), in_width=6)
    st = {k: v.detach().numpy().copy() for k, v in model.state_dict().items()}
    pre = variant + '/sha256/'
    assert sorted(st) == sorted(k[len(pre):] for k in g.files if k.startswith(pre))
    for k, v in st.items():
        assert hashlib.sha256(v.tobytes()).hexdigest() == str(g[pre + k]), 're-drawn %s/%s differs' % (variant, k)
    return st


class DenseNetLike(torch.nn.Module):
    """Same module tree / state-dict keys as the reference's DenseNet (utilities.py:201-227):
    self.layers = ModuleList([Linear, ReLU, Linear, ..., Linear])."""

    def __init__(self, layers):
        super().__init__()
        self.layers = torch.nn.ModuleList()
        for j in range(len(layers) - 1):
            self.layers.append(torch.nn.Linear(layers[j], layers[j + 1]))
            if j != len(layers) - 2:
                self.layers.append(torch.nn.ReLU())

    def forward(self, x):
        for l in self.layers:
            x = l(x)
        return x


def make_conv(cls, ws, bs, root, bias, aggr, cin, cout, precision, device):
    dims = [ws[0].shape[1]] + [w.shape[0] for w in ws]
    mlp = DenseNetLike(dims)
    conv = cls(cin, cout, mlp, aggr=aggr, root_weight=root is not None, bias=bias is not None, precision=precision)
    with torch.no_grad():
        lin = [m for m in mlp.layers if isinstance(m, torch.nn.Linear)]
        for l, w, b in zip(lin, ws, bs):
            l.weight.copy_(torch.as_tensor(w))
            l.bias.copy_(torch.as_tensor(b))
        if root is not None:
            conv.root.copy_(torch.as_tensor(root))
        if bias is not None:
            conv.bias.copy_(torch.as_tensor(bias))
    return conv.to(device)


def oracle_stack_on_cuda(x, ei, ea, ws, bs, root, bias, depth, aggr='mean', edge_chunk=65536, relu_last=True):
    """The reference-equivalent torch ops (oracle port) on CUDA tensors, fp32 with TF32 off: the checker for the
    full-size configurations (the CPU oracle would need minutes to hours there)."""
    from oracle import nnconv_oracle as O
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            outs = []
            for k in range(depth):
                x = O.nnconv_forward(x, ei, ea, ws, bs, root, bias, aggr, edge_chunk=edge_chunk)
                if relu_last or k != depth - 1:
                    x = torch.relu(x)
                outs.append(x)
            return outs
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


# ---- mask-consistent references for the 16-bit GRADIENT tests -------------------------------------------------
# The gradient of a ReLU network is discontinuous in its pre-activations: a 16-bit forward flips the ReLU mask of the
# ~1e-4 fraction of units whose pre-activation is within rounding distance of zero, and in a sum of N random-sign
# terms that fraction p shows up as a sqrt(p) ~ 1e-2 relative change of the parameter gradients -- of the function
# the 16-bit forward actually computes, which is what the backward must (and does) differentiate.  The tight
# gradient tests therefore compare against autograd through a forward that rounds at the SAME points as the kernels
# (straight-through rounding: values rounded, gradients passed), restating oracle.nnconv_forward
# (graph-neural-operator/nn_conv.py:267-282, utilities.py:223-227); the exact fp64 oracle is kept as a loose bound.
def ste_round(t, prec):
    dt = torch.float16 if prec in ('f16', 'fp16') else torch.bfloat16
    return t + (t.to(dt).to(t.dtype) - t).detach()


def emulated_nnconv_forward(x, edge_index, edge_attr, weights, biases, root, bias, aggr, prec, edge_chunk=None):
    n, cin = x.shape
    cout = weights[-1].size(0) // cin
    e_total = edge_index.size(1)
    step = e_total if not edge_chunk else edge_chunk
    out = torch.zeros(n, cout, dtype=x.dtype, device=x.device)
    wq = [weights[0]] + [ste_round(w, prec) for w in weights[1:-1]]      # layer 1 runs fp32-grade (hi/lo split)
    for s0 in range(0, max(e_total, 1), max(step, 1)):
        sl = slice(s0, min(s0 + step, e_total))
        h = edge_attr[sl]
        for l in range(len(weights) - 1):
            h = ste_round(torch.relu(h @ wq[l].t() + biases[l]), prec)   # activations are stored in 16 bit
        k = (h @ weights[-1].t() + biases[-1]).view(-1, cin, cout)
        msg = torch.matmul(x.index_select(0, edge_index[0, sl]).unsqueeze(1), k).squeeze(1)
        out = out.index_add(0, edge_index[1, sl], msg)
    if aggr == 'mean':
        cnt = torch.zeros(n, dtype=x.dtype, device=x.device).index_add_(
            0, edge_index[1], torch.ones(e_total, dtype=x.dtype, device=x.device))
        out = out / cnt.clamp(min=1).unsqueeze(-1)
    if root is not None:
        out = out + x @ root
    if bias is not None:
        out = out + bias
    return out
