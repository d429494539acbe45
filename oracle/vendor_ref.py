"""Put an UNMODIFIED copy of the reference's hot-path files under oracle/_ref/ (git-ignored build output) so that
`bench.py --impl reference` times the reference's OWN code.

TEST / MEASUREMENT INFRASTRUCTURE, never imported by the product path.

The reference is a directory of scripts without setup.py / pyproject.toml, so there is nothing to pip-install;
this recipe is the equivalent: from the reference checkout (REF: $GRAPH_PDE_REFERENCE, default /root/reference) it
copies, byte for byte,
    graph-neural-operator/nn_conv.py          (NNConv_old: the operator)
    graph-neural-operator/utilities.py        (DenseNet: the edge MLP)
    multipole-graph-neural-operator/utilities.py
and records their sha256 in oracle/_ref/MANIFEST.json.  Third-party torch_geometric / torch_scatter are
not needed: the copied files run over oracle/pyg_stub, the restated MessagePassing boundary (see its docstring).
When REF is absent or unreadable nothing is copied and the benchmark's CPU baseline uses the oracle port instead.
Nothing is copied into tracked paths.
"""
import hashlib
import json
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DST = os.path.join(HERE, '_ref')
REF = os.environ.get('GRAPH_PDE_REFERENCE') or '/root/reference'
FILES = [
    ('graph-neural-operator/nn_conv.py', 'graph-neural-operator/nn_conv.py'),
    ('graph-neural-operator/utilities.py', 'graph-neural-operator/utilities.py'),
    ('multipole-graph-neural-operator/utilities.py', 'multipole-graph-neural-operator/utilities.py'),
]


def vendor(verbose=False):
    """Returns True when oracle/_ref holds the files (copied now or earlier), False when there is no
    reference to copy from and nothing was vendored before."""
    if not all(os.access(os.path.join(REF, src), os.R_OK) for src, _ in FILES):
        return os.path.exists(os.path.join(DST, 'MANIFEST.json'))
    manifest = {}
    for src, dst in FILES:
        s, d = os.path.join(REF, src), os.path.join(DST, dst)
        os.makedirs(os.path.dirname(d), exist_ok=True)
        shutil.copyfile(s, d)
        manifest[dst] = hashlib.sha256(open(d, 'rb').read()).hexdigest()
        if verbose:
            print('vendored', src, manifest[dst][:12])
    json.dump(dict(source=REF, files=manifest), open(os.path.join(DST, 'MANIFEST.json'), 'w'), indent=1)
    return True


def import_reference_gno():
    """(nn_conv, utilities) modules of the vendored copy, imported over oracle/pyg_stub; None if not vendored."""
    gno = os.path.join(DST, 'graph-neural-operator')
    if not os.path.exists(os.path.join(gno, 'nn_conv.py')):
        return None
    import importlib.util
    stub = os.path.join(HERE, 'pyg_stub')
    added = [p for p in (stub, gno) if p not in sys.path]
    sys.path[:0] = added
    try:
        mods = []
        for name in ('utilities', 'nn_conv'):
            spec = importlib.util.spec_from_file_location('graph_pde_ref_' + name, os.path.join(gno, name + '.py'))
            m = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(m)
            mods.append(m)
        return mods[1], mods[0]
    finally:
        for p in added:
            sys.path.remove(p)


if __name__ == '__main__':
    print('vendored' if vendor(verbose=True) else 'no reference available')
