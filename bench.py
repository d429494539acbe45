#!/usr/bin/env python
"""bench.py -- NNConv edge-applications/s on synthetic Darcy-2D radius graphs (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload darcy241|darcy85]
                    [--dump-outputs DIR]

One "step" = one KernelNN conv stack (T applications of the shared NNConv, graph-neural-operator/
UAI1_full_resolution.py:29-30) over ONE graph sample per GPU: the x-independent edge features are
recomputed every step (each step is a new sample: new edge_attr), then T applications run.
value = (ranks x E x T x K) / max-over-ranks device time  [edge-applications/s], inputs resident in HBM.
e2e   = same through the public module call KernelNN.forward with pinned-host inputs copied H2D and the
        result read back D2H inside the timed region, every step.
Weak scaling: every rank owns its own graph sample(s); no data-path collective (batch sharding).
--steps K sets the timed steps of value and e2e (the metric); the secondary lines keep fixed step counts: train
2..3 steps (K clamped), fp32_grade 3, configs 3-50 repetitions, gpu_reference_port 1, cpu_baseline 2, strip 2..5.
--impl reference: the CPU oracle port (oracle/nnconv_oracle.py, torch CPU, all host threads) on a bounded
sample of the same workload (rank 0 only).
--dump-outputs DIR: after the timed steps, rank 0 writes what the last timed step of each timed path returned,
DIR/conv_stack.npy (resident path: node features after the T applications, [N, width]) and DIR/model_out.npy
(e2e path: KernelNN.forward, [N, 1]), float32.  Inputs and weights are seeded, so two builds run with the same
arguments can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # BASELINE.json configs[2] / metric config: Darcy-2D 241^2, r=0.05, w=64, T=6 (ker_width of the named
    # script UAI1_full_resolution.py:57 = 1024); ties-in rule -> E = 24,557,297
    'darcy241': dict(s=241, r=0.05, width=64, ker_width=1024, depth=6),
    # BASELINE.json configs[1]
    'darcy85': dict(s=85, r=0.10, width=64, ker_width=1024, depth=6),
    # BASELINE.json configs[0] (CPU-runnable case)
    'darcy16': dict(s=16, r=0.25, width=32, ker_width=1024, depth=4),
}
KIND_NAMES = ['edge_layer1', 'hidden_gemm', 'node_prologue', 'y_gemm', 'conv_scatter', 'apply_fused']


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d['hbm_gbs'], tf_burst=d['bf16_tflops'], tf_sustained=d.get('bf16_tflops_sustained',
                    d['bf16_tflops']), source='measured')
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source='fallback')


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm = []
        mx = None
        reasons = set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith('active'):
                        reasons.add(nm)
            except Exception:
                continue
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=mx, reasons=sorted(reasons),
                    samples=len(sm))


REF_SAMPLE_SOURCES = 192     # fixed, so that reference-arm numbers are comparable run to run


def cpu_reference_rate(cfg, steps=1, warmup=0, n_src=REF_SAMPLE_SOURCES):
    """The reference's CPU path on a bounded, FIXED sample: out-edges of the first n_src source nodes of the
    workload graph, T applications of one NNConv.  Runs the reference's OWN files (oracle/_ref, vendored
    unmodified by oracle/vendor_ref.py; kind 'reference') over oracle/pyg_stub, exactly as the reference runs them
    (one shot over all edges of the sample, torch CPU fp32); falls back to the oracle port (kind 'port') only when
    the vendored copy is absent.  Returns (edge_apps_per_s, cores, kind, sample_description, ms_per_step)."""
    from graph_pde_b200 import graphs
    from oracle import nnconv_oracle as O
    from oracle import vendor_ref
    cores = os.cpu_count() or 1
    s, r, w, kw, T = cfg['s'], cfg['r'], cfg['width'], cfg['ker_width'], cfg['depth']
    n = s * s
    n_src = min(n, n_src)
    torch.manual_seed(0)
    grid = graphs.square_grid(s)
    theta = torch.randn(n)
    x = torch.randn(n, w)
    ei = graphs.ball_connectivity(s, r, 'cpu', True, nodes=(0, n_src))
    ea = graphs.ball_edge_attr(grid, ei, theta)
    ref = vendor_ref.import_reference_gno()
    if ref is not None:
        ref_nn_conv, ref_util = ref
        torch.manual_seed(0)
        kernel = ref_util.DenseNet([6, kw, kw, w * w], torch.nn.ReLU)
        conv = ref_nn_conv.NNConv_old(w, w, kernel, aggr='mean')
        kind = 'reference'

        def stack():
            h = x
            for _ in range(T):                                # UAI1_full_resolution.py:29-30
                h = torch.relu(conv(h, ei, ea))
            return h
    else:
        ws, bs, root, bias = O.reference_init(w, w, [6, kw, kw, w * w], seed=0)
        kind = 'port'

        def stack():
            return O.kernelnn_conv_stack(x, ei, ea, ws, bs, root, bias, T, 'mean')

    def run():
        t0 = time.perf_counter()
        with torch.no_grad():
            stack()
        return time.perf_counter() - t0

    torch.set_num_threads(cores)
    run()                                         # first-call warm-up (thread pool, allocator)
    # "all the host threads it can use": more threads than the GEMMs can feed only adds contention on
    # big boxes, so pick the fastest power-of-two thread count up to the core count on the same sample.
    best = (float('inf'), cores)
    for c in sorted({c for c in (cores, 64, 32, 16, 8) if c <= cores}, reverse=True):
        torch.set_num_threads(c)
        dt = run()
        if dt < best[0]:
            best = (dt, c)
    cores = best[1]
    torch.set_num_threads(cores)
    for _ in range(warmup):
        run()
    times = [run() for _ in range(max(1, steps))]
    tot = sum(times)
    desc = ('out-edges of the first %d of %d source nodes of the %dx%d r=%g graph (%d edges) x T=%d, fp32, '
            'torch CPU %d threads, %s' % (n_src, n, s, s, r, ei.size(1), T, cores,
                                          "reference's own nn_conv.py + utilities.py over oracle/pyg_stub, one shot"
                                          if kind == 'reference' else 'oracle port'))
    return ei.size(1) * T * len(times) / tot, cores, kind, desc, 1e3 * tot / len(times)


def gpu_reference_rate(cfg, dev, n_src=2048, chunk=65536):
    """SURVEY 8(d)(ii): the reference-equivalent PyTorch path (the oracle port, fp32, allow_tf32=False, scatter =
    index_add_) on CUDA tensors, edge-chunked, on a bounded sample -- the 'reference single-GPU path' the north
    star's >= 10x refers to.  CUDA-event timing.  Baseline only; never part of the product path."""
    from graph_pde_b200 import graphs
    from oracle import nnconv_oracle as O
    s, r, w, kw, T = cfg['s'], cfg['r'], cfg['width'], cfg['ker_width'], cfg['depth']
    n = s * s
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        ws, bs, root, bias = O.reference_init(w, w, [6, kw, kw, w * w], seed=0)
        ws, bs, root, bias = [t.to(dev) for t in ws], [t.to(dev) for t in bs], root.to(dev), bias.to(dev)
        n_src = min(n, n_src)
        ei = graphs.ball_connectivity(s, r, dev, True, nodes=(0, n_src))
        grid = graphs.square_grid(s, dev)
        ea = graphs.ball_edge_attr(grid, ei, torch.randn(n, device=dev))
        x = torch.randn(n, w, device=dev)

        def run():
            with torch.no_grad():
                O.kernelnn_conv_stack(x, ei, ea, ws, bs, root, bias, T, 'mean', edge_chunk=chunk)
        run()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        run()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    return dict(value=ei.size(1) * T / (ms * 1e-3), unit='edge-apps/s', kind='port-on-cuda',
                sample='out-edges of the first %d source nodes (%d edges) x T=%d, fp32 torch ops (allow_tf32=False), '
                       'edge_chunk %d, one timed pass after one warm-up' % (n_src, ei.size(1), T, chunk))


TOL = {'f16': 2e-3, 'bf16': 2e-2, 'f16x2': 2e-5, 'fp32': 2e-5}   # stated tolerances (DESIGN.md section 5)


def oracle_stack_cuda(cfg, model, x0, ei, ea, chunk=1 << 16):
    """The FULL workload graph, all T applications, through the reference-equivalent fp32 torch ops (oracle port,
    TF32 off) on CUDA tensors, edge-chunked -- the checker for the parity field.  ~30 s at 241^2."""
    from oracle import nnconv_oracle as O
    lin = [m for m in model.conv1.nn.layers if isinstance(m, torch.nn.Linear)]
    ws = [l.weight.detach().float() for l in lin]
    bs = [l.bias.detach().float() for l in lin]
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            return O.kernelnn_conv_stack(x0, ei, ea, ws, bs, model.conv1.root.detach(), model.conv1.bias.detach(),
                                         cfg['depth'], 'mean', edge_chunk=chunk)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def rel_err(out, ref):
    return float((out.double() - ref.double()).abs().max() / ref.double().abs().max().clamp(min=1e-30))


def _time_ms(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """Write {name: tensor} as path/<name>.npy in float32 (darcy241: 15 MB in all)."""
    arrays = {name: t.detach().float().cpu().numpy() for name, t in arrays.items()}
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_MAX_BYTES, 'outputs larger than DUMP_MAX_BYTES'
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + '.npy'), a)


def other_configs(dev, precision):
    """The BASELINE.json configs that are not the metric configuration, each as value + parity (rank 0, one GPU):
    config 2 (GKN 85^2), config 4 (MGKN V-cycle, neurips1_MGKN.py case 0 on the 241^2 grid), config 5 (orthogonal MGKN,
    Burgers 1-D, s=8192, 5 levels).  Parity = whole-model output against the oracle port run with fp32 torch ops on
    the same GPU; `ref_ms` is that path's time (the 'reference single-GPU path')."""
    from graph_pde_b200 import GraphedForward, graphs, nn_conv
    from graph_pde_b200.models import MGKN, KernelInduced, KernelNN
    from oracle import nnconv_oracle as O
    out = {}
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            # ---- config 2
            cfg = WORKLOADS['darcy85']
            s, r, w, kw, T = cfg['s'], cfg['r'], cfg['width'], cfg['ker_width'], cfg['depth']
            torch.manual_seed(0)
            m = KernelNN(w, kw, T, 6, in_width=6, precision=precision).to(dev).eval()
            x6, ei, ea = graphs.darcy_sample(s, r, dev, seed=5)
            x0 = m.fc1(x6)

            def step2():
                m.conv1._h_cache.clear()
                return m.conv_stack(x0, ei, ea)
            ms = _time_ms(step2, 10)
            ref = oracle_stack_cuda(cfg, m, x0, ei, ea)
            out['darcy85'] = dict(config='GKN Darcy-2D 85x85 r=0.10 width=64 ker_width=1024 T=6 (BASELINE configs[1])',
                                  edges=int(ei.size(1)), value=ei.size(1) * T / (ms * 1e-3), unit='edge-apps/s', ms_per_step=ms,
                                  parity=dict(max_rel_err=rel_err(step2(), ref), tol=TOL.get(precision)),
                                  hbm_stream_frac=ei.size(1) * T * (2 * kw + 4) / (ms * 1e-3) / 1e9 / peaks()['hbm_gbs'])
            del m
            # ---- config 4
            torch.manual_seed(0)
            s4, mm = 241, [2400, 1600, 400, 100, 25]
            ri = [0.5 / 8 * 1.41, 0.5 / 8, 0.5 / 4, 0.5 / 2, 0.5]
            rx = [0.5 / 8 * 1.1, 0.5 / 8 * 1.41, 0.5 / 4 * 1.41, 0.5 / 2 * 1.41]
            t0 = time.perf_counter()
            g = graphs.multi_level_ball_graph(s4, mm, ri, rx, theta=torch.randn(s4 * s4), device=dev)
            torch.cuda.synchronize()
            build_ms = (time.perf_counter() - t0) * 1e3
            depth = 4
            mk = KernelInduced(width=64, ker_width=256, depth=depth, ker_in=6, points=mm, level=len(mm), in_width=6,
                               precision=precision).to(dev).eval()
            g.x = torch.randn(sum(mm), 6, device=dev)
            ea4 = depth * (g.edge_index_mid.size(1) + g.edge_index_down.size(1) + g.edge_index_up.size(1))
            o4 = mk(g)
            ms_e = _time_ms(lambda: mk(g), 20)
            l0 = nn_conv.stats['launches']
            mk(g)
            launches = nn_conv.stats['launches'] - l0
            ms_g = None
            try:
                gf = GraphedForward(mk, g)
                ms_g = _time_ms(gf.replay, 50)
            except Exception:      # capture is an optimisation; the eager number stands on its own
                pass
            p = {k: v.detach() for k, v in mk.state_dict().items()}
            data = dict(edge_index_down=g.edge_index_down, edge_index_mid=g.edge_index_mid, edge_index_up=g.edge_index_up,
                        edge_attr_down=g.edge_attr_down, edge_attr_mid=g.edge_attr_mid, edge_attr_up=g.edge_attr_up,
                        range_down=g.edge_index_down_range.tolist(), range_mid=g.edge_index_range.tolist(),
                        range_up=g.edge_index_up_range.tolist())
            ref4 = O.mgkn_vcycle_forward(g.x, data, p, depth, len(mm), mm, variant='neurips1')
            ms_r = _time_ms(lambda: O.mgkn_vcycle_forward(g.x, data, p, depth, len(mm), mm, variant='neurips1'), 3, 1)
            out['mgkn241'] = dict(config='MGKN V-cycle (neurips1_MGKN.py case 0): 5 levels m=%s on the 241^2 grid, width 64, '
                                         'ker_width 256, depth 4 (BASELINE configs[3])' % mm,
                                  edge_apps_per_forward=int(ea4), value=ea4 / (ms_e * 1e-3), unit='edge-apps/s',
                                  ms_per_forward=ms_e, ms_per_forward_cuda_graph=ms_g, nnconv_launches_per_forward=int(launches),
                                  graph_build_ms=build_ms, ref_ms=ms_r,
                                  parity=dict(max_rel_err=rel_err(o4, ref4), tol=TOL.get(precision)))
            del mk, g
            # ---- config 5
            torch.manual_seed(0)
            s5, levels, width = 8192, 5, 64
            X, eis, eas = graphs.multi_pole_grid1d(torch.randn(s5), s5, is_periodic=True, levels=levels, device=dev)
            m5 = MGKN(width=width, ker_width=1024, depth=depth, ker_in=4, in_width=2, s=s5, precision=precision).to(dev).eval()
            data5 = (X, None, eis, eas)
            ea5 = depth * sum(e.size(1) for e in eis)
            o5 = m5(data5)
            ms_e = _time_ms(lambda: m5(data5), 20)
            ms_g = None
            try:
                gf = GraphedForward(m5, data5)
                ms_g = _time_ms(gf.replay, 50)
            except Exception:
                pass
            p5 = {k: v.detach() for k, v in m5.state_dict().items()}
            ref5 = O.mgkn_orthogonal_forward(X[0], eis, eas, p5, depth, width, s5)
            ms_r = _time_ms(lambda: O.mgkn_orthogonal_forward(X[0], eis, eas, p5, depth, width, s5), 3, 1)
            kbytes = sum(e.size(1) for e in eis) * depth * width * width * 2
            out['burgers8192'] = dict(config='orthogonal MGKN (MGKN_orthogonal_burgers1d.py), s=8192, 5 levels, width 64, '
                                             'ker_width 1024, depth 4 (BASELINE configs[4]); 2-4 out-edges per node -> per-edge '
                                             'kernel matrices (formulation B)',
                                      edge_sets=[int(e.size(1)) for e in eis], edge_apps_per_forward=int(ea5),
                                      value=ea5 / (ms_e * 1e-3), unit='edge-apps/s', ms_per_forward=ms_e,
                                      ms_per_forward_cuda_graph=ms_g, ref_ms=ms_r,
                                      kmat_stream_gb_per_forward=kbytes / 1e9,
                                      hbm_stream_frac=kbytes / ((ms_g or ms_e) * 1e-3) / 1e9 / peaks()['hbm_gbs'],
                                      parity=dict(max_rel_err=rel_err(o5, ref5), tol=TOL.get(precision)))
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
        torch.cuda.empty_cache()
    return out


def strip_child_main(args):
    """`bench.py --strip-only` (spawned by every rank of the main bench, own process group): ONE mesh cut into N row
    strips (strong scaling; SURVEY 8(e) "single big mesh").  Every rank owns the edges that END in its strip, computes
    their edge features, and the T applications exchange 2R boundary rows with the two neighbours by peer stores over
    NVLink (partition.PeerHalo, csrc/halo.cu) -- inside the timed region.  Runs in child processes so that a failure
    of the peer mapping on some box cannot take the headline line down with it.  Rank 0 prints one JSON object."""
    import torch.distributed as dist
    from graph_pde_b200 import graphs, partition
    from graph_pde_b200.models import KernelNN
    cfg = WORKLOADS[args.workload]
    rank, world, local_rank = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    dist.init_process_group('nccl', device_id=dev)
    s, r, w, kw, T = cfg['s'], cfg['r'], cfg['width'], cfg['ker_width'], cfg['depth']
    torch.manual_seed(0)
    model = KernelNN(w, kw, T, 6, in_width=6, precision=args.precision).to(dev).eval()
    ei = graphs.ball_connectivity(s, r, dev, True)
    E = ei.size(1)
    x6c, _, _ = graphs.darcy_sample(s, r, dev, seed=4242, edge_index=ei[:, :1])     # the SAME sample on every rank
    part = partition.StripPartition(s, r, rank, world, device=dev)
    grid = graphs.square_grid(s, dev)
    ea_loc = graphs.ball_edge_attr(grid, part.edge_index_global, x6c[:, 2])
    with torch.no_grad():
        x0g = model.fc1(x6c)
    x_loc = part.local_slice(x0g).clone()
    mode = 'peer stores + flags (CUDA IPC over NVLink)'
    try:
        halo = partition.PeerHalo(part, w, dev)
    except Exception as exc:                                   # e.g. IPC not permitted in this container
        halo = None
        mode = 'NCCL all-gather per application (peer mapping failed: %s)' % type(exc).__name__
    ok_all = torch.tensor([1 if halo is not None else 0], device=dev)
    dist.all_reduce(ok_all, op=dist.ReduceOp.MIN)
    if int(ok_all.item()) == 0 and halo is not None:
        halo, mode = None, 'NCCL all-gather per application (peer mapping failed on another rank)'
    conv_fn = lambda xl, e, a: model.conv1(xl, e, a)          # noqa: E731

    def step_strip(i):
        model.conv1._h_cache.clear()
        with torch.no_grad():
            if halo is not None:
                return partition.partitioned_conv_stack_peer(conv_fn, x_loc, part, ea_loc, T, halo)
            return partition.partitioned_conv_stack(conv_fn, x_loc.clone(), part, ea_loc, T)

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()
    ssteps = max(2, min(args.steps, 5))
    for i in range(3):
        step_strip(i)
    barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(ssteps):
        step_strip(i)
    b.record()
    barrier()
    ms = torch.tensor([a.elapsed_time(b)], device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_strip = float(ms.item())
    got = step_strip(0)
    # parity against the unpartitioned stack on the same sample (every rank computes it: 1 step)
    model.conv1._h_cache.clear()
    torch.cuda.empty_cache()
    with torch.no_grad():
        ea_full = graphs.ball_edge_attr(grid, ei, x6c[:, 2])
        full = model.conv_stack(x0g, ei, ea_full)
    ref = full[part.row_lo * s:part.row_hi * s]
    err = torch.tensor([float((got - ref).abs().max() / ref.abs().max())], device=dev)
    dist.all_reduce(err, op=dist.ReduceOp.MAX)
    halo_bytes = 2 * part.R * s * w * 4 * (T - 1)
    if rank == 0:
        print(json.dumps(dict(
            value=E * T * ssteps / (ms_strip * 1e-3), unit='edge-apps/s', scaling='strong', ms_per_step=ms_strip / ssteps,
            steps=ssteps, n_gpus=world, halo=mode, nvlink_bytes_per_rank_per_step=halo_bytes,
            local_edges=int(part.edge_index.size(1)), parity_vs_unpartitioned=float(err.item()),
            note='one %dx%d mesh (E=%d) cut into %d row strips, edges owned by their destination; a step = edge features '
                 'of the local edges + T applications with a halo push after each; timed with CUDA events, max over '
                 'ranks' % (s, s, E, world))))
    if halo is not None:
        halo.close()
    dist.barrier()
    dist.destroy_process_group()
    return 0


def run_strip_children(args, rank):
    """Every rank of the main bench spawns its own child (same RANK / WORLD_SIZE / LOCAL_RANK, MASTER_PORT + 23);
    rank 0 returns the child's JSON object (or an error record)."""
    # the children rendezvous among themselves: not through the elastic agent's store of the parent job (with
    # TORCHELASTIC_USE_AGENT_STORE every rank is a CLIENT of MASTER_PORT and nobody would serve the new port: run r2h)
    env = {k: v for k, v in os.environ.items() if not k.startswith('TORCHELASTIC_')}
    env['MASTER_PORT'] = str(int(env.get('MASTER_PORT', '29500')) + 23)
    env.setdefault('MASTER_ADDR', '127.0.0.1')
    cmd = [sys.executable, os.path.abspath(__file__), '--strip-only', '--workload', args.workload, '--precision',
           args.precision, '--steps', str(args.steps)]
    try:
        res = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
        if rank != 0:
            return None
        lines = [l for l in res.stdout.splitlines() if l.startswith('{')]
        if res.returncode == 0 and lines:
            return json.loads(lines[-1])
        return dict(error='strip child rc=%d: %s' % (res.returncode, res.stderr.strip().splitlines()[-1][:300] if res.stderr.strip() else ''))
    except subprocess.TimeoutExpired:
        return dict(error='strip child timed out') if rank == 0 else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5,
                    help='timed steps of the metric and e2e lines (secondary lines: fixed counts, see the docstring)')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default=os.environ.get('NNCONV_BENCH_WORKLOAD', 'darcy241'), choices=sorted(WORKLOADS))
    ap.add_argument('--precision', default=os.environ.get('NNCONV_B200_PRECISION', 'f16'))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-parity', action='store_true', help='skip the full-graph parity check and the fp32-grade line')
    ap.add_argument('--no-train', action='store_true', help='skip the training-step measurement')
    ap.add_argument('--no-other-configs', action='store_true', help='skip BASELINE configs 2, 4, 5')
    ap.add_argument('--no-strip', action='store_true', help='skip the single-mesh strip-partition measurement (N > 1)')
    ap.add_argument('--strip-only', action='store_true', help=argparse.SUPPRESS)
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the outputs of the last timed step as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs writes the outputs of the b200 arm')
    if args.strip_only:
        return strip_child_main(args)
    cfg = WORKLOADS[args.workload]
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    T = cfg['depth']
    config = dict(workload='GKN KernelNN conv stack, synthetic Darcy-2D %dx%d r=%g width=%d ker_width=%d T=%d, '
                           '1 graph sample per GPU per step' % (cfg['s'], cfg['s'], cfg['r'], cfg['width'],
                                                                cfg['ker_width'], T),
                  parallelism='batch-sharded dp%d (no data-path collective)' % world,
                  tie_rule='lattice distances == r included (exact integer rule)',
                  l2='inputs larger than L2 (per-edge feature stream >= 3 GB per step)')

    if args.impl == 'reference':
        if rank != 0:
            return 0
        rate, cores, kind, desc, ms = cpu_reference_rate(cfg, steps=args.steps, warmup=min(args.warmup, 1))
        line = dict(metric='NNConv edge-applications/s', value=rate, unit='edge-apps/s', n_gpus=args.gpus,
                    steps=args.steps, warmup=args.warmup, ms_per_step=ms, higher_is_better=True, scaling='weak',
                    vs_baseline=None, dtype='f32', data='synthetic', impl='reference', config=config,
                    cpu_baseline=dict(value=rate, unit='edge-apps/s', cores=cores, kind=kind, sample=desc),
                    e2e=dict(value=rate, unit='edge-apps/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                    gpu_launches=0)
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------------------------ B200 arm
    import torch.distributed as dist
    from graph_pde_b200 import _lib, graphs, nn_conv
    from graph_pde_b200.models import KernelNN
    assert torch.cuda.is_available(), 'bench.py (impl b200) needs a CUDA device; there is no CPU fallback'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    L = _lib.lib()
    _lib.check(L.nnconv_init())

    s, r, w, kw = cfg['s'], cfg['r'], cfg['width'], cfg['ker_width']
    torch.manual_seed(0)
    model = KernelNN(w, kw, T, 6, in_width=6, precision=args.precision).to(dev).eval()
    ei = graphs.ball_connectivity(s, r, dev, True)
    E, N = ei.size(1), s * s
    n_samples = 2
    host_x, host_ea, dev_x, dev_ea = [], [], [], []
    for i in range(n_samples):
        x_i, _, ea_i = graphs.darcy_sample(s, r, dev, seed=1000 * rank + i, edge_index=ei)
        dev_x.append(x_i)
        dev_ea.append(ea_i)
        host_x.append(x_i.cpu().pin_memory())
        host_ea.append(ea_i.cpu().pin_memory())
    # e2e staging: two device buffers, filled from pinned host memory on a copy stream while the previous step
    # computes (what any input pipeline does); every step's copy is inside the timed region.
    stage = [(torch.empty_like(dev_x[0]), torch.empty_like(dev_ea[0])) for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    host_out = torch.empty(N, 1).pin_memory()
    e2e_state = {'prefetched': -1}

    class D(object):
        pass

    def step_resident(i):
        model.conv1._h_cache.clear()                  # every step is a new sample: recompute edge features
        with torch.no_grad():
            x0 = model.fc1(dev_x[i % n_samples])
            return model.conv_stack(x0, ei, dev_ea[i % n_samples])

    def prefetch(i):
        sx, sea = stage[i % 2]
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[i % 2])   # the step that last used this buffer has finished with it
            sx.copy_(host_x[i % n_samples], non_blocking=True)
            sea.copy_(host_ea[i % n_samples], non_blocking=True)   # bumps _version -> edge features recomputed
            ready[i % 2].record(copy_stream)
        e2e_state['prefetched'] = i

    def step_e2e(i):
        if e2e_state['prefetched'] < i:
            prefetch(i)
        torch.cuda.current_stream().wait_event(ready[i % 2])
        prefetch(i + 1)                               # next step's inputs travel while this step computes
        d = D()
        d.x, d.edge_index, d.edge_attr = stage[i % 2][0], ei, stage[i % 2][1]
        with torch.no_grad():
            out = model(d)
        consumed[i % 2].record()
        host_out.copy_(out, non_blocking=False)
        return host_out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last = {}                 # what the last timed step of each path returned (--dump-outputs)

    def timed(fn, steps, warmup, pre=None, keep=False):
        for i in range(warmup):
            fn(i)
        barrier()
        if pre is not None:
            pre()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(steps):
            out = fn(warmup + i)
            if keep:
                last[fn] = out
            del out
        b.record()
        barrier()
        ms = torch.tensor([a.elapsed_time(b)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    sampler = ClockSampler(local_rank)
    launches0 = nn_conv.stats['launches']
    if rank == 0:
        sampler.start()
    ms_total = timed(step_resident, args.steps, max(args.warmup, 3), keep=bool(args.dump_outputs))
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dumped = {'conv_stack': last.pop(step_resident).cpu()}
    launches = nn_conv.stats['launches'] - launches0
    launches_timed = int(round(launches * args.steps / float(args.steps + max(args.warmup, 3))))
    value = world * E * T * args.steps / (ms_total * 1e-3)

    def e2e_reset():          # nothing copied outside the timed region: the first timed step fetches its own inputs
        copy_stream.synchronize()
        e2e_state['prefetched'] = -1

    ms_e2e = timed(step_e2e, args.steps, 1, pre=e2e_reset, keep=bool(args.dump_outputs))
    if args.dump_outputs:
        dumped['model_out'] = last.pop(step_e2e).clone()
        if rank == 0:
            dump_outputs(args.dump_outputs, dumped)
        del dumped
    e2e_value = world * E * T * args.steps / (ms_e2e * 1e-3)
    h2d = host_x[0].numel() * 4 + host_ea[0].numel() * 4
    d2h = host_out.numel() * 4

    # per-kernel-class device time of ONE step (CUDA events on the launch stream, inside the library)
    prof = None
    if rank == 0:
        _lib.check(L.nnconv_profile_begin())
        step_resident(0)
        ms_k = (ctypes.c_double * 8)()
        n_k = (ctypes.c_int64 * 8)()
        _lib.check(L.nnconv_profile_end(ms_k, n_k, 8))
        prof = {KIND_NAMES[k]: dict(ms=ms_k[k], launches=int(n_k[k])) for k in range(6)}
    barrier()

    # ---- training step (forward + tensor-core backward + Adam), one graph sample per rank per step, parameter
    # gradients sum-reduced over the ranks with ONE flat all-reduce (partition.allreduce_gradients; the reference's
    # loss is a sum over the batch, UAI1_full_resolution.py:262-271).  Same timing rules as the main number.
    train = None
    if not args.no_train and args.precision in ('f16', 'bf16'):
        from graph_pde_b200 import partition
        model.conv1._h_cache.clear()
        torch.cuda.empty_cache()
        tmodel = KernelNN(w, kw, T, 6, in_width=6, precision=args.precision).to(dev)
        tmodel.load_state_dict(model.state_dict())
        opt = torch.optim.Adam(tmodel.parameters(), lr=1e-4)
        targets = [torch.randn(N, 1, device=dev, generator=torch.Generator(device=dev).manual_seed(7 + i + 10 * rank))
                   for i in range(n_samples)]
        n_params = sum(p.numel() for p in tmodel.parameters())
        loss_hist = []

        def step_train(i):
            d = D()
            d.x, d.edge_index, d.edge_attr = dev_x[i % n_samples], ei, dev_ea[i % n_samples]
            opt.zero_grad(set_to_none=True)
            out = tmodel(d)
            loss = torch.norm(out.view(-1) - targets[i % n_samples].view(-1), 1)      # UAI1_full_resolution.py:265
            loss.backward()
            partition.allreduce_gradients(tmodel)
            opt.step()
            loss_hist.append(loss.detach())
        tsteps = max(2, min(args.steps, 3))
        ms_train = timed(step_train, tsteps, 2)
        losses = [float(v) for v in loss_hist]
        train = dict(value=world * E * T * tsteps / (ms_train * 1e-3), unit='edge-apps/s (forward + backward + Adam)',
                     ms_per_step=ms_train / tsteps, steps=tsteps, warmup=2, n_gpus=world,
                     allreduce_bytes_per_step=4 * n_params if world > 1 else 0, params=n_params,
                     backward='tensor cores (csrc/backward_tc.cu): per-application k_dy + GEMMs, one deferred pass over the '
                              'hidden layers for all T applications',
                     loss_first=losses[0], loss_last=losses[-1],
                     note='one 241^2-class graph per rank per step, L1 loss, Adam; gradients sum-reduced with one flat '
                          'all-reduce per step' if world > 1 else 'one graph per step, L1 loss, Adam')
        tmodel.conv1.invalidate()                 # the closure above still references the model: drop its 2 KB/edge
        tmodel.conv1._tstate = None               # buffers (edge features + kept activations, ~94 GB at 241^2) explicitly
        del step_train, tmodel, opt
        import gc
        gc.collect()
        torch.cuda.empty_cache()
    barrier()

    # ---- parity at the benchmarked configuration and precision + the fp32-grade (f16x2) line, rank 0 only
    parity, fp32_grade = None, None
    if rank == 0 and not args.no_parity:
        with torch.no_grad():
            x0 = model.fc1(dev_x[0])
            got = model.conv_stack(x0, ei, dev_ea[0])
        model.conv1._h_cache.clear()
        torch.cuda.empty_cache()
        ref = oracle_stack_cuda(cfg, model, x0, ei, dev_ea[0])
        err = rel_err(got, ref)
        parity = dict(max_rel_err=err, tol=TOL.get(args.precision), ok=bool(err < TOL.get(args.precision, 2e-3)),
                      vs='oracle port, fp32 torch ops on CUDA (allow_tf32=False), edge-chunked',
                      config='%s, full graph (E=%d), all T=%d applications, metric max|out-ref|/max|ref| of the final '
                             'node features' % (args.workload, E, T))
        del got
        if args.precision == 'f16':
            m2 = KernelNN(w, kw, T, 6, in_width=6, precision='f16x2').to(dev).eval()
            m2.load_state_dict(model.state_dict())

            def step_x2(i):
                m2.conv1._h_cache.clear()
                with torch.no_grad():
                    return m2.conv_stack(m2.fc1(dev_x[i % n_samples]), ei, dev_ea[i % n_samples])
            st2 = 3
            for i in range(2):
                step_x2(i)
            torch.cuda.synchronize()
            a2, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a2.record()
            for i in range(st2):
                step_x2(i)
            b2.record()
            torch.cuda.synchronize()
            ms2 = a2.elapsed_time(b2) / st2
            with torch.no_grad():
                got2 = m2.conv_stack(x0, ei, dev_ea[0])
            err2 = rel_err(got2, ref)
            fp32_grade = dict(precision='f16x2', value=E * T / (ms2 * 1e-3), unit='edge-apps/s', ms_per_step=ms2, steps=st2,
                              n_gpus=1, parity=dict(max_rel_err=err2, tol=TOL['f16x2'], ok=bool(err2 < TOL['f16x2'])),
                              note='every tensor-core operand as an fp16 (hi, lo) pair, products hi*hi+hi*lo+lo*hi '
                                   'in fp32: the like-for-like line against the reference\'s fp32 arithmetic')
            del got2, m2
        torch.cuda.empty_cache()
    barrier()

    configs = None
    if rank == 0 and not args.no_other_configs and args.precision in ('f16', 'bf16'):
        model.conv1._h_cache.clear()
        torch.cuda.empty_cache()
        try:
            configs = other_configs(dev, args.precision)
        except Exception as exc:           # never lose the headline line to a secondary measurement
            configs = dict(error='%s: %s' % (type(exc).__name__, str(exc)[:300]))
    barrier()

    # ---- ONE mesh cut into N row strips (strong scaling), in child processes: see strip_child_main
    strip = None
    if world > 1 and not args.no_strip:
        model.conv1._h_cache.clear()
        nn_conv.clear_caches()
        torch.cuda.empty_cache()
        strip = run_strip_children(args, rank)
        barrier()

    if rank == 0:
        pk = peaks()
        Kp = ((kw + 63) // 64) * 64
        es = 4 if args.precision in ('fp32', 'f16x2') else 2
        conv_bytes = T * E * (Kp * es + 4)                       # h_e stream + dst index, per step
        gemm_flops = 2.0 * E * Kp * Kp                           # hidden layer 2 (1024 x 1024) per step
        fused = prof['apply_fused']['launches'] > 0
        conv_key = 'apply_fused' if fused else 'conv_scatter'
        conv_ms, gemm_ms = prof[conv_key]['ms'], prof['hidden_gemm']['ms']
        rf_conv = dict(kernel='k_apply_tc (Y GEMM + contraction/scatter, persistent)' if fused else 'k_conv_tc', bound='hbm', achieved=conv_bytes / (conv_ms * 1e-3) / 1e9 if conv_ms else None,
                       peak=pk['hbm_gbs'], unit='GB/s', traffic=None,
                       ms_per_launch=conv_ms / max(1, prof[conv_key]['launches']),
                       alg_bytes_per_edge_app=Kp * es + 4)
        rf_gemm = dict(kernel='k_gemm_tc(hidden)', bound='tensor', achieved=gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms else None,
                       peak=pk['tf_sustained'], unit='TFLOP/s', traffic=None,
                       ms_per_launch=gemm_ms / max(1, prof['hidden_gemm']['launches']))
        for rf in (rf_conv, rf_gemm):
            rf['frac'] = (rf['achieved'] / rf['peak']) if rf['achieved'] else None
            rf['peak_source'] = pk['source']
        if fused and args.workload == 'darcy241' and args.precision == 'f16':
            # dram__bytes_read.sum + dram__bytes_write.sum of ONE k_apply_tc launch, ncu --set full capture of this
            # command (profiles/r2r_k_apply_tc_full.md); algorithmic bytes per launch = E * 2052 B
            rf_conv['traffic'] = 56.86e9
            rf_conv['traffic_source'] = 'profiles/r2r_k_apply_tc_full.md (per launch: 52.50 GB read + 4.36 GB written; algorithmic %.2f GB per launch)' % (E * (Kp * es + 4) / 1e9)
        dominant = rf_conv if conv_ms >= gemm_ms else rf_gemm
        f_alg = 2.0 * (6 * kw + kw * kw + kw * w * w + w * w)    # SURVEY 8(d), reference formulation A
        b_alg = 16 + 24 + 4.0 * 2 * w * N / E
        line = dict(metric='NNConv edge-applications/s', value=value, unit='edge-apps/s', n_gpus=world,
                    steps=args.steps, warmup=max(args.warmup, 3), ms_per_step=ms_total / args.steps,
                    higher_is_better=True, scaling='weak', vs_baseline=None,
                    dtype=args.precision, data='synthetic', config=config, clocks=clocks,
                    e2e=dict(value=e2e_value, unit='edge-apps/s', h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
                             ms_per_step=ms_e2e / args.steps,
                             note='x and edge_attr from pinned host memory every step (double-buffered prefetch on a '
                                  'copy stream overlaps the next step\'s H2D with this step\'s kernels); edge_index '
                                  '(shared mesh) resident; output [N,1] read back'),
                    gpu_launches=launches_timed, roofline=dominant,
                    roofline_kernels=[rf_conv, rf_gemm], kernel_ms_per_step=prof,
                    roofline_survey=dict(formA_tensor_frac=value / world * f_alg / (pk['tf_sustained'] * 1e12),
                                         fused_hbm_frac=value / world * b_alg / (pk['hbm_gbs'] * 1e9),
                                         note='SURVEY 8(d) reconciliation: F_alg=%.4g FLOP, B_alg=%.3g B per '
                                              'edge-app of the reference formulation; the hoisted/reassociated '
                                              'kernels execute ~40x fewer FLOPs, so formA_tensor_frac may exceed 1'
                                              % (f_alg, b_alg)),
                    edges=E, nodes=N, parity=parity, fp32_grade=fp32_grade, train=train, strip=strip, configs=configs)
        if not args.no_cpu_baseline:
            line['gpu_reference_port'] = gpu_reference_rate(cfg, dev)
            rate, cores, kind, desc, _ = cpu_reference_rate(cfg, steps=2)
            line['cpu_baseline'] = dict(value=rate, unit='edge-apps/s', cores=cores, kind=kind, sample=desc)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0 and fp32_grade is not None and not fp32_grade['parity']['ok']:
        sys.stderr.write('bench.py: fp32-grade (f16x2) line outside its tolerance: %s\n' % fp32_grade['parity'])
    if rank == 0 and parity is not None and not parity['ok']:      # the benchmarked precision itself: hard failure
        sys.stderr.write('bench.py: PARITY FAILED: %s\n' % parity)
        return 1
    return 0


if __name__ == '__main__':
    sys.exit(main())
