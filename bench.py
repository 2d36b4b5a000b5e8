"""bench.py — headline benchmark of the B200 hot paths (contract: see the task statement / DESIGN.md §5).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

metric  : sampled edges/s of pyg_lib.sampler.neighbor_sample.
N = 1   : BASELINE.json configs[1] — ogbn-products-shaped CSR (2,449,029 nodes / 123,718,280 edges, int64), fan-out
          [15,10], 1024 seeds per step, no replacement, return_edge_id.  One step = one call on one batch.
          `value` = graph AND seeds resident in HBM (each call still ends with the API's own host sync, because the op
          returns Python lists); `e2e` = the same through the public API with HOST buffers: pinned seeds -> device
          every step, sampled (row, col, node_id, edge_id) -> pinned host memory every step.
          Same JSON line: `parity` (gates run BEFORE timing, against the reference's CPU implementation in a
          subprocess: C2 bit-exact incl. generator state, C3 bf16 <= 1e-3 rel. Frobenius and <= 1 ulp), `roofline`
          (dominant sampler kernel, device-timed, actual edges), `cpu_baseline`, `segment_matmul` (configs[2]: 64
          relations, N = 2^20 ragged rows, 128 -> 128 bf16: TFLOP/s, roofline, its own e2e), `c5_single_gpu`
          (configs[4]'s graph and batch on one GPU: the strong-scaling baseline of the N > 1 lines).
N > 1   : BASELINE.json configs[4] — papers100M-shaped CSR (111,059,956 nodes / 1,615,685,872 edges) replicated on
          every GPU, ONE batch of 65,536 seeds per step, frontier-sharded over the ranks: each rank draws its slice of
          every hop's frontier, the sampled edges are all-gathered over NVLink (peer-memory stores fused into the
          sampling kernel), dedup is partitioned by key; every rank returns the full, reference-exact result.
          `scaling` = "strong" (work per step is fixed as N grows); `c5.single_gpu_edges_per_s` is measured in the
          same run, `replicas` keeps the collective-free weak-scaling number of round 1 as a secondary key.
"""
import argparse
import ctypes as C
import json
import os
import os.path as osp
import queue
import statistics
import subprocess
import sys
import threading
import time

ROOT = osp.dirname(osp.abspath(__file__))
for p in (ROOT, osp.join(ROOT, 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)

N_NODES, N_EDGES = 2_449_029, 123_718_280            # C2
BATCH, FANOUT = 1024, [15, 10]
C5_NODES, C5_EDGES, C5_BATCH = 111_059_956, 1_615_685_872, 65_536
BYTES_PER_EDGE = 41.0  # SURVEY.md 8(d): algorithmic bytes per sampled edge at fan-out [15,10], int64


class ClockMonitor:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index: int):
        self.index, self.proc, self.lines, self.lo, self.hi = index, None, [], 0, None

    def start(self):
        """Launch nvidia-smi and wait for its first sample: NVML start-up takes ~100 ms and holds driver locks,
        so it must not overlap the timed region."""
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '50'], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)

            def pump():
                for ln in self.proc.stdout:
                    self.lines.append(ln)
            self.t = threading.Thread(target=pump, daemon=True)
            self.t.start()
            t0 = time.time()
            while not self.lines and time.time() - t0 < 3.0:
                time.sleep(0.01)
        except Exception:  # noqa
            self.proc = None
        return self

    def __enter__(self):   # marks the start of the timed region
        self.lo = len(self.lines)
        return self

    def __exit__(self, *a):  # marks its end
        time.sleep(0.06)       # one more sample so that short regions are covered
        self.hi = len(self.lines)

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.lines[max(self.lo - 1, 0):self.hi]:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': mx or None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def run_ref_bench(args, timeout=3000):
    out = subprocess.run([sys.executable, osp.join(ROOT, 'oracle', 'ref_bench.py')] + args, stdout=subprocess.PIPE,
                         stderr=subprocess.PIPE, text=True, timeout=timeout)
    for ln in out.stdout.splitlines():
        if ln.startswith('REFBENCH '):
            return json.loads(ln[len('REFBENCH '):])
    raise RuntimeError('ref_bench failed: ' + out.stderr[-2000:])


def host_cores():
    """Cores this process may run on (the cgroup's share of the box), not os.cpu_count()."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:  # noqa
        return os.cpu_count() or 1


def config_dict(n_gpus):
    if n_gpus == 1:
        return {'workload': 'neighbor_sample ogbn-products-shaped CSR (2,449,029 nodes / 123,718,280 edges, int64, '
                            'log-normal degrees), fanout [15,10], 1024 seeds/step, replace=False, return_edge_id=True',
                'batch_seeds': BATCH, 'fanout': FANOUT, 'index_dtype': 'int64', 'parallelism': 'single GPU',
                'l2': 'inputs_larger_than_L2 (col = 990 MB, new random seeds every step)'}
    return {'workload': 'neighbor_sample papers100M-shaped CSR (111,059,956 nodes / 1,615,685,872 edges, int64, log-normal '
                        'degrees), fanout [15,10], ONE batch of 65,536 seeds per step, replace=False, return_edge_id=True',
            'batch_seeds': C5_BATCH, 'fanout': FANOUT, 'index_dtype': 'int64',
            'parallelism': 'frontier-sharded x%d: CSR replicated, each rank draws 1/%d of every frontier, sampled edges '
                           'all-gathered by peer-memory stores over NVLink, dedup partitioned by key hash, identical full '
                           'result on every rank' % (n_gpus, n_gpus),
            'l2': 'inputs_larger_than_L2 (col = 12.9 GB, new random seeds every step)'}


def reference_arm(a):
    """--impl reference: the reference's CPU implementation on the host cores, same metric/config as our arm at this N:
    one single-threaded worker process per core of the cgroup (how PyG deploys CPU sampling), each step a bounded
    sample; median over three repeats."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    workers = host_cores()
    if a.gpus == 1:
        calls = max(2, min(2 * (a.steps + a.warmup), 40))
        reps = [run_ref_bench(['sampler', '--workers', str(workers), '--calls', str(calls)]) for _ in range(3)]
    else:   # configs[4]: papers100M-shaped graph, 65,536-seed batches (a call is ~1 s of one core)
        reps = [run_ref_bench(['sampler', '--workers', str(workers), '--calls', '2', '--graph', 'papers', '--batch', str(C5_BATCH)])]
    reps.sort(key=lambda r: r['edges_per_s'])
    r = reps[len(reps) // 2]
    line = {'impl': 'reference', 'metric': 'sampled_edges_per_s', 'value': r['edges_per_s'], 'unit': 'edges/s',
            'n_gpus': a.gpus, 'steps': a.steps, 'warmup': a.warmup,
            'ms_per_step': 1e3 * r['seconds'] / max(r['calls'] / workers, 1), 'higher_is_better': True,
            'scaling': 'weak' if a.gpus == 1 else 'strong', 'vs_baseline': None, 'dtype': 'int64', 'data': 'synthetic',
            'config': config_dict(a.gpus),
            'cpu_baseline': {'value': r['edges_per_s'], 'unit': 'edges/s', 'cores': r['cores'], 'kind': r['kind'],
                             'sample': r['sample'], 'repeats': [x['edges_per_s'] for x in reps]},
            'e2e': {'value': r['edges_per_s'], 'unit': 'edges/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ parity gates
def parity_gates(P, dev, rowptr_c, col_c, rowptr, col, perm, with_matmul=True):
    """BASELINE.md 4.4: parity before timing, at config size, against the reference in a subprocess."""
    import torch
    from graphs import ragged_ptr
    from refproc import RefSession, accumulation_bound, compare_homo, lowp_ulp_excess, rng_prefix
    res = {}
    seeds = [perm[b * BATCH:(b + 1) * BATCH].clone() for b in (0, 1)]
    with RefSession() as rs:
        ref = rs.run(dict(kind='homo', rowptr=rs.share(rowptr_c), col=rs.share(col_c), seeds=seeds, num_neighbors=FANOUT, rng_seed=777))
        saved = torch.get_rng_state()
        torch.manual_seed(777)
        cmp = [compare_homo(P.sampler.neighbor_sample(rowptr, col, s.to(dev), FANOUT), c) for s, c in zip(seeds, ref['calls'])]
        rng_ok = bool(torch.equal(rng_prefix(), ref['rng_after']))
        torch.set_rng_state(saved)
        res['c2_neighbor_sample'] = {'against': ref['kind'], 'calls': len(cmp), 'edges': sum(c['edges'] for c in cmp),
                                     'bit_exact': all(c['bit_exact'] for c in cmp), 'generator_state_equal': rng_ok,
                                     'mismatch': sum((c['mismatch'] for c in cmp), [])}
        ok = res['c2_neighbor_sample']['bit_exact'] and rng_ok
        if with_matmul:
            Nn, K, M, B = 1 << 20, 128, 128, 64
            g = torch.Generator().manual_seed(0)
            x = torch.randn(Nn, K, generator=g).to(torch.bfloat16)
            w = (torch.randn(B, K, M, generator=g) / K ** 0.5).to(torch.bfloat16)
            ptr = ragged_ptr(Nn, B, 100)
            y_path = rs.out_file(Nn * M, torch.bfloat16)
            refm = rs.run(dict(kind='matmul', x=rs.share(x), w=rs.share(w), ptr=ptr, y_path=y_path))
            y_ref = torch.from_file(y_path, shared=False, size=Nn * M, dtype=torch.bfloat16).view(Nn, M)
            y = P.ops.segment_matmul(x.to(dev), ptr.to(dev), w.to(dev)).cpu()
            rel = float((y.float() - y_ref.float()).norm() / y_ref.float().norm())
            ulp = lowp_ulp_excess(y, y_ref, accumulation_bound(x.to(dev), ptr, w.to(dev)).cpu())
            res['c3_segment_matmul'] = {'against': refm['kind'], 'rel_frobenius': rel, 'max_ulp': ulp,
                                        'tolerance': '<= 1e-3 and <= 1 bf16 ulp (+ the fp32 summation-order bound 2K 2^-24 |x||w| for cancelling results)',
                                        'pass': rel <= 1e-3 and ulp <= 1.0}
            ok = ok and res['c3_segment_matmul']['pass']
            del y_ref
    res['pass'] = bool(ok)
    return res


# ------------------------------------------------------------------------------------------------ helpers
class Timer:
    def __init__(self, torch, dist, dev, world, mon, P):
        self.torch, self.dist, self.dev, self.world, self.mon, self.P = torch, dist, dev, world, mon, P

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def run(self, step_fn, steps, warmup, finish=None, first=0):
        """`warmup` untimed calls, then exactly `steps` timed ones between barrier + synchronize; CUDA events on the
        current stream; max over ranks; edges summed over ranks unless the step is collective (same result everywhere)."""
        torch = self.torch
        for i in range(warmup):
            step_fn(first + i)
        if finish is not None:
            finish()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = self.P.kernel_launches()
        edges = 0
        with self.mon:
            e0.record()
            for i in range(warmup, warmup + steps):
                edges += step_fn(first + i)
            if finish is not None:
                finish()   # e.g. make the timed stream wait for outstanding result copies
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        launches = self.P.kernel_launches() - l0
        t = torch.tensor([ms, float(edges), float(launches)], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            tmax = t.clone(); self.dist.all_reduce(tmax, op=self.dist.ReduceOp.MAX)
            tsum = t.clone(); self.dist.all_reduce(tsum, op=self.dist.ReduceOp.SUM)
            ms, edges_sum, launches = float(tmax[0]), float(tsum[1]), float(tsum[2])
        else:
            edges_sum = float(edges)
        self.barrier()
        return ms, float(edges), edges_sum, int(launches), self.mon.summary()


class HostCopier:
    """The loader side of the e2e leg: a second host thread queues the device -> pinned-host copies of step i on a copy
    stream while the main thread is already inside the next sampling call (the op releases the GIL while it waits
    for the GPU).  Four rotating sets of pinned buffers."""
    def __init__(self, torch, dev, caps, n_slots=4):
        self.torch, self.dev = torch, dev
        self.bufs = [[torch.empty(c, dtype=torch.int64).pin_memory() for c in caps] for _ in range(n_slots)]
        self.done = [torch.cuda.Event() for _ in range(n_slots)]
        self.stream = torch.cuda.Stream(device=dev)
        self.q = queue.Queue()
        self.bytes = 0
        self.n = 0
        self.t = threading.Thread(target=self._loop, daemon=True)
        self.t.start()

    def _loop(self):
        torch = self.torch
        torch.cuda.set_device(self.dev)
        while True:
            item = self.q.get()
            if item is None:
                self.q.task_done()
                return
            outs, ready = item
            slot = self.n % len(self.bufs)
            self.n += 1
            self.done[slot].synchronize()           # the buffers of step i - n_slots are free again
            with torch.cuda.stream(self.stream):
                self.stream.wait_event(ready)
                for h, t in zip(self.bufs[slot], outs):
                    t.record_stream(self.stream)
                    h[:t.numel()].copy_(t.reshape(-1), non_blocking=True)
                self.done[slot].record()
            self.bytes += 8 * sum(t.numel() for t in outs)
            self.q.task_done()

    def submit(self, outs):
        ready = self.torch.cuda.Event()
        ready.record()
        self.q.put((outs, ready))

    def drain(self):
        self.q.join()
        self.torch.cuda.current_stream().wait_stream(self.stream)

    def close(self):
        self.q.put(None)
        self.t.join(timeout=5)


def sampler_roofline(abi, step_dev, first, n_prof, torch, peaks, hbm_peak, peak_src, traffic):
    """CUDA events on the launching stream around every launch of the sampler's kernels (pygb200_profile_*);
    `work` = edges the timed calls actually emitted (not the static bound)."""
    abi.pygb200_profile_enable(1)
    edges = 0
    for i in range(first, first + n_prof):
        edges += step_dev(i)
    torch.cuda.synchronize()
    abi.pygb200_profile_enable(0)
    prof = {}
    for name in ('count', 'sample', 'mark', 'assign', 'lookup', 'seed', 'insert', 'rows', 'push', 'pref', 'reduce', 'xbarrier', 'final', 'cleanup', 'export'):
        msv, ln, wk = C.c_double(), C.c_int64(), C.c_int64()
        abi.pygb200_profile_read(name.encode(), C.byref(msv), C.byref(ln), C.byref(wk))
        prof[name] = (msv.value, ln.value, wk.value)
    dom = max(prof, key=lambda k: prof[k][0])
    d_ms, d_launches, _ = prof[dom]
    launches_per_call = max(d_launches, 1) / max(n_prof, 1)
    # every edge of a call passes through exactly one launch of the kernel: bytes per launch = 41 B x edges per launch
    bytes_per_launch = BYTES_PER_EDGE * edges / max(d_launches, 1)
    avg_s = d_ms / max(d_launches, 1) * 1e-3
    achieved = bytes_per_launch / avg_s / 1e9 if d_ms > 0 else 0.0
    return {'bound': 'hbm', 'kernel': 'k_' + dom, 'achieved': achieved, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': achieved / hbm_peak,
            'traffic': traffic, 'peak_source': peak_src, 'avg_launch_us': 1e6 * avg_s, 'bytes_per_launch': bytes_per_launch,
            'launches_per_call': launches_per_call, 'edges_per_call': edges / max(n_prof, 1),
            'kernel_ms_per_call': {k: v[0] / max(n_prof, 1) for k, v in prof.items() if v[1]}}


def load_traffic():
    """DRAM bytes per launch of the dominant kernels from the committed `ncu --set full` captures (profiles/)."""
    out = {}
    for fn in ('ncu_summary_r2.json', 'ncu_summary_r1.json'):
        try:
            summ = json.load(open(osp.join(ROOT, 'profiles', fn)))
        except Exception:  # noqa
            continue
        for grp in summ.values():
            for d in grp:
                for nm in ('k_v2_sample', 'k_sample_s', 'k_sample', 'k_segment_matmul_tc'):
                    if nm in d['Kernel Name']:
                        out.setdefault(nm, []).append(1e6 * (float(d['dram__bytes_read.sum']) + float(d['dram__bytes_write.sum'])))
                        break
        if out:
            break
    return {k: sum(v) / len(v) for k, v in out.items()}


DUMP_BYTES = 60 << 20   # stays under 64 MB (decimal) in all, .npy headers included


def dump_outputs(out_dir, out):
    """What a caller of (dist_)neighbor_sample receives, as float64 arrays (node and edge ids < 2^53 are exact).  A
    result larger than DUMP_BYTES in all (a 65,536-seed batch) is written as a fixed sample: the same seeded, sorted
    positions of row, col and edge_id (edge_positions.npy) and of node (node_positions.npy); the counts stay whole."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    row, col, node, eid, nph, eph = out
    arrays = {'row': row, 'col': col, 'node': node, 'edge_id': eid}
    n_e, n_n = row.size(0), node.size(0)
    if 8 * (3 * n_e + n_n) > DUMP_BYTES:
        keep = DUMP_BYTES / (8 * (4 * n_e + 2 * n_n))   # the position files count too

        def positions(n):
            g = torch.Generator().manual_seed(0)
            return torch.randperm(n, generator=g)[:int(n * keep)].sort().values
        pe, pn = positions(n_e), positions(n_n)
        arrays = {'row': row.cpu()[pe], 'col': col.cpu()[pe], 'node': node.cpu()[pn], 'edge_id': eid.cpu()[pe],
                  'edge_positions': pe, 'node_positions': pn}
    arrays.update(num_sampled_nodes_per_hop=torch.tensor(nph), num_sampled_edges_per_hop=torch.tensor(eph))
    for name, v in arrays.items():
        np.save(osp.join(out_dir, name + '.npy'), v.cpu().numpy().astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=1000,
                    help='timed steps of the headline path (N = 1: configs[1]; N > 1: configs[4] sharded), also of the N = 1 '
                         'e2e and configs[4] legs; the other legs time at most 20-200 steps and report their own count')
    ap.add_argument('--warmup', type=int, default=20)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-matmul', action='store_true')
    ap.add_argument('--no-parity', action='store_true')
    ap.add_argument('--no-c5', action='store_true', help='N=1: skip the papers100M-shaped single-GPU leg')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the results of the headline path\'s last timed call to DIR/<name>.npy (float64; rank 0)')
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    a.warmup = max(a.warmup, 3)
    if a.dump_outputs and a.impl != 'b200':
        ap.error('--dump-outputs: only for this implementation')
    if a.impl == 'reference':
        return reference_arm(a)

    import torch
    import torch.distributed as dist
    from graphs import lognormal_csr, ragged_ptr
    rank, world = int(os.environ.get('RANK', '0')), int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    import pyg_lib_b200 as P
    abi = C.CDLL(osp.join(osp.dirname(P.__file__), 'libpyg_b200.so'))
    peaks = {}
    try:
        peaks = json.load(open(osp.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:  # noqa
        pass
    hbm_peak = float(peaks.get('hbm_gbs', 6650.0))
    peak_src = 'measured (MEASURED_PEAKS.json)' if 'hbm_gbs' in peaks else 'fallback 6.65 TB/s (B200_PROFILING.md)'
    traffic = load_traffic()
    mon = ClockMonitor(local).start()
    T = Timer(torch, dist, dev, world, mon, P)

    # ---- C2 inputs (deterministic; CPU-generated so that the reference process sees the same graph)
    rowptr_c, col_c = lognormal_csr(N_NODES, N_EDGES, seed=1)
    rowptr, col = rowptr_c.to(dev), col_c.to(dev)
    perm = torch.randperm(N_NODES, generator=torch.Generator().manual_seed(2))
    n_batches = N_NODES // BATCH

    line = {}
    if world == 1:
        # ================================================================ N = 1: configs[1] (+ configs[2], configs[4] on one GPU)
        parity = None
        if not a.no_parity:
            parity = parity_gates(P, dev, rowptr_c, col_c, rowptr, col, perm, with_matmul=not a.no_matmul)
            if not parity['pass']:
                print(json.dumps({'metric': 'sampled_edges_per_s', 'value': None, 'parity': parity,
                                  'error': 'parity gate failed: nothing was timed'}), flush=True)
                mon.stop()
                sys.exit(1)
        del col_c
        my_batches = [i % n_batches for i in range(a.steps + a.warmup + 64)]
        seeds_host = [perm[b * BATCH:(b + 1) * BATCH].clone().pin_memory() for b in my_batches]
        seeds_dev = [s.to(dev) for s in seeds_host]
        torch.manual_seed(12345)
        last = [None]

        def step_dev(i):
            o = P.sampler.neighbor_sample(rowptr, col, seeds_dev[i], FANOUT)
            if a.dump_outputs:
                last[0] = o
            return o[0].numel()
        ms, edges, _, launches, clocks = T.run(step_dev, a.steps, a.warmup)
        value = edges / (ms * 1e-3)
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, last[0])
        last[0] = None

        # e2e: pinned seeds -> device and (row, col, edge_id, node_id) -> pinned host EVERY step, through the public API.  The
        # calls themselves cannot overlap (each consumes the CPU generator where the previous one left it, and returns its
        # counts as host integers); the result copies run on a copy stream beside the next call.  The consumer is what a C++
        # loader would be: cudaMemcpyAsync of exactly the four results (the op hands them out as views of one allocation, so
        # holding the views keeps the storage alive until the copy is done) — 3.9 MB per step instead of the 5.4 MB of the
        # bound-sized buffer, which at this link's ~55 GB/s is the difference between a copy-bound and a call-bound step.
        import ctypes
        rt = ctypes.CDLL('libcudart.so.12')
        rt.cudaMemcpyAsync.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p]
        rt.cudaMemcpyAsync.restype = ctypes.c_int
        cap = BATCH * (FANOUT[0] + FANOUT[0] * FANOUT[1])
        n_slots = 4
        host_bufs = [torch.empty(4 * cap + BATCH, dtype=torch.int64).pin_memory() for _ in range(n_slots)]
        host_ptr = [b.data_ptr() for b in host_bufs]
        seed_bufs = [torch.empty(BATCH, dtype=torch.int64, device=dev) for _ in range(n_slots)]
        copy_stream = torch.cuda.Stream(device=dev)
        cs, ms_ = ctypes.c_void_p(copy_stream.cuda_stream), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        rt.cudaMemcpy2DAsync.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_size_t,
                                         ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p]
        rt.cudaMemcpy2DAsync.restype = ctypes.c_int
        done = [torch.cuda.Event() for _ in range(n_slots)]
        ready = [torch.cuda.Event() for _ in range(n_slots)]
        held = [None] * n_slots
        d2h = [0]
        use_2d = os.environ.get('PYGB200_BENCH_E2E_2D', '1') != '0'

        def step_e2e(i):
            slot = i % n_slots
            done[slot].synchronize()          # step i - 4's copies are done: its host buffer, seed buffer and results are free
            rc = rt.cudaMemcpyAsync(seed_bufs[slot].data_ptr(), seeds_host[i].data_ptr(), BATCH * 8, 1, ms_)
            row, colv, node, eid = outs = P.sampler.neighbor_sample(rowptr, col, seed_bufs[slot], FANOUT)[:4]
            ready[slot].record()
            copy_stream.wait_event(ready[slot])
            E, nb_node = row.numel(), node.numel() * 8
            pitch = colv.data_ptr() - row.data_ptr()
            if use_2d and E and eid.data_ptr() - colv.data_ptr() == pitch:   # views of one allocation: row | col | edge_id at one pitch
                rc |= rt.cudaMemcpy2DAsync(host_ptr[slot], E * 8, row.data_ptr(), pitch, E * 8, 3, 2, cs)
            else:
                for j, t in enumerate((row, colv, eid)):
                    rc |= rt.cudaMemcpyAsync(host_ptr[slot] + j * E * 8, t.data_ptr(), E * 8, 2, cs)
            rc |= rt.cudaMemcpyAsync(host_ptr[slot] + 3 * E * 8, node.data_ptr(), nb_node, 2, cs)
            done[slot].record(copy_stream)
            held[slot] = outs                  # the views keep the storage alive until the slot comes round again
            if rc:
                raise RuntimeError('cudaMemcpyAsync failed')
            d2h[0] += 3 * E * 8 + nb_node
            return E

        def finish_e2e():
            torch.cuda.current_stream().wait_stream(copy_stream)
        ms_e, edges_e, _, _, _ = T.run(step_e2e, a.steps, a.warmup, finish=finish_e2e)
        # what the link gives a copy of that size (same pinned buffers, device-timed): the floor of a copy-bound step
        nb_step = int(d2h[0] / max(a.steps + a.warmup, 1))
        src_probe = torch.empty(nb_step // 8, dtype=torch.int64, device=dev)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for rep in range(3):
            if rep == 1:
                ev0.record()
            rt.cudaMemcpyAsync(host_ptr[0], src_probe.data_ptr(), nb_step, 2, ms_)
        ev1.record(); torch.cuda.synchronize()
        d2h_us = ev0.elapsed_time(ev1) / 2 * 1e3
        e2e = {'value': edges_e / (ms_e * 1e-3), 'unit': 'edges/s', 'h2d_bytes_per_step': BATCH * 8,
               'd2h_bytes_per_step': nb_step, 'ms_per_step': ms_e / a.steps,
               'd2h_alone_us': d2h_us, 'd2h_link_gbs': nb_step / d2h_us / 1e3,
               'how': 'every step: pinned seeds H2D (cudaMemcpyAsync), neighbor_sample through the public API, its four results (row, col, '
                      'edge_id, node_id; exact sizes) D2H to pinned memory on a copy stream beside the next call '
                      '(cudaMemcpy2DAsync for row | col | edge_id, one copy for node_id)' if use_2d else 'every step: pinned seeds H2D, '
                      'neighbor_sample through the public API, four exact-size cudaMemcpyAsync D2H on a copy stream beside the next call'}

        line = {'metric': 'sampled_edges_per_s', 'value': value, 'unit': 'edges/s', 'n_gpus': 1, 'steps': a.steps,
                'warmup': a.warmup, 'ms_per_step': ms / a.steps, 'higher_is_better': True, 'scaling': 'weak',
                'vs_baseline': None, 'dtype': 'int64', 'data': 'synthetic', 'config': config_dict(1), 'clocks': clocks,
                'e2e': e2e, 'gpu_launches': launches, 'edges_per_step': edges / a.steps}
        if parity is not None:
            line['parity'] = parity
        rf = sampler_roofline(abi, step_dev, a.warmup, min(50, a.steps), torch, peaks, hbm_peak, peak_src, None)
        rf['traffic'] = traffic.get(rf['kernel'] + '_s') or traffic.get(rf['kernel'])
        rf['kernel'] += '_s'   # C2 runs the latency-path kernels (k_sample_s, ...)
        rf['note'] = 'C2 is latency-bound (~5 MB per call): the HBM fraction is reported, the binding limit is the ' \
                     'per-call chain of dependent launches + one host round trip'
        line['roofline'] = rf

        # ---- segment_matmul (BASELINE configs[2])
        if not a.no_matmul:
            Nn, K, M, B = 1 << 20, 128, 128, 64
            g = torch.Generator().manual_seed(0)
            xh = torch.randn(Nn, K, generator=g).to(torch.bfloat16).pin_memory()
            x = xh.to(dev)
            w = (torch.randn(B, K, M, generator=g) / K ** 0.5).to(torch.bfloat16).to(dev)
            ptr = ragged_ptr(Nn, B, 100).to(dev)
            for _ in range(5):
                y = P.ops.segment_matmul(x, ptr, w)
            torch.cuda.synchronize()
            iters = 50
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                y = P.ops.segment_matmul(x, ptr, w)
            e1.record(); torch.cuda.synchronize()
            mm_ms = e0.elapsed_time(e1) / iters
            # e2e: features from pinned host memory in, result back to pinned host memory, every call
            yh = torch.empty(Nn, M, dtype=torch.bfloat16).pin_memory()
            for _ in range(2):
                yh.copy_(P.ops.segment_matmul(xh.to(dev, non_blocking=True), ptr, w), non_blocking=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(10):
                yh.copy_(P.ops.segment_matmul(xh.to(dev, non_blocking=True), ptr, w), non_blocking=True)
            e1.record(); torch.cuda.synchronize()
            mm_e2e_ms = e0.elapsed_time(e1) / 10
            flops, byts = 2.0 * Nn * K * M, Nn * K * 2 + Nn * M * 2 + B * K * M * 2 + (B + 1) * 8
            tf_peak = float(peaks.get('bf16_tflops', 1590.0))
            line['segment_matmul'] = {
                'config': '64 relations, N=2^20 ragged rows (log-normal lengths, one empty), 128->128 bf16, ptr on device',
                'ms': mm_ms, 'tflops': flops / (mm_ms * 1e-3) / 1e12, 'algorithmic_bytes': byts,
                'roofline': {'bound': 'hbm', 'achieved': byts / (mm_ms * 1e-3) / 1e9, 'peak': hbm_peak, 'unit': 'GB/s',
                             'frac': byts / (mm_ms * 1e-3) / 1e9 / hbm_peak, 'traffic': traffic.get('k_segment_matmul_tc'),
                             'tensor_frac_of_bf16_peak': flops / (mm_ms * 1e-3) / 1e12 / tf_peak},
                'e2e': {'value': flops / (mm_e2e_ms * 1e-3) / 1e12, 'unit': 'TFLOP/s', 'ms': mm_e2e_ms,
                        'h2d_bytes_per_step': Nn * K * 2, 'd2h_bytes_per_step': Nn * M * 2,
                        'note': '512 MiB over PCIe per call: the link, not the kernel, is the bound'},
                'note': 'x (256 MiB) + out (256 MiB) > L2; arithmetic intensity 63.75 FLOP/B => HBM-bound'}
            del x, w, y, xh, yh

        # ---- configs[4] on one GPU: the strong-scaling baseline of the N > 1 lines, and the throughput schedule's roofline
        if not a.no_c5:
            del rowptr, col
            torch.cuda.empty_cache()
            line['c5_single_gpu'] = c5_leg(a, P, abi, T, torch, dev, 1, 0, peaks, hbm_peak, peak_src, traffic, None)
            torch.cuda.empty_cache()
            # ---- configs[3]: hetero_neighbor_sample on the MAG240M-shaped graph at FULL size (3 node types / 6 edge types,
            # 3.46 G edges = 27.7 GB of col), fan-out [25,15] for every relation, 1024 paper seeds per call.  Parity at 0.1
            # scale against the 1-thread reference: tests/test_config_parity.py.
            try:
                from graphs import mag240m_shaped
                t0 = time.time()
                sizes, rp_d, col_d = mag240m_shaped(1.0, device=dev)
                torch.cuda.synchronize()
                gen_s = time.time() - t0
                nn_d = {k: [25, 15] for k in rp_d}
                permp = torch.randperm(sizes['paper'], device=dev)
                torch.manual_seed(12345)
                h_steps = min(a.steps, 100)
                ms_h, edges_h, _, launches_h, _ = T.run(
                    lambda i: sum(v.numel() for v in P.sampler.hetero_neighbor_sample(rp_d, col_d, {'paper': permp[i * 1024:(i + 1) * 1024]}, nn_d)[0].values()),
                    h_steps, a.warmup)
                line['c4_hetero'] = {'workload': 'hetero_neighbor_sample, MAG240M-shaped (121.7 M papers / 122.4 M authors / 25.7 k institutions, 6 relations, '
                                                 '3.46 G edges), fanout [25,15] per relation, 1024 paper seeds per call',
                                     'value': edges_h / (ms_h * 1e-3), 'unit': 'edges/s', 'ms_per_step': ms_h / h_steps, 'steps': h_steps,
                                     'edges_per_step': edges_h / h_steps, 'gpu_launches_per_step': launches_h / h_steps, 'graph_gen_s': gen_s,
                                     'graph_bytes': int(sum(v.numel() for v in col_d.values()) * 8)}
                del rp_d, col_d, permp
                torch.cuda.empty_cache()
            except Exception as ex:  # noqa  (e.g. a smaller GPU: the leg is informative, not the headline)
                line['c4_hetero'] = {'error': str(ex)[:300]}

        # ---- CPU baseline: the reference's own CPU path on this box's host cores (bounded sample)
        if not a.no_cpu_baseline:
            try:
                r = run_ref_bench(['sampler', '--workers', '1', '--calls', '200'])
                line['cpu_baseline'] = {'value': r['edges_per_s'], 'unit': 'edges/s', 'cores': r['cores'], 'kind': r['kind'],
                                        'sample': r['sample'], 'host_cores_available': host_cores()}
                if not a.no_matmul:
                    best = None
                    for th in (8, 16, 32, 64):   # an oversubscribed thread pool is not a baseline: keep the best
                        if th > host_cores():
                            break
                        rm = run_ref_bench(['matmul', '--calls', '3', '--workers', str(th)])
                        if best is None or rm['tflops'] > best['tflops']:
                            best = rm
                    if best is not None:
                        line['segment_matmul']['cpu_baseline'] = {'value': best['tflops'], 'unit': 'TFLOP/s', 'cores': best['cores'],
                                                                  'kind': best['kind'], 'sample': best['sample']}
            except Exception as ex:  # noqa
                line['cpu_baseline'] = {'value': None, 'unit': 'edges/s', 'cores': 0, 'kind': 'failed', 'sample': str(ex)[:300]}
        print(json.dumps(line), flush=True)
    else:
        # ================================================================ N > 1: configs[4], frontier-sharded
        del col_c
        # secondary: round 1's replicas (every rank its own 1024-seed batches on its own CSR replica, no collective)
        rep_steps = min(a.steps, 200)
        my_batches = [(rank + i * world) % n_batches for i in range(rep_steps + a.warmup)]
        seeds_dev = [perm[b * BATCH:(b + 1) * BATCH].to(dev) for b in my_batches]
        torch.manual_seed(12345 + rank)

        def step_rep(i):
            return P.sampler.neighbor_sample(rowptr, col, seeds_dev[i], FANOUT)[0].numel()
        ms_r, _, edges_r, _, _ = T.run(step_rep, rep_steps, a.warmup)
        replicas = {'value': edges_r / (ms_r * 1e-3), 'unit': 'edges/s', 'ms_per_step': ms_r / rep_steps, 'steps': rep_steps,
                    'workload': 'configs[1] on every rank (CSR replicated, disjoint 1024-seed batches, no data-path collective)'}
        del rowptr, col, seeds_dev
        torch.cuda.empty_cache()
        c5 = c5_leg(a, P, abi, T, torch, dev, world, rank, peaks, hbm_peak, peak_src, traffic, dist)
        if rank == 0:
            line = {'metric': 'sampled_edges_per_s', 'value': c5['value'], 'unit': 'edges/s', 'n_gpus': world, 'steps': a.steps,
                    'warmup': a.warmup, 'ms_per_step': c5['ms_per_step'], 'higher_is_better': True, 'scaling': 'strong',
                    'vs_baseline': None, 'dtype': 'int64', 'data': 'synthetic', 'config': config_dict(world),
                    'clocks': c5.pop('clocks'), 'e2e': c5.pop('e2e'), 'gpu_launches': c5.pop('gpu_launches'),
                    'edges_per_step': c5['edges_per_step'], 'parity': c5.pop('parity'), 'roofline': c5.pop('roofline'),
                    'c5': c5, 'replicas': replicas}
            print(json.dumps(line), flush=True)
    mon.stop()
    if world > 1:
        dist.destroy_process_group()


def c5_leg(a, P, abi, T, torch, dev, world, rank, peaks, hbm_peak, peak_src, traffic, dist):
    """configs[4]: papers100M-shaped CSR generated on the device (same CUDA generator seed on every rank -> identical
    replicas), one 65,536-seed batch per step.  world == 1: the single-GPU op.  world > 1: the frontier-sharded op, gated
    on being bit-identical to the single-GPU op on every rank, with the single-GPU time measured beside it."""
    from graphs import lognormal_csr
    t0 = time.time()
    rowptr, col = lognormal_csr(C5_NODES, C5_EDGES, seed=1, device=dev)
    torch.cuda.synchronize()
    gen_s = time.time() - t0
    steps = a.steps
    perm = torch.randperm(C5_NODES, generator=torch.Generator().manual_seed(2))
    n_seeds = min(steps + a.warmup + 8, C5_NODES // C5_BATCH)   # step i takes batch i % n_seeds: a batch is 512 KB here and on the device
    seeds_host = [perm[i * C5_BATCH:(i + 1) * C5_BATCH].clone().pin_memory() for i in range(n_seeds)]
    seeds_dev = [s.to(dev) for s in seeds_host]
    del perm

    def single(i):
        return P.sampler.neighbor_sample(rowptr, col, seeds_dev[i % n_seeds], FANOUT)

    def sharded(i):
        return P.sampler.dist_neighbor_sample(rowptr, col, seeds_dev[i % n_seeds], FANOUT)
    op = single if world == 1 else sharded
    out = {'graph_gen_s': gen_s, 'steps': steps}
    if world > 1:
        # gate: the sharded result equals the single-GPU result (which tests/test_config_parity.py pins to the reference at
        # this size) — same generator state, every tensor and count, on every rank
        torch.manual_seed(4321)
        o1 = [single(i) for i in (0, 1)]
        s1 = torch.get_rng_state()
        torch.manual_seed(4321)
        oN = [sharded(i) for i in (0, 1)]
        same = all(torch.equal(x, y) for p, q in zip(o1, oN) for x, y in zip(p[:4], q[:4])) and \
            all(p[4] == q[4] and p[5] == q[5] for p, q in zip(o1, oN)) and bool(torch.equal(s1, torch.get_rng_state()))
        flag = torch.tensor([1 if same else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        out['parity'] = {'c5_sharded_equals_single_gpu_on_every_rank': bool(int(flag[0])), 'calls': 2, 'edges': int(sum(o[0].numel() for o in oN)),
                         'pass': bool(int(flag[0])), 'note': 'the single-GPU op is pinned to the reference at this size by tests/test_config_parity.py'}
        del o1, oN
        if not out['parity']['pass']:
            if rank == 0:
                print(json.dumps({'metric': 'sampled_edges_per_s', 'value': None, 'parity': out['parity'],
                                  'error': 'parity gate failed: nothing was timed'}), flush=True)
            sys.exit(1)
    torch.manual_seed(999)
    last = [None]
    keep = bool(a.dump_outputs) and world > 1 and rank == 0   # N > 1: the headline path; its result is the same on every rank

    def step(i):
        o = op(i)
        if keep:
            last[0] = o
        return o[0].numel()
    ms, edges, _, launches, clocks = T.run(step, steps, a.warmup)
    if keep:
        dump_outputs(a.dump_outputs, last[0])
    last[0] = None
    out.update({'value': edges / (ms * 1e-3), 'unit': 'edges/s', 'ms_per_step': ms / steps, 'edges_per_step': edges / steps,
                'clocks': clocks, 'gpu_launches': launches})
    # e2e: seeds from pinned host memory, the full result back to pinned host memory on every rank
    cap = C5_BATCH * (FANOUT[0] + FANOUT[0] * FANOUT[1])
    copier = HostCopier(torch, dev, [cap, cap, cap + C5_BATCH, cap], n_slots=2)

    def step_e2e(i):
        s = seeds_host[i % n_seeds].to(dev, non_blocking=True)
        o = (P.sampler.neighbor_sample(rowptr, col, s, FANOUT) if world == 1 else P.sampler.dist_neighbor_sample(rowptr, col, s, FANOUT))[:4]
        copier.submit(o)
        return o[0].numel()
    e_steps = min(steps, 20)
    b0 = copier.bytes
    ms_e, edges_e, _, _, _ = T.run(step_e2e, e_steps, 3, finish=copier.drain)
    out['e2e'] = {'value': edges_e / (ms_e * 1e-3), 'unit': 'edges/s', 'h2d_bytes_per_step': C5_BATCH * 8,
                  'd2h_bytes_per_step': int((copier.bytes - b0) / (e_steps + 3)), 'ms_per_step': ms_e / e_steps, 'steps': e_steps,
                  'how': 'pinned seeds H2D + 4 result tensors D2H (pinned) every step on every rank; copies on a copy stream'}
    copier.close()
    if rank == 0 or world == 1:
        pass
    # roofline of the dominant kernel of the throughput schedule (rank 0's launches)
    if rank == 0:
        rf = sampler_roofline(abi, lambda i: op(i)[0].numel(), a.warmup, min(10, steps), torch, peaks, hbm_peak, peak_src, None)
        rf['kernel'] = {'k_sample': 'k_v2_sample', 'k_mark': 'k_v2_mark', 'k_assign': 'k_v2_assign'}.get(rf['kernel'], rf['kernel'])
        rf['traffic'] = traffic.get(rf['kernel'])
        if world > 1:
            rf['note'] = 'per-launch bytes count all edges of the pass (every rank streams all of them); the draws and table atomics are 1/N of that'
        out['roofline'] = rf
    elif world > 1:
        for i in range(a.warmup, a.warmup + min(10, steps)):   # keep the collective in step with rank 0's profiling calls
            op(i)
    if world > 1:
        # the same batches on ONE GPU, measured on every rank at once (they do not interact), for the speed-up
        torch.manual_seed(999)
        ms1, ed1, _, _, _ = T.run(lambda i: single(i)[0].numel(), min(steps, 20), 3)
        out['single_gpu_edges_per_s'] = ed1 / (ms1 * 1e-3)
        out['single_gpu_ms_per_step'] = ms1 / min(steps, 20)
        out['single_gpu_steps'] = min(steps, 20)
        out['speedup_vs_1gpu'] = out['value'] / out['single_gpu_edges_per_s']
        out['strong_scaling_efficiency'] = out['speedup_vs_1gpu'] / world
    del rowptr, col
    return out


if __name__ == '__main__':
    main()
