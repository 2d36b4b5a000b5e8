"""Reference outputs for config-size parity gates.  TEST/BENCH INFRASTRUCTURE ONLY — run as a subprocess by
bench.py's parity gate (and by tests/test_refproc.py, which checks that plumbing); never imported by the product.

    python oracle/ref_parity.py SPEC.pt

SPEC.pt is a torch.save'd dict written by tests/refproc.py: large inputs are raw files (normally under /dev/shm)
described as {'path', 'dtype', 'numel'} and mapped with torch.from_file, small ones are tensors.  The
reference is oracle/_ref/libpyg_ref.so — the reference's own sources compiled by oracle/build_ref.sh — through its
stock torch.ops.pyg.* operators (neighbor_kernel.cpp:899-955, ops/cpu/matmul_kernel.cpp); if that library is
absent the C restatement (oracle/oracle.py) answers instead and the result says kind='port'.  It cannot share a
process with libpyg.so (both register the pyg:: schemas), hence the subprocess.

kinds:
  homo    calls x neighbor_sample on one CSR, consecutively from torch.manual_seed(rng_seed)
  hetero  calls x hetero_neighbor_sample (torch.set_num_threads(1): the reference's multi-threaded hetero path
          shares its generator unsafely, SURVEY.md appendix A)
  matmul  segment_matmul(x, ptr, w)
Outputs go to spec['out'] (torch.save; big matmul outputs as a raw file next to it).
"""
import os.path as osp
import sys
import time

import torch

ROOT = osp.dirname(osp.dirname(osp.abspath(__file__)))
sys.path.insert(0, ROOT)

_REF = osp.join(ROOT, 'oracle', '_ref', 'libpyg_ref.so')
KIND = 'port'
if osp.exists(_REF):
    try:
        torch.ops.load_library(_REF)
        KIND = 'reference'
    except Exception:  # noqa
        KIND = 'port'
if KIND == 'port':
    from oracle import oracle as O

_DT = {'int64': torch.int64, 'int32': torch.int32, 'bfloat16': torch.bfloat16, 'float16': torch.float16,
       'float32': torch.float32}


def load(x):
    if isinstance(x, dict) and 'path' in x:
        return torch.from_file(x['path'], shared=False, size=x['numel'], dtype=_DT[x['dtype']]).view(x.get('shape', [-1]))
    return x


def rng_prefix():
    return torch.get_rng_state()[:24 + 624 * 8].clone()


def run_homo(spec):
    rowptr, col = load(spec['rowptr']), load(spec['col'])
    kw = spec.get('kwargs', {})
    torch.manual_seed(spec['rng_seed'])
    outs, secs = [], []
    for seed in spec['seeds']:
        seed = load(seed)
        t0 = time.perf_counter()
        if KIND == 'reference':
            r = torch.ops.pyg.neighbor_sample(rowptr, col, seed, spec['num_neighbors'], None, None, None, None,
                                              kw.get('csc', False), kw.get('replace', False), True, kw.get('disjoint', False),
                                              'uniform', kw.get('return_edge_id', True))
        else:
            r = O.neighbor_sample(rowptr, col, seed, spec['num_neighbors'], **kw)
        secs.append(time.perf_counter() - t0)
        outs.append(dict(row=r[0], col=r[1], node=r[2], eid=r[3], nph=list(r[4]), eph=list(r[5])))
    return dict(kind=KIND, calls=outs, rng_after=rng_prefix(), seconds=secs)


def run_hetero(spec):
    torch.set_num_threads(1)
    rowptr_d = {k: load(v) for k, v in spec['rowptr_dict'].items()}
    col_d = {k: load(v) for k, v in spec['col_dict'].items()}
    kw = spec.get('kwargs', {})
    torch.manual_seed(spec['rng_seed'])
    outs, secs = [], []
    for seed_d in spec['seeds']:
        seed_d = {k: load(v) for k, v in seed_d.items()}
        t0 = time.perf_counter()
        if KIND == 'reference':
            r = torch.ops.pyg.hetero_neighbor_sample(spec['node_types'], [tuple(e) for e in spec['edge_types']], rowptr_d, col_d,
                                                     seed_d, spec['num_neighbors_dict'], None, None, None, None,
                                                     kw.get('csc', False), kw.get('replace', False), True,
                                                     kw.get('disjoint', False), 'uniform', True)
        else:
            r = O.hetero_neighbor_sample(spec['node_types'], [tuple(e) for e in spec['edge_types']], rowptr_d, col_d, seed_d,
                                         spec['num_neighbors_dict'], **kw)
        secs.append(time.perf_counter() - t0)
        outs.append(dict(row=dict(r[0]), col=dict(r[1]), node=dict(r[2]), eid=dict(r[3]) if r[3] is not None else None,
                         nph={k: list(v) for k, v in r[4].items()}, eph={k: list(v) for k, v in r[5].items()}))
    return dict(kind=KIND, calls=outs, rng_after=rng_prefix(), seconds=secs)


def run_matmul(spec):
    x, w, ptr = load(spec['x']), load(spec['w']), load(spec['ptr'])
    if spec.get('threads'):
        torch.set_num_threads(spec['threads'])
    t0 = time.perf_counter()
    y = torch.ops.pyg.segment_matmul(x, ptr, w) if KIND == 'reference' else O.segment_matmul(x, ptr, w)
    dt = time.perf_counter() - t0
    if 'y_path' in spec:   # big result: raw file, viewed as int16 / int32 words by the reader
        out = torch.from_file(spec['y_path'], shared=True, size=y.numel(), dtype=y.dtype)
        out.copy_(y.reshape(-1))
        return dict(kind=KIND, y_shape=list(y.shape), seconds=[dt])
    return dict(kind=KIND, y=y, seconds=[dt])


if __name__ == '__main__':
    spec = torch.load(sys.argv[1], weights_only=False)
    res = {'homo': run_homo, 'hetero': run_hetero, 'matmul': run_matmul}[spec['kind']](spec)
    torch.save(res, spec['out'])
    print('REFPARITY_OK', KIND)
