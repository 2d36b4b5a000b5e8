"""Fixtures of the config-size parity tests (tests/test_config_parity.py) from the REFERENCE itself
(oracle/_ref/libpyg_ref.so, built by oracle/build_ref.sh):

    python tests/golden/make_golden_config.py [--out DIR] c2 c3 c4 c5

Writes DIR/config_<name>_outputs.npz (default DIR: tests/golden).  c4 and c5 draw their graphs from the CUDA generator
(tests/graphs.py), so they are made where a CUDA device is present; c2 and c3 need only the CPU.  The outputs are too
large to keep whole: every index tensor is stored as its shape and SHA-256 digest (next to the per-hop counts and the
state the calls leave the CPU generator in), the bf16 contraction as a seeded sample of rows (at least 8 of every
non-empty segment) plus the norm of every segment of the whole result.
"""
import argparse
import os
import os.path as osp
import sys

import numpy as np
import torch

HERE = osp.dirname(osp.abspath(__file__))
ROOT = osp.dirname(osp.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, osp.join(ROOT, 'tests'))

torch.ops.load_library(osp.join(ROOT, 'oracle', '_ref', 'libpyg_ref.so'))

from graphs import config_c2_inputs, config_c3_inputs, config_c4_inputs, config_c5_inputs  # noqa: E402
from refproc import rng_prefix, sha256  # noqa: E402


def put(out, key, t):
    out[key + '/shape'] = np.asarray(t.shape, dtype=np.int64)
    out[key + '/sha256'] = np.frombuffer(sha256(t), dtype=np.uint8)


def homo(rowptr, col, seeds, num_neighbors, rng_seed):
    """Consecutive neighbor_sample calls from one torch.manual_seed."""
    out = {}
    torch.manual_seed(rng_seed)
    for i, seed in enumerate(seeds):
        r = torch.ops.pyg.neighbor_sample(rowptr, col, seed, num_neighbors, None, None, None, None, False, False, True, False,
                                          'uniform', True)
        for k, t in zip(('row', 'col', 'node', 'eid'), r[:4]):
            put(out, f'call{i}/{k}', t)
        out[f'call{i}/nph'] = np.asarray(r[4], dtype=np.int64)
        out[f'call{i}/eph'] = np.asarray(r[5], dtype=np.int64)
        print(f'  call {i}: {r[0].numel()} edges')
    out['rng_after'] = rng_prefix().numpy()
    return out


def make_c2():
    rowptr, col, seeds = config_c2_inputs()
    return homo(rowptr, col, seeds, [15, 10], 12345)


def make_c3():
    x, ptr, w = config_c3_inputs()
    y = torch.ops.pyg.segment_matmul(x, ptr, w)
    p = ptr.tolist()
    g = torch.Generator().manual_seed(3)
    rows = [torch.randint(0, x.size(0), (512,), generator=g)]
    rows += [torch.randint(p[b], p[b + 1], (8,), generator=g) for b in range(len(p) - 1) if p[b + 1] > p[b]]
    rows = torch.unique(torch.cat(rows))
    return {'rows': rows.numpy(), 'y_bits': y[rows].view(torch.int16).numpy(),
            'segment_norm': np.array([float(y[p[b]:p[b + 1]].double().norm()) for b in range(len(p) - 1)])}


def make_c4():
    sizes, rowptr_d, col_d, seed = config_c4_inputs('cuda')
    edge_types = list(rowptr_d.keys())
    rel = {k: '__'.join(k) for k in edge_types}
    rowptr_d = {rel[k]: v.cpu() for k, v in rowptr_d.items()}
    col_d = {rel[k]: v.cpu() for k, v in col_d.items()}
    torch.cuda.empty_cache()
    nn = {rel[k]: [25, 15] for k in edge_types}
    threads = torch.get_num_threads()
    torch.set_num_threads(1)   # the reference's multi-threaded hetero path shares its generator unsafely (SURVEY.md appendix A)
    out = {}
    torch.manual_seed(4242)
    for i in range(2):
        r = torch.ops.pyg.hetero_neighbor_sample(['paper', 'author', 'institution'], edge_types, rowptr_d, col_d, {'paper': seed},
                                                 nn, None, None, None, None, False, False, True, False, 'uniform', True)
        for j, key in enumerate(('row', 'col', 'node', 'eid')):
            for k, v in r[j].items():
                put(out, f'call{i}/{key}/{k}', v)
        for k, v in r[4].items():
            out[f'call{i}/nph/{k}'] = np.asarray(v, dtype=np.int64)
        for k, v in r[5].items():
            out[f'call{i}/eph/{k}'] = np.asarray(v, dtype=np.int64)
        print(f'  call {i}: {sum(v.numel() for v in r[0].values())} edges')
    out['rng_after'] = rng_prefix().numpy()
    torch.set_num_threads(threads)
    return out


def make_c5():
    rowptr, col, seed = config_c5_inputs('cuda')
    rowptr, col = rowptr.cpu(), col.cpu()
    torch.cuda.empty_cache()
    return homo(rowptr, col, [seed], [15, 10], 7)


MAKERS = {'c2': make_c2, 'c3': make_c3, 'c4': make_c4, 'c5': make_c5}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('configs', nargs='+', choices=list(MAKERS))
    ap.add_argument('--out', default=HERE)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    for name in a.configs:
        print(name)
        path = osp.join(a.out, f'config_{name}_outputs.npz')
        np.savez_compressed(path, **MAKERS[name]())
        print('wrote', path, osp.getsize(path), 'bytes')


if __name__ == '__main__':
    main()
