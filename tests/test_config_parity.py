"""Parity at the BASELINE.json configurations themselves (VERDICT r1 "missing #5"; BASELINE.md 4.4): the CUDA path
against outputs of the reference's own CPU implementation (tests/golden/config_*_outputs.npz, made by
tests/golden/make_golden_config.py) on the full-size synthetic inputs of C2, C3 and C5 and on a 0.1-scale C4 —
bit-exact index tensors (SHA-256 of every tensor), counts and CPU generator state for the samplers; <= 1e-3 relative
Frobenius error and <= 1 storage ulp for the bf16 contraction on a sample of rows that covers every segment, and the norm
of every segment of the whole result within 1e-3."""
import os.path as osp

import numpy as np
import pytest
import torch

from graphs import config_c2_inputs, config_c3_inputs, config_c4_inputs, config_c5_inputs
from refproc import accumulation_bound, lowp_ulp_excess, rng_prefix, sha256

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


@pytest.fixture(scope='module')
def lib():
    import pyg_lib_b200 as P
    return P


def _gold(name):
    return np.load(osp.join(osp.dirname(osp.abspath(__file__)), 'golden', f'config_{name}_outputs.npz'))


def _check_tensor(t, gold, key):
    assert list(t.shape) == gold[key + '/shape'].tolist(), key
    assert sha256(t) == gold[key + '/sha256'].tobytes(), key


def _check_homo(out, gold, call):
    for k, t in zip(('row', 'col', 'node', 'eid'), out[:4]):
        _check_tensor(t, gold, f'call{call}/{k}')
    assert list(out[4]) == gold[f'call{call}/nph'].tolist()
    assert list(out[5]) == gold[f'call{call}/eph'].tolist()


def test_c2_products_full_size(lib):
    """configs[1]: ogbn-products-shaped CSR (2,449,029 nodes / 123,718,280 edges), fan-out [15,10], 1024 seeds —
    three consecutive calls from one torch.manual_seed, exactly bench.py's inputs."""
    rowptr, col, seeds = config_c2_inputs()
    gold = _gold('c2')
    d_rowptr, d_col = rowptr.to(DEV), col.to(DEV)
    torch.manual_seed(12345)
    for i, s in enumerate(seeds):
        out = lib.sampler.neighbor_sample(d_rowptr, d_col, s.to(DEV), [15, 10])
        assert out[0].numel() > 100_000
        _check_homo(out, gold, i)
    assert np.array_equal(rng_prefix().numpy(), gold['rng_after'])


def test_c3_segment_matmul_full_size(lib):
    """configs[2]: 64 relations, N = 2^20 ragged rows (one empty segment), 128 -> 128 bf16 — against the reference's
    CPU bf16 result on its stored rows (at least 8 of every segment), and every segment's norm."""
    x, ptr, w = config_c3_inputs()
    gold = _gold('c3')
    rows = torch.from_numpy(gold['rows'])
    y_ref = torch.from_numpy(gold['y_bits']).view(torch.bfloat16)
    seg_norm = gold['segment_norm']
    N = x.size(0)
    seg = torch.searchsorted(ptr, rows, right=True) - 1
    tol = accumulation_bound(x.to(DEV), ptr, w.to(DEV)).cpu()[rows]   # (checker arithmetic; torch on the GPU only because it is quick)
    for ptr_arg in (ptr.to(DEV), ptr):
        y = lib.ops.segment_matmul(x.to(DEV), ptr_arg, w.to(DEV)).cpu()
        ys = y[rows]
        rel = float((ys.float() - y_ref.float()).norm() / y_ref.float().norm())
        assert rel <= 1e-3, rel
        assert lowp_ulp_excess(ys, y_ref, tol) <= 1.0
        sizes = (ptr[1:] - ptr[:-1]).tolist()
        for b, (lo, n_b) in enumerate(zip(ptr[:-1].tolist(), sizes)):   # per segment, so a wrong W[b] cannot hide in the norm
            if n_b:
                sel = seg == b
                d = (ys[sel].float() - y_ref[sel].float()).norm() / y_ref[sel].float().norm().clamp_min(1e-30)
                assert float(d) <= 1e-3, (b, float(d))
                assert abs(float(y[lo:lo + n_b].double().norm()) - seg_norm[b]) <= 1e-3 * seg_norm[b], b
    # and against exact arithmetic (fp64 of the bf16 inputs), SURVEY.md 8(c): <= 2e-3
    rows = torch.arange(0, N, 997)
    seg = torch.searchsorted(ptr, rows, right=True) - 1
    exact = torch.einsum('nk,nkm->nm', x[rows].double(), w[seg].double())
    assert float((y[rows].double() - exact).norm() / exact.norm()) <= 2e-3


def test_c4_mag240m_shaped_tenth_scale(lib):
    """configs[3] at 0.1 scale (12.2 M papers / 12.2 M authors / 2.6 k institutions, 346 M edges over 6 relations),
    fan-out [25,15] for every relation, 1024 paper seeds, against the 1-thread reference."""
    sizes, rowptr_d, col_d, seed = config_c4_inputs(DEV)
    rel = {k: '__'.join(k) for k in rowptr_d}
    nn = {k: [25, 15] for k in rowptr_d}
    gold = _gold('c4')
    torch.manual_seed(4242)
    for call in range(2):
        out = lib.sampler.hetero_neighbor_sample(rowptr_d, col_d, {'paper': seed.to(DEV)}, nn)
        total = 0
        for i, key in enumerate(('row', 'col', 'node', 'eid')):
            for k, v in out[i].items():
                kk = rel[k] if isinstance(k, tuple) else k
                _check_tensor(v, gold, f'call{call}/{key}/{kk}')
                total += v.numel() if key == 'row' else 0
        for j, key in ((4, 'nph'), (5, 'eph')):
            p = f'call{call}/{key}/'
            assert {rel.get(k, k): list(v) for k, v in out[j].items()} == \
                {f[len(p):]: gold[f].tolist() for f in gold.files if f.startswith(p)}, key
        assert total > 100_000
    assert np.array_equal(rng_prefix().numpy(), gold['rng_after'])


def test_c5_papers100m_shaped_full_size_single_gpu(lib):
    """configs[4]'s graph and batch on ONE GPU (the multi-GPU run must return exactly this, tests/test_dist.py and the
    bench's own gate check that): papers100M-shaped CSR (111,059,956 nodes / 1,615,685,872 edges), 65,536 seeds."""
    rowptr, col, seed = config_c5_inputs(DEV)
    gold = _gold('c5')
    torch.manual_seed(7)
    out = lib.sampler.neighbor_sample(rowptr, col, seed.to(DEV), [15, 10])
    assert out[0].numel() > 3_000_000
    _check_homo(out, gold, 0)
    assert np.array_equal(rng_prefix().numpy(), gold['rng_after'])
