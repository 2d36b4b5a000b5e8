"""Deterministic synthetic inputs shared by the golden generator, the oracle tests, the GPU parity
tests and bench.py.  Everything is derived from integer seeds with CPU torch.Generator streams, so
the GPU box regenerates bit-identical inputs (same image, same torch build)."""
from typing import Dict, List, Tuple

import torch


def cycle_graph(n: int):
    """test/csrc/graph.h:5-13 (note Python-style modulo: node 0's neighbours are [n-1, 1])."""
    rowptr = torch.arange(0, 2 * n + 1, 2)
    col = torch.stack([torch.arange(-1, n - 1) % n, torch.arange(1, n + 1) % n], dim=1).flatten()
    return rowptr, col


def random_csr(n: int, avg_deg: int, seed: int, big: List[Tuple[int, int]] = (), zero_frac: float = 0.1):
    g = torch.Generator().manual_seed(seed)
    deg = torch.randint(0, 2 * avg_deg + 1, (n,), generator=g)
    deg[torch.rand(n, generator=g) < zero_frac] = 0
    for i, d in big:
        deg[i] = d
    rowptr = torch.zeros(n + 1, dtype=torch.int64)
    rowptr[1:] = deg.cumsum(0)
    col = torch.randint(0, n, (int(rowptr[-1]),), generator=g)
    return rowptr, col


def lognormal_csr(n: int, e: int, seed: int, device='cpu', dtype=torch.int64, mean=3.0, std=1.2):
    """SURVEY.md 8(d) C2 recipe: log-normal degrees scaled to sum E, uniform random targets."""
    g = torch.Generator(device=device).manual_seed(seed)
    w = torch.empty(n, device=device, dtype=torch.float64).log_normal_(mean, std, generator=g)
    deg = torch.floor(w * (e / w.sum())).to(torch.int64)
    rem = int(e - int(deg.sum()))
    if rem > 0:
        deg[:rem] += 1
    rowptr = torch.zeros(n + 1, dtype=torch.int64, device=device)
    torch.cumsum(deg, 0, out=rowptr[1:])
    col = torch.randint(0, n, (e,), generator=g, device=device, dtype=dtype)
    return rowptr.to(dtype), col


HOMO_CASES: Dict[str, dict] = {
    # known-answer vectors of test/csrc/sampler/test_neighbor.cpp (cycle graph, seeds [2,3])
    'cycle_full': dict(graph=('cycle', 6), seeds=[2, 3], num_neighbors=[-1, -1], rng_seed=0),
    'cycle_norep': dict(graph=('cycle', 6), seeds=[2, 3], num_neighbors=[1, 1], rng_seed=123456),
    'cycle_rep': dict(graph=('cycle', 6), seeds=[2, 3], num_neighbors=[1, 1], rng_seed=123456, replace=True),
    'cycle_disjoint': dict(graph=('cycle', 6), seeds=[2, 3], num_neighbors=[2, 2], rng_seed=0, disjoint=True),
    'zero_deg': dict(graph=('zero', 5), seeds=[0, 1, 2, 3, 4], num_neighbors=[-1, -1], rng_seed=0),
    # random graphs
    'rand_15_10': dict(graph=('rand', 2000, 20, 1), n_seeds=64, num_neighbors=[15, 10], rng_seed=12345),
    'rand_15_10_rep': dict(graph=('rand', 2000, 20, 1), n_seeds=64, num_neighbors=[15, 10], rng_seed=12345,
                           replace=True),
    'rand_csc': dict(graph=('rand', 2000, 20, 2), n_seeds=32, num_neighbors=[10, 5], rng_seed=7, csc=True),
    'rand_3hop': dict(graph=('rand', 3000, 8, 3), n_seeds=16, num_neighbors=[5, 5, 5], rng_seed=99),
    'rand_full': dict(graph=('rand', 1500, 6, 4), n_seeds=8, num_neighbors=[-1, 4, -1], rng_seed=5),
    'rand_k40': dict(graph=('rand', 1000, 60, 5), n_seeds=8, num_neighbors=[40, 3], rng_seed=11),
    'rand_k40_rep': dict(graph=('rand', 1000, 60, 5), n_seeds=8, num_neighbors=[40, 3], rng_seed=11,
                         replace=True),
    'rand_k100': dict(graph=('rand', 600, 150, 6), n_seeds=4, num_neighbors=[100], rng_seed=13),
    'rand_dupseeds': dict(graph=('rand', 2000, 20, 1), seeds=[4, 4, 9, 4, 9, 1, 1500, 4], num_neighbors=[5, 5],
                          rng_seed=1),
    'rand_zero_fanout': dict(graph=('rand', 2000, 20, 1), n_seeds=16, num_neighbors=[0, 3], rng_seed=3),
    # degrees >= 65536 -> mixed 16/32-bit draws (rand_engine.h:43-61)
    'bigdeg': dict(graph=('rand', 400, 10, 7, [(5, 70000), (77, 65540), (100, 65536), (101, 65535)]),
                   seeds=[5, 3, 77, 100, 8, 101, 5], num_neighbors=[9, 4], rng_seed=21),
    'bigdeg_rep': dict(graph=('rand', 400, 10, 7, [(5, 70000), (77, 65540), (100, 65536), (101, 65535)]),
                       seeds=[5, 3, 77, 100, 8, 101], num_neighbors=[9, 4], rng_seed=21, replace=True),
    'bigdeg_k40': dict(graph=('rand', 400, 10, 7, [(5, 70000), (77, 65540), (100, 65536), (101, 65535)]),
                       seeds=[77, 100, 101, 5], num_neighbors=[40], rng_seed=22),
    'rand_disjoint': dict(graph=('rand', 2000, 20, 1), n_seeds=24, num_neighbors=[6, 4], rng_seed=17,
                          disjoint=True),
    'rand_disjoint_rep': dict(graph=('rand', 2000, 20, 1), n_seeds=24, num_neighbors=[6, 4], rng_seed=17,
                              disjoint=True, replace=True),
}


# temporal cases: neighbourhoods sorted by time (node time of the neighbour, or edge time); need disjoint
HOMO_CASES.update({
    'temporal_node': dict(graph=('rand', 1500, 14, 41), n_seeds=40, num_neighbors=[5, 4], rng_seed=31, disjoint=True,
                          temporal='node'),
    'temporal_node_last': dict(graph=('rand', 1500, 14, 41), n_seeds=40, num_neighbors=[5, 4], rng_seed=31, disjoint=True,
                               temporal='node', strategy='last'),
    'temporal_node_seedtime_rep': dict(graph=('rand', 1500, 14, 42), n_seeds=40, num_neighbors=[6, 3], rng_seed=32,
                                       disjoint=True, temporal='node', seed_time=True, replace=True),
    'temporal_edge': dict(graph=('rand', 1500, 14, 43), n_seeds=40, num_neighbors=[5, 4], rng_seed=33, disjoint=True,
                          temporal='edge', seed_time=True),
    'temporal_edge_last': dict(graph=('rand', 1500, 14, 43), n_seeds=40, num_neighbors=[-1, 3], rng_seed=33, disjoint=True,
                               temporal='edge', seed_time=True, strategy='last'),
})


def build_temporal(case: dict, rowptr, col, seed):
    """(col', node_time, edge_time, seed_time) for a temporal case; col' has time-sorted neighbourhoods."""
    n = rowptr.numel() - 1
    g = torch.Generator().manual_seed(5000 + case['rng_seed'])
    node_time = edge_time = seed_time = None
    deg = rowptr[1:] - rowptr[:-1]
    row_of_edge = torch.repeat_interleave(torch.arange(n), deg)
    if case['temporal'] == 'node':
        node_time = torch.randint(0, 50, (n,), generator=g)
        key = row_of_edge * 1000 + node_time[col]          # sort each neighbourhood by neighbour time (stable)
        order = torch.sort(key, stable=True).indices
        col = col[order]
    else:
        et = torch.randint(0, 50, (col.numel(),), generator=g)
        key = row_of_edge * 1000 + et
        order = torch.sort(key, stable=True).indices
        col, edge_time = col[order], et[order]
    if case.get('seed_time'):
        seed_time = torch.randint(5, 60, (seed.numel(),), generator=g)
    return col.contiguous(), node_time, edge_time, seed_time


def build_homo(case: dict):
    g = case['graph']
    if g[0] == 'cycle':
        rowptr, col = cycle_graph(g[1])
        n = g[1]
    elif g[0] == 'zero':
        rowptr, col = torch.zeros(g[1] + 1, dtype=torch.int64), torch.zeros(0, dtype=torch.int64)
        n = g[1]
    else:
        rowptr, col = random_csr(g[1], g[2], g[3], big=g[4] if len(g) > 4 else ())
        n = g[1]
    if 'seeds' in case:
        seed = torch.tensor(case['seeds'], dtype=torch.int64)
    else:
        gg = torch.Generator().manual_seed(1000 + case['rng_seed'])
        seed = torch.randperm(n, generator=gg)[:case['n_seeds']]
    return rowptr, col, seed


# ------------------------------------------------------------------------------------- hetero
_MAG_TYPES = ['paper', 'author', 'institution']
_MAG_RELS = [('paper', 'cites', 'paper'), ('author', 'writes', 'paper'), ('author', 'affiliated_with', 'institution'),
             ('paper', 'rev_writes', 'author'), ('institution', 'rev_affiliated_with', 'author'),
             ('paper', 'rev_cites', 'paper')]

HETERO_CASES: Dict[str, dict] = {
    'cycle_single_rel': dict(kind='cycle', num_neighbors=[2, 2], rng_seed=0),
    'mag_small': dict(kind='mag', sizes=dict(paper=600, author=400, institution=20), avg_deg=6,
                      n_seeds=dict(paper=16), num_neighbors=[5, 3], rng_seed=12345, gseed=31),
    'mag_small_csc': dict(kind='mag', sizes=dict(paper=600, author=400, institution=20), avg_deg=6,
                          n_seeds=dict(paper=16), num_neighbors=[5, 3], rng_seed=12345, gseed=31, csc=True),
    'mag_25_15': dict(kind='mag', sizes=dict(paper=3000, author=2000, institution=40), avg_deg=30,
                      n_seeds=dict(paper=4), num_neighbors=[25, 15], rng_seed=5, gseed=32),
    'mag_two_seed_types_rep': dict(kind='mag', sizes=dict(paper=600, author=400, institution=20), avg_deg=6,
                                   n_seeds=dict(author=8, paper=8), num_neighbors=[4, 4], rng_seed=77, gseed=33,
                                   replace=True),
    'mag_disjoint': dict(kind='mag', sizes=dict(paper=600, author=400, institution=20), avg_deg=6,
                         n_seeds=dict(paper=6, author=5), num_neighbors=[4, 3], rng_seed=8, gseed=34,
                         disjoint=True),
}


def build_hetero(case: dict):
    """Returns (node_types, edge_types, rowptr_dict, col_dict, seed_dict, num_neighbors_dict) with
    'src__rel__dst' string keys, i.e. the operator-level arguments (neighbor.cpp:137-147)."""
    if case['kind'] == 'cycle':
        rowptr, col = cycle_graph(6)
        return (['paper'], [('paper', 'to', 'paper')], {'paper__to__paper': rowptr}, {'paper__to__paper': col},
                {'paper': torch.arange(2, 4)}, {'paper__to__paper': list(case['num_neighbors'])})
    sizes = case['sizes']
    csc = case.get('csc', False)
    rowptr_d, col_d, nn_d = {}, {}, {}
    for i, (a, r, b) in enumerate(_MAG_RELS):
        # CSR over the *source* side (rows) of the traversal: src = a (csr) or b (csc)
        rows_t, cols_t = (a, b) if not csc else (b, a)
        g = torch.Generator().manual_seed(case['gseed'] * 100 + i)
        n_rows, n_cols = sizes[rows_t], sizes[cols_t]
        avg = case['avg_deg'] if n_rows > 50 else case['avg_deg'] * 20
        deg = torch.randint(0, 2 * avg + 1, (n_rows,), generator=g)
        rowptr = torch.zeros(n_rows + 1, dtype=torch.int64)
        rowptr[1:] = deg.cumsum(0)
        col = torch.randint(0, n_cols, (int(rowptr[-1]),), generator=g)
        key = '__'.join((a, r, b))
        rowptr_d[key], col_d[key], nn_d[key] = rowptr, col, list(case['num_neighbors'])
    seed_d = {}
    for t, ns in case['n_seeds'].items():
        g = torch.Generator().manual_seed(case['gseed'] * 7 + len(seed_d))
        seed_d[t] = torch.randperm(sizes[t], generator=g)[:ns]
    return list(_MAG_TYPES), list(_MAG_RELS), rowptr_d, col_d, seed_d, nn_d


# ------------------------------------------------------------------------------------- matmul
MATMUL_CASES: Dict[str, dict] = {
    # test/ops/test_matmul.py:14-45
    'ref_test_f32': dict(N=8, K=16, M=32, ptr=[0, 5, 8], dtype='float32', seed=0),
    'ref_test_bf16': dict(N=8, K=16, M=32, ptr=[0, 5, 8], dtype='bfloat16', seed=0),
    # BASELINE.json configs[0]
    'c1_f32': dict(N=1024, K=64, M=64, ptr=[0, 256, 512, 768, 1024], dtype='float32', seed=0),
    # ragged, one empty segment, not tile aligned (SURVEY 8d C3 recipe, scaled down)
    'ragged_bf16': dict(N=3000, K=128, M=128, B=8, dtype='bfloat16', seed=1, ragged=True),
    'ragged_f16': dict(N=1000, K=64, M=96, B=5, dtype='float16', seed=2, ragged=True),
    'ragged_f32_odd': dict(N=777, K=40, M=24, B=6, dtype='float32', seed=3, ragged=True),
}


def ragged_ptr(N: int, B: int, seed: int, empty: int = 1) -> torch.Tensor:
    """Segment lengths ~ log-normal(0,1) normalised to N (largest remainder), one forced empty."""
    g = torch.Generator().manual_seed(seed)
    w = torch.empty(B, dtype=torch.float64).log_normal_(0.0, 1.0, generator=g)
    if B > 1 and empty is not None:
        w[empty % B] = 0.0
    ideal = w / w.sum() * N
    ln = torch.floor(ideal).to(torch.int64)
    rem = int(N - int(ln.sum()))
    if rem > 0:
        order = torch.argsort(ideal - ln.double(), descending=True)
        order = order[w[order] > 0][:rem]
        ln[order] += 1
    ptr = torch.zeros(B + 1, dtype=torch.int64)
    ptr[1:] = ln.cumsum(0)
    assert int(ptr[-1]) == N
    return ptr


def build_matmul(case: dict, device='cpu'):
    dt = getattr(torch, case['dtype'])
    g = torch.Generator().manual_seed(case['seed'])
    if 'ptr' in case:
        ptr = torch.tensor(case['ptr'], dtype=torch.int64)
    else:
        ptr = ragged_ptr(case['N'], case['B'], case['seed'] + 100)
    B = ptr.numel() - 1
    x = torch.randn(case['N'], case['K'], generator=g).to(dt)
    w = (torch.randn(B, case['K'], case['M'], generator=g) / case['K'] ** 0.5).to(dt)
    return x.to(device), ptr, w.to(device)


# pyg::subgraph cases: (graph spec as in HOMO_CASES, how the node set is drawn)
SUBGRAPH_CASES: Dict[str, dict] = {
    # known-answer vector of test/csrc/sampler/test_subgraph.cpp:7-24 (cycle graph, nodes 1..4)
    'cycle_kat': dict(graph=('cycle', 6), nodes=[1, 2, 3, 4]),
    'cycle_dups_unsorted': dict(graph=('cycle', 6), nodes=[4, 1, 4, 2, 1]),
    'empty_set': dict(graph=('cycle', 6), nodes=[]),
    'rand_small': dict(graph=('rand', 2000, 20, 1), n_nodes=300, seed=5),
    'rand_dense_set': dict(graph=('rand', 1500, 30, 2), n_nodes=1200, seed=6),
    'rand_dups': dict(graph=('rand', 3000, 12, 3), n_nodes=500, seed=7, dup=200),
    'bigdeg': dict(graph=('rand', 400, 10, 7, [(5, 70000), (77, 65540)]), n_nodes=150, seed=8, must=[5, 77]),
}


def build_subgraph(case):
    """(rowptr, col, nodes) of a SUBGRAPH_CASES entry (int64 CPU tensors)."""
    rowptr, col, _ = build_homo(dict(graph=case['graph'], seeds=[0], num_neighbors=[1], rng_seed=0))
    n = rowptr.numel() - 1
    if 'nodes' in case:
        return rowptr, col, torch.tensor(case['nodes'], dtype=torch.int64)
    g = torch.Generator().manual_seed(case['seed'])
    nodes = torch.randperm(n, generator=g)[:case['n_nodes']]
    if 'must' in case:
        nodes = torch.cat([torch.tensor(case['must'], dtype=torch.int64), nodes[~torch.isin(nodes, torch.tensor(case['must']))]])
    if case.get('dup', 0):
        extra = nodes[torch.randint(0, nodes.numel(), (case['dup'],), generator=g)]
        nodes = torch.cat([nodes, extra])[torch.randperm(nodes.numel() + case['dup'], generator=g)]
    return rowptr, col, nodes.to(torch.int64)


# pyg::dist_neighbor_sample cases (one hop, no mapping); first four = test/csrc/sampler/test_dist_neighbor.cpp
DIST_CASES: Dict[str, dict] = {
    'cycle_full': dict(graph=('cycle', 6), seeds=[2, 3], k=-1, rng_seed=0),
    'cycle_norep': dict(graph=('cycle', 6), seeds=[2, 3], k=1, rng_seed=123456),
    'cycle_rep': dict(graph=('cycle', 6), seeds=[2, 3], k=2, rng_seed=123456, replace=True),
    'cycle_disjoint': dict(graph=('cycle', 6), seeds=[2, 3], k=2, rng_seed=0, disjoint=True),
    'rand_15': dict(graph=('rand', 2000, 20, 1), n_seeds=64, k=15, rng_seed=12345),
    'rand_15_rep': dict(graph=('rand', 2000, 20, 1), n_seeds=64, k=15, rng_seed=12345, replace=True),
    'rand_all': dict(graph=('rand', 1500, 6, 4), n_seeds=40, k=-1, rng_seed=5),
    'rand_k40_disjoint': dict(graph=('rand', 1000, 60, 5), n_seeds=8, k=40, rng_seed=11, disjoint=True),
    'rand_dupseeds': dict(graph=('rand', 2000, 20, 1), seeds=[4, 4, 9, 4, 9, 1, 1500, 4], k=5, rng_seed=1),
    'rand_zero': dict(graph=('rand', 2000, 20, 1), n_seeds=16, k=0, rng_seed=3),
    'bigdeg': dict(graph=('rand', 400, 10, 7, [(5, 70000), (77, 65540), (100, 65536), (101, 65535)]),
                   seeds=[5, 3, 77, 100, 8, 101, 5], k=9, rng_seed=21),
}


def build_dist(case):
    """(rowptr, col, seed) of a DIST_CASES entry."""
    return build_homo(dict(case, num_neighbors=[case['k']]))


# pyg::relabel_neighborhood cases: inputs are what one hop of dist_neighbor_sample returns for a DIST_CASES entry
# (seeds, the unmapped neighbours, neighbours per seed), plus hand-made ones
RELABEL_CASES: Dict[str, dict] = {
    # test/csrc/sampler/test_dist_relabel.cpp:9-36 and :38-60
    'kat': dict(seed=[2, 3], sampled=[1, 3, 2, 4], counts=[2, 2], num_nodes=6),
    'kat_disjoint': dict(seed=[2, 3], sampled=[1, 3, 2, 4], counts=[2, 2], num_nodes=6, batch=[0, 0, 1, 1]),
    'zero_counts_dup_seeds': dict(seed=[5, 5, 1], sampled=[7, 5, 7, 9, 1], counts=[0, 3, 0, 2, 0], num_nodes=12),
    'from_rand_15': dict(dist='rand_15'),
    'from_rand_15_rep_csc': dict(dist='rand_15_rep', csc=True),
    'from_rand_k40_disjoint': dict(dist='rand_k40_disjoint'),
    'from_bigdeg': dict(dist='bigdeg'),
}


def build_relabel(case, oracle_dist):
    """(seed, sampled, counts, num_nodes, batch, csc, disjoint); `oracle_dist(rowptr, col, seed, k, **kw)` supplies the
    one-hop sample the derived cases relabel (tests pass oracle.dist_neighbor_sample, make_golden passes the reference)."""
    if 'dist' not in case:
        b = case.get('batch')
        return (torch.tensor(case['seed']), torch.tensor(case['sampled']), list(case['counts']), case['num_nodes'],
                None if b is None else torch.tensor(b), case.get('csc', False), b is not None)
    dc = DIST_CASES[case['dist']]
    rowptr, col, seed = build_dist(dc)
    torch.manual_seed(dc['rng_seed'])
    node, eid, cum = oracle_dist(rowptr, col, seed, dc['k'], replace=dc.get('replace', False), disjoint=dc.get('disjoint', False))
    S = seed.numel()
    counts = [int(cum[i + 1] - cum[i]) for i in range(S)]
    if dc.get('disjoint', False):
        return seed, node[S:, 1].contiguous(), counts, rowptr.numel() - 1, node[S:, 0].contiguous(), case.get('csc', False), True
    return seed, node[S:].contiguous(), counts, rowptr.numel() - 1, None, case.get('csc', False), False


# pyg::hetero_relabel_neighborhood: synthetic inputs (the op does not need a graph): random seeds, random per-layer
# neighbour counts per (edge type, source node) and random sampled ids per destination type
HETERO_RELABEL_CASES: Dict[str, dict] = {
    'two_types': dict(node_types=['a', 'b'], edge_types=[('a', 'x', 'b'), ('b', 'y', 'a'), ('a', 'z', 'a')],
                      seeds={'a': 5, 'b': 3}, layers=[{'a': None, 'b': None}, {'a': 9, 'b': 7}], id_range=40, rng=1),
    'two_types_csc': dict(node_types=['a', 'b'], edge_types=[('a', 'x', 'b'), ('b', 'y', 'a'), ('a', 'z', 'a')],
                          seeds={'a': 5, 'b': 3}, layers=[{'a': None, 'b': None}, {'a': 9, 'b': 7}], id_range=40, rng=2, csc=True),
    'one_seed_type_3_layers': dict(node_types=['p', 'q', 'r'], edge_types=[('p', 'w', 'q'), ('q', 'v', 'p'), ('q', 'u', 'r'), ('r', 't', 'q')],
                                   seeds={'p': 16}, layers=[{'p': None, 'q': 0, 'r': 0}, {'p': 3, 'q': 30, 'r': 5}, {'p': 20, 'q': 11, 'r': 17}],
                                   id_range=200, rng=3),
    'disjoint': dict(node_types=['a', 'b'], edge_types=[('a', 'x', 'b'), ('b', 'y', 'a')], seeds={'a': 4, 'b': 6},
                     layers=[{'a': None, 'b': None}, {'a': 8, 'b': 5}], id_range=12, rng=4, disjoint=True),
}


def build_hetero_relabel(case):
    """(node_types, edge_types, seed_dict, sampled_dict, counts_dict {rel: [[...] per layer]}, num_nodes_dict, batch_dict|None,
    csc, disjoint).  layers[l][t] = number of source nodes of type t in layer l (None: its seeds)."""
    g = torch.Generator().manual_seed(case['rng'])
    csc, disjoint = case.get('csc', False), case.get('disjoint', False)
    nt, et = case['node_types'], case['edge_types']
    R = case['id_range']
    seed_dict = {t: torch.randint(0, R, (n,), generator=g) for t, n in case['seeds'].items()}
    counts = {'__'.join(k): [] for k in et}
    total = {t: 0 for t in nt}
    n_batches = sum(case['seeds'].values())
    for layer in case['layers']:
        for k in et:
            src, dst = (k[2], k[0]) if csc else (k[0], k[2])
            n_src = layer[src]
            if n_src is None:
                n_src = case['seeds'].get(src, 0)
            c = torch.randint(0, 4, (n_src,), generator=g).tolist()
            counts['__'.join(k)].append(c)
            total[dst] += sum(c)
    sampled = {t: torch.randint(0, R, (total[t],), generator=g) for t in nt}
    batch = {t: torch.randint(0, max(n_batches, 1), (total[t],), generator=g) for t in nt} if disjoint else None
    return nt, et, seed_dict, sampled, counts, {t: R for t in nt}, batch, csc, disjoint


# pyg::merge_sampler_outputs: the seeds of a DIST_CASES-like problem are dealt to P partitions, every partition
# samples its own seeds with dist_neighbor_sample, merge restores the seed order
MERGE_CASES: Dict[str, dict] = {
    # test/csrc/sampler/test_dist_merge_outputs.cpp:7-48 and :50-91
    'kat': dict(node_ids=[[2, 7, 8], [0, 1, 4, 5, 6], [3, 9, 10]], edge_ids=[[17, 18], [14, 15, 16], [19, 20]],
                cumsum=[[1, 3], [2, 4, 5], [1, 3]], partition_ids=[1, 1, 0, 2], partition_orders=[0, 1, 0, 0], k=2),
    'kat_all': dict(node_ids=[[2, 7, 8], [0, 1, 4, 5, 6], [3, 9, 10, 11]], edge_ids=[[17, 18], [14, 15, 16], [19, 20, 21]],
                    cumsum=[[1, 3], [2, 4, 5], [1, 4]], partition_ids=[1, 1, 0, 2], partition_orders=[0, 1, 0, 0], k=-1),
    'rand_3parts': dict(graph=('rand', 2000, 20, 1), n_seeds=200, k=7, parts=3, rng_seed=8),
    'rand_5parts_rep_disjoint': dict(graph=('rand', 1500, 12, 2), n_seeds=97, k=4, parts=5, rng_seed=9, replace=True, disjoint=True),
    'rand_all_neighbors': dict(graph=('rand', 1200, 6, 4), n_seeds=60, k=-1, parts=4, rng_seed=10),
}


def build_merge(case, oracle_dist):
    """(node_ids, edge_ids, cumsum lists, partition_ids, partition_orders, num_partitions, num_neighbors, batch|None, disjoint)"""
    if 'node_ids' in case:
        t = lambda x: torch.tensor(x, dtype=torch.int64)  # noqa: E731
        return ([t(x) for x in case['node_ids']], [t(x) for x in case['edge_ids']], [list(c) for c in case['cumsum']],
                list(case['partition_ids']), list(case['partition_orders']), len(case['node_ids']), case['k'], None, False)
    rowptr, col, seed = build_homo(dict(graph=case['graph'], n_seeds=case['n_seeds'], num_neighbors=[1], rng_seed=0))
    g = torch.Generator().manual_seed(case['rng_seed'])
    P = case['parts']
    part = torch.randint(0, P, (seed.numel(),), generator=g)
    disjoint = case.get('disjoint', False)
    node_ids, edge_ids, cums, orders = [], [], [], [0] * seed.numel()
    torch.manual_seed(case['rng_seed'])
    for p in range(P):
        idx = (part == p).nonzero().flatten()
        for o, j in enumerate(idx.tolist()):
            orders[j] = o
        # (merge reads node ids as one flat list: the plain node column, also for disjoint sampling)
        node, eid, cum = oracle_dist(rowptr, col, seed[idx], case['k'], replace=case.get('replace', False), disjoint=False)
        node_ids.append(node.contiguous()); edge_ids.append(eid.contiguous()); cums.append([int(x) for x in cum])
    batch = torch.arange(seed.numel(), dtype=torch.int64) if disjoint else None
    return node_ids, edge_ids, cums, part.tolist(), orders, P, case['k'], batch, disjoint


# ------------------------------------------------------------------------------------- config-size generators
MAG240M_NODES = {'paper': 121_751_666, 'author': 122_383_112, 'institution': 25_721}
MAG240M_EDGES = {('paper', 'cites', 'paper'): 1_297_748_926, ('author', 'writes', 'paper'): 386_022_720,
                 ('author', 'affiliated_with', 'institution'): 44_592_586, ('paper', 'rev_writes', 'author'): 386_022_720,
                 ('institution', 'rev_affiliated_with', 'author'): 44_592_586, ('paper', 'rev_cites', 'paper'): 1_297_748_926}


def mag240m_shaped(scale: float, device='cpu', seed0: int = 10):
    """BASELINE.json configs[3]: 3 node types / 6 edge types with MAG240M's node and edge counts times `scale`
    (SURVEY.md 8d C4), log-normal degrees per relation, uniform targets.  Returns (sizes, rowptr_dict, col_dict) keyed by
    edge-type tuples.  Generated with `device`'s generator: bit-identical across runs on the same device type."""
    sizes = {k: max(int(v * scale), 64) for k, v in MAG240M_NODES.items()}
    rowptr_d, col_d = {}, {}
    for i, (k, e) in enumerate(MAG240M_EDGES.items()):
        e = int(e * scale)
        g = torch.Generator(device=device).manual_seed(seed0 + i)
        w = torch.empty(sizes[k[0]], device=device, dtype=torch.float32).log_normal_(3.0, 1.2, generator=g)
        deg = torch.floor(w.double() * (e / float(w.double().sum()))).to(torch.int64)
        del w
        rem = e - int(deg.sum())
        deg[:rem] += 1
        rowptr = torch.zeros(sizes[k[0]] + 1, dtype=torch.int64, device=device)
        torch.cumsum(deg, 0, out=rowptr[1:])
        del deg
        col_d[k] = torch.randint(0, sizes[k[2]], (e,), generator=g, device=device, dtype=torch.int64)
        rowptr_d[k] = rowptr
    return sizes, rowptr_d, col_d


# Inputs of the config-size parity tests (tests/test_config_parity.py) and of the fixtures they compare with
# (tests/golden/make_golden_config.py).  c4 and c5 draw their graphs from the CUDA generator of `device`.
def config_c2_inputs():
    """configs[1]: ogbn-products-shaped CSR (bench.py's graph) and three 1024-seed batches."""
    n, e = 2_449_029, 123_718_280
    rowptr, col = lognormal_csr(n, e, seed=1)
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(2))
    return rowptr, col, [perm[b * 1024:(b + 1) * 1024].clone() for b in (0, 1, 2)]


def config_c3_inputs():
    """configs[2]: 64 relations, N = 2^20 ragged rows (one empty segment), 128 -> 128 bf16.  Returns (x, ptr, w)."""
    N, K, M, B = 1 << 20, 128, 128, 64
    g = torch.Generator().manual_seed(0)
    x = torch.randn(N, K, generator=g).to(torch.bfloat16)
    w = (torch.randn(B, K, M, generator=g) / K ** 0.5).to(torch.bfloat16)
    return x, ragged_ptr(N, B, 100), w


def config_c4_inputs(device):
    """configs[3] at 0.1 scale: (sizes, rowptr_dict, col_dict, 1024 paper seeds)."""
    sizes, rowptr_d, col_d = mag240m_shaped(0.1, device=device)
    seed = torch.randperm(sizes['paper'], generator=torch.Generator().manual_seed(3))[:1024]
    return sizes, rowptr_d, col_d, seed


def config_c5_inputs(device):
    """configs[4]'s graph and batch: papers100M-shaped CSR (111,059,956 nodes / 1,615,685,872 edges), 65,536 seeds."""
    n, e = 111_059_956, 1_615_685_872
    rowptr, col = lognormal_csr(n, e, seed=1, device=device)
    seed = torch.randperm(n, generator=torch.Generator().manual_seed(2))[:65536]
    return rowptr, col, seed


# ------------------------------------------------------------------------------------- biased (edge_weight) sampling
# graph / seeds as in HOMO_CASES; `weights`: how the float32 edge weights are drawn (build_weights)
WEIGHTED_CASES: Dict[str, dict] = {
    # known-answer vector of test/csrc/sampler/test_neighbor.cpp:300-329 (cycle graph, only even edges have weight)
    'kat_cycle': dict(graph=('cycle', 6), seeds=[0, 1], num_neighbors=[1], rng_seed=0, weights='even_edges'),
    'rand_float': dict(graph=('rand', 2000, 20, 1), n_seeds=64, num_neighbors=[10, 5], rng_seed=11, weights='uniform'),
    'rand_float_rep': dict(graph=('rand', 2000, 20, 1), n_seeds=64, num_neighbors=[10, 5], rng_seed=12, weights='uniform', replace=True),
    # masked neighbours (weight 0 -> key -inf): fan-out > number of positive weights -> at::topk's tie order decides
    'masked': dict(graph=('rand', 1500, 16, 2), n_seeds=48, num_neighbors=[8, 4], rng_seed=13, weights='masked'),
    'masked_rep': dict(graph=('rand', 1500, 16, 2), n_seeds=48, num_neighbors=[8, 4], rng_seed=14, weights='masked_pos', replace=True),
    'ones': dict(graph=('rand', 2500, 24, 3), n_seeds=40, num_neighbors=[15, 10], rng_seed=15, weights='ones'),
    'quantized': dict(graph=('rand', 1200, 18, 4), n_seeds=40, num_neighbors=[6, 6], rng_seed=16, weights='quantized'),
    'three_hops_csc': dict(graph=('rand', 3000, 8, 5), n_seeds=16, num_neighbors=[4, 4, 4], rng_seed=17, weights='uniform', csc=True),
    # hubs: 70,000 neighbours -> std::partial_sort branch of at::topk (k * 64 <= n), long running sums under replacement
    'hub': dict(graph=('rand', 400, 10, 7, [(5, 70000), (77, 65540)]), seeds=[5, 77, 3, 9, 200], num_neighbors=[10, 5], rng_seed=18,
                weights='uniform'),
    'hub_masked': dict(graph=('rand', 400, 10, 7, [(5, 70000), (77, 65540)]), seeds=[5, 77, 3, 9, 200], num_neighbors=[12, 3], rng_seed=19,
                       weights='masked_heavy'),
    'hub_rep': dict(graph=('rand', 400, 10, 7, [(5, 70000), (77, 65540)]), seeds=[5, 77, 3, 9, 200], num_neighbors=[10, 5], rng_seed=20,
                    weights='uniform', replace=True),
    'zero_fanout_mix': dict(graph=('rand', 800, 12, 8), n_seeds=20, num_neighbors=[5, 0, 3], rng_seed=21, weights='uniform'),
    'dup_seeds': dict(graph=('rand', 600, 12, 9), seeds=[7, 7, 3, 7, 11, 3], num_neighbors=[4, 4], rng_seed=22, weights='uniform'),
    # disjoint subgraphs ((batch, node) keys) and "all neighbours" hops mixed with biased ones
    'disjoint': dict(graph=('rand', 1500, 14, 41), n_seeds=40, num_neighbors=[5, 4], rng_seed=23, weights='uniform', disjoint=True),
    'disjoint_masked_rep': dict(graph=('rand', 1500, 14, 41), n_seeds=40, num_neighbors=[5, 4], rng_seed=24, weights='masked_pos',
                                disjoint=True, replace=True),
    'full_then_k': dict(graph=('rand', 900, 6, 42), n_seeds=12, num_neighbors=[-1, 4], rng_seed=25, weights='masked'),
    'k_then_full_rep': dict(graph=('rand', 900, 6, 42), n_seeds=12, num_neighbors=[6, -1], rng_seed=26, weights='masked_pos', replace=True),
}
HETERO_WEIGHTED_CASES: Dict[str, dict] = {
    'kat_cycle': dict(kind='cycle', num_neighbors=[1], rng_seed=0, weights='even_edges', seeds=[0, 1]),   # test_neighbor.cpp:331-378
    'mag_w': dict(kind='mag', sizes=dict(paper=600, author=400, institution=20), avg_deg=6, n_seeds=dict(paper=16),
                  num_neighbors=[5, 3], rng_seed=31, gseed=31, weights='uniform'),
    'mag_w_rep': dict(kind='mag', sizes=dict(paper=600, author=400, institution=20), avg_deg=6, n_seeds=dict(paper=8, author=8),
                      num_neighbors=[4, 4], rng_seed=32, gseed=33, weights='uniform', replace=True),
    'mag_w_masked_csc': dict(kind='mag', sizes=dict(paper=600, author=400, institution=20), avg_deg=6, n_seeds=dict(paper=16),
                             num_neighbors=[6, 3], rng_seed=33, gseed=31, weights='masked', csc=True),
    'mag_w_disjoint': dict(kind='mag', sizes=dict(paper=600, author=400, institution=20), avg_deg=6, n_seeds=dict(paper=6, author=5),
                           num_neighbors=[4, 3], rng_seed=34, gseed=34, weights='uniform', disjoint=True),
    # weights for SOME relations (`weighted_rels`: indices into the edge type list): biased and uniform relations take turns on the
    # engine stream, the RandintEngine refills (one block = 512 16-bit draws) land between the biased relations' outputs
    'mag_mixed': dict(kind='mag', sizes=dict(paper=3000, author=2000, institution=40), avg_deg=30, n_seeds=dict(paper=8),
                      num_neighbors=[10, 6], rng_seed=35, gseed=32, weights='uniform', weighted_rels=[0, 1, 4]),
    'mag_mixed_rep': dict(kind='mag', sizes=dict(paper=3000, author=2000, institution=40), avg_deg=30, n_seeds=dict(paper=8, author=4),
                          num_neighbors=[8, 5], rng_seed=36, gseed=32, weights='masked_pos', weighted_rels=[1, 3], replace=True),
    'mag_mixed_disjoint_masked': dict(kind='mag', sizes=dict(paper=600, author=400, institution=20), avg_deg=6, n_seeds=dict(paper=6, author=5),
                                      num_neighbors=[4, 3, 2], rng_seed=37, gseed=34, weights='masked', weighted_rels=[2, 3, 5], disjoint=True),
    'mag_mixed_csc_one': dict(kind='mag', sizes=dict(paper=3000, author=2000, institution=40), avg_deg=30, n_seeds=dict(paper=16),
                              num_neighbors=[12, 4], rng_seed=38, gseed=32, weights='uniform', weighted_rels=[5], csc=True),
}


def build_weights(kind: str, rowptr: torch.Tensor, seed: int) -> torch.Tensor:
    E = int(rowptr[-1])
    g = torch.Generator().manual_seed(77000 + seed)
    if kind == 'even_edges':
        return torch.stack([torch.ones(E // 2), torch.zeros(E // 2)], -1).view(-1)
    if kind == 'uniform':
        return torch.rand(E, generator=g)
    if kind == 'ones':
        return torch.ones(E)
    if kind == 'quantized':
        return torch.randint(0, 3, (E,), generator=g).float()
    if kind in ('masked', 'masked_heavy', 'masked_pos'):
        w = torch.rand(E, generator=g) * (torch.rand(E, generator=g) < (0.03 if kind == 'masked_heavy' else 0.4))
        if kind == 'masked_pos':   # at::multinomial wants a positive sum in every sampled row
            first = rowptr[:-1][rowptr[:-1] < rowptr[1:]]
            w[first] += 0.25
        return w
    raise ValueError(kind)


def build_weighted(case: dict):
    rowptr, col, seed = build_homo(case)
    return rowptr, col, seed, build_weights(case['weights'], rowptr, case['rng_seed'])


def build_hetero_weighted(case: dict):
    node_types, edge_types, rowptr_d, col_d, seed_d, nn_d = build_hetero(case)
    if 'seeds' in case:
        seed_d = {'paper': torch.tensor(case['seeds'])}
    w_d = {k: build_weights(case['weights'], rowptr_d[k], case['rng_seed'] + i) for i, k in enumerate(rowptr_d)
           if 'weighted_rels' not in case or i in case['weighted_rels']}
    return node_types, edge_types, rowptr_d, col_d, seed_d, nn_d, w_d
