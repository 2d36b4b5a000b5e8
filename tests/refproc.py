"""Run the reference (oracle/ref_parity.py, a subprocess: oracle/_ref/libpyg_ref.so and libpyg.so both register the
pyg:: schemas) on inputs that may be too large to pickle: big tensors go through raw files under /dev/shm (or the
temp dir) that the child maps with torch.from_file.  Used by bench.py's parity gate; the comparison helpers below also
serve tests/test_config_parity.py, which compares with stored outputs of the reference instead."""
import hashlib
import os
import os.path as osp
import shutil
import subprocess
import sys
import tempfile

import torch

ROOT = osp.dirname(osp.dirname(osp.abspath(__file__)))
_NAMES = {torch.int64: 'int64', torch.int32: 'int32', torch.bfloat16: 'bfloat16', torch.float16: 'float16',
          torch.float32: 'float32'}


class RefSession:
    """Scratch directory for one exchange with the reference process; removes itself."""
    def __init__(self):
        base = '/dev/shm' if osp.isdir('/dev/shm') and os.access('/dev/shm', os.W_OK) else None
        self.dir = tempfile.mkdtemp(prefix='pygb200_ref_', dir=base)
        self.n = 0

    def __enter__(self):
        return self

    def __exit__(self, *a):
        shutil.rmtree(self.dir, ignore_errors=True)

    def share(self, t: torch.Tensor, small_bytes: int = 1 << 20):
        """Tensor (any device) -> spec entry.  Small tensors travel inside the spec, big ones as raw files."""
        t = t.detach()
        if t.numel() * t.element_size() <= small_bytes:
            return t.cpu().contiguous()
        self.n += 1
        path = osp.join(self.dir, f'in{self.n}.bin')
        f = torch.from_file(path, shared=True, size=t.numel(), dtype=t.dtype)
        f.copy_(t.reshape(-1))      # device -> mapped file directly when t is a CUDA tensor
        del f
        return {'path': path, 'dtype': _NAMES[t.dtype], 'numel': t.numel(), 'shape': list(t.shape)}

    def out_file(self, numel: int, dtype: torch.dtype):
        self.n += 1
        return osp.join(self.dir, f'out{self.n}.bin')

    def run(self, spec: dict, timeout: int = 1800) -> dict:
        spec = dict(spec)
        spec['out'] = osp.join(self.dir, 'result.pt')
        spec_path = osp.join(self.dir, 'spec.pt')
        torch.save(spec, spec_path)
        env = dict(os.environ)
        p = subprocess.run([sys.executable, osp.join(ROOT, 'oracle', 'ref_parity.py'), spec_path], stdout=subprocess.PIPE,
                           stderr=subprocess.PIPE, text=True, timeout=timeout, env=env, cwd=ROOT)
        if p.returncode != 0 or 'REFPARITY_OK' not in p.stdout:
            raise RuntimeError('reference process failed:\n' + p.stdout[-2000:] + '\n' + p.stderr[-4000:])
        return torch.load(spec['out'], weights_only=False)


def compare_homo(out, ref_call) -> dict:
    """Our (row, col, node, eid, nph, eph) vs one call of the reference: bit-exact or a description of the mismatch."""
    bad = []
    for k, t in zip(('row', 'col', 'node', 'eid'), out[:4]):
        r = ref_call[k]
        if (t is None) != (r is None):
            bad.append(k + ': presence')
        elif t is not None and not torch.equal(t.cpu(), r):
            bad.append(f'{k}: {tuple(t.shape)} vs {tuple(r.shape)}')
    if list(out[4]) != list(ref_call['nph']):
        bad.append('nodes_per_hop')
    if list(out[5]) != list(ref_call['eph']):
        bad.append('edges_per_hop')
    return {'bit_exact': not bad, 'mismatch': bad, 'edges': int(out[0].numel()), 'nodes': int(out[2].shape[0])}


def rng_prefix():
    return torch.get_rng_state()[:24 + 624 * 8].clone()


def sha256(t: torch.Tensor) -> bytes:
    """SHA-256 of a tensor's elements in row-major order: how the config-size fixtures keep index tensors that are too
    large to store (equal digests of same-shape, same-dtype tensors = bit-exact)."""
    return hashlib.sha256(t.detach().cpu().contiguous().numpy().tobytes()).digest()


def accumulation_bound(x: torch.Tensor, ptr: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
    """Rigorous bound on how far two fp32-accumulated K-term dot products of the same inputs can be apart because of
    their summation ORDER (Higham, gamma_K): 2 K 2^-24 sum_k |x_ik| |w_kj|, per output element [N, M] (fp32, on x's
    device).  It only matters for results that cancel to almost zero, where an error in ulps of the RESULT says nothing."""
    K = x.size(1)
    out = torch.empty(x.size(0), w.size(2), dtype=torch.float32, device=x.device)
    p = ptr.tolist()
    for b in range(len(p) - 1):
        if p[b + 1] > p[b]:
            out[p[b]:p[b + 1]] = x[p[b]:p[b + 1]].float().abs() @ w[b].float().abs()
    return out * (2.0 * K * 2.0 ** -24)


def lowp_ulp_excess(out: torch.Tensor, ref: torch.Tensor, abs_tol=None) -> float:
    """max (|out - ref| - abs_tol) in units of one storage ulp of the reference value: ulp(v) = 2^-7 |v| for bf16,
    2^-10 |v| for fp16 (an upper bound of the true spacing, within 2x).  `abs_tol` (tensor like out, or None) is the
    fp32 accumulation-order allowance of `accumulation_bound`.  SURVEY.md 8(c): parity holds when the result is <= 1."""
    rel = 2.0 ** -7 if out.dtype == torch.bfloat16 else 2.0 ** -10
    worst = 0.0
    step = 1 << 16
    for i in range(0, out.size(0), step):   # chunked: full-size outputs are 134 M elements
        oc, rc = out[i:i + step].float(), ref[i:i + step].float()
        if not oc.numel():
            continue
        d = (oc - rc).abs()
        if abs_tol is not None:
            d = (d - abs_tol[i:i + step].to(d.device)).clamp_min(0)
        worst = max(worst, float((d / (rel * rc.abs().clamp_min(1e-30))).max()))
    return worst
