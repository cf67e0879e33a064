"""Run in a subprocess by tests/test_gpu_selfloop_gemm.py: the persistent self-loop kernel (engine 1, N = K = 200) against
fp64 and against the packed tcgen05 kernel it replaces (engine 2), which computes the same products in the same order."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from renet_b200 import _lib  # noqa: E402

L = _lib.lib()
dev = 'cuda:0'
H = 200


def selfloop(A, idx, W, M):
    # one spare row after the M output rows: it must stay untouched
    out = torch.full((M + 1, H), float('nan'), device=dev)
    _lib.check(L.renet_selfloop_gemm(_lib.ptr(A), _lib.ptr(idx), _lib.ptr(W), _lib.ptr(out), M, H, H, _lib.stream()),
               'renet_selfloop_gemm')
    torch.cuda.synchronize()
    assert torch.isnan(out[M]).all(), 'row M was written'
    return out[:M]


def run(A, idx, W, M, what):
    ref = (A[idx.long()] if idx is not None else A[:M]).double() @ W.double()
    L.renet_set_gemm_engine(2)
    old = selfloop(A, idx, W, M)
    L.renet_set_gemm_engine(1)
    new = selfloop(A, idx, W, M)
    assert not torch.isnan(new).any(), '%s: outputs left unwritten' % what
    err = (new.double() - ref).abs().max().item() / ref.abs().max().item()
    same = torch.equal(new, old)
    print('%-40s rel err vs fp64 %.2e  bit-identical to engine 2: %s' % (what, err, same))
    assert err <= 1e-4, (what, err)
    assert same, '%s: max |new - old| = %.3e' % (what, (new - old).abs().max().item())
    return err


torch.manual_seed(0)
worst = 0.0
table = torch.randn(23033, H, device=dev) * 0.3
W = torch.randn(H, H, device=dev) * 0.1
for M in (64, 127, 128, 129, 255, 257, 8573, 34483, 37889, 100000):
    idx = torch.randint(0, table.shape[0], (M,), device=dev, dtype=torch.int32)       # repeated ids
    worst = max(worst, run(table, idx, W, M, 'M=%d indexed' % M))
    A = torch.randn(M, H, device=dev) * 0.3
    worst = max(worst, run(A, None, W, M, 'M=%d dense' % M))

# weight generations: the packed image is reused while the generation holds and rebuilt when it changes
M = 8573
idx = torch.randint(0, table.shape[0], (M,), device=dev, dtype=torch.int32)
L.renet_set_weight_generation(1)
worst = max(worst, run(table, idx, W, M, 'generation 1'))
W.mul_(-0.5).add_(0.01)                  # same buffer, new values
L.renet_set_weight_generation(2)
worst = max(worst, run(table, idx, W, M, 'generation 2 (weights changed in place)'))
L.renet_set_weight_generation(-1)
assert L.renet_get_gemm_engine() == 1
print('SELFLOOP_OK worst %.2e' % worst)
