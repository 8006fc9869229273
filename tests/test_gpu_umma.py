"""GPU: the tcgen05/TMA building blocks (on-device self test) and size-independent properties of the tensor-core
attention at BASELINE sizes (Lmax up to 8192), where the CPU oracle is too slow to be the checker."""
import ctypes as C

import pytest
import torch

from util import assert_rel, offsets_from

pytestmark = pytest.mark.gpu


def test_umma_selftest_report():
    from generative_recommenders_b200 import _lib

    buf = C.create_string_buffer(1 << 16)
    fails = _lib.selftest_lib().hstu_umma_selftest(buf, len(buf))
    report = buf.value.decode()
    print(report)
    assert fails == 0, report


def _inputs(B, H, d, lmax, seed, dtype=torch.bfloat16, scale=0.5):
    from generative_recommenders_b200.common import generate_sparse_seq_len

    dev = torch.device("cuda")
    torch.manual_seed(seed)
    lengths = generate_sparse_seq_len(B, lmax, 0.95, dev)
    nt = torch.clamp(torch.randint(1, 21, (B,), device=dev, dtype=torch.int32), max=lengths)
    off = torch.zeros(B + 1, dtype=torch.int64, device=dev)
    off[1:] = torch.cumsum(lengths, 0)
    L = int(off[-1])
    x = torch.empty(L, H, 3 * d, device=dev, dtype=dtype).uniform_(-scale, scale)
    q, k, v = torch.split(x, [d, d, d], dim=-1)
    return q, k, v, off, nt


@pytest.mark.parametrize("d,lmax,B,H", [(32, 8192, 2, 8), (64, 2048, 4, 4), (128, 4096, 2, 2), (128, 512, 16, 4)])
def test_umma_matches_generic_at_full_size(d, lmax, B, H):
    """Two independent implementations (tcgen05 vs CUDA-core fp32) agree at sizes the CPU oracle cannot reach."""
    from generative_recommenders_b200 import _lib
    from generative_recommenders_b200.common import HammerKernel
    from generative_recommenders_b200.ops.hstu_attention import hstu_mha

    q, k, v, off, nt = _inputs(B, H, d, lmax, 3)
    alpha = 1.0 / d**0.5
    o_ref = hstu_mha(lmax, alpha, q.float(), k.float(), v.float(), off, num_targets=nt, kernel=HammerKernel.CUDA,
                     impl=_lib.IMPL_GENERIC)
    o = hstu_mha(lmax, alpha, q, k, v, off, num_targets=nt, kernel=HammerKernel.CUDA, impl=_lib.IMPL_UMMA)
    assert_rel(o, o_ref, f"umma vs generic d={d} lmax={lmax}")
    # backward: tcgen05 (where supported) vs the CUDA-core kernels on the same bf16 inputs
    do = torch.randn_like(o)
    grads = {}
    for impl in (_lib.IMPL_GENERIC, _lib.IMPL_AUTO):
        qq, kk, vv = (t.detach().clone().requires_grad_() for t in (q, k, v))
        hstu_mha(lmax, alpha, qq, kk, vv, off, num_targets=nt, kernel=HammerKernel.CUDA, impl=impl).backward(do)
        grads[impl] = (qq.grad, kk.grad, vv.grad)
    for name, a, r in zip(("dq", "dk", "dv"), grads[_lib.IMPL_AUTO], grads[_lib.IMPL_GENERIC]):
        # both sides are bf16: the reference side of this self-comparison carries its own 1.7e-3 storage rounding
        assert_rel(a, r.float(), f"bwd umma vs generic {name} d={d} lmax={lmax}", tol=2.0e-3)


def test_linearity_in_v_and_sequence_permutation():
    """O is linear in V for fixed Q,K; and permuting whole sequences of the batch permutes the output rows."""
    from generative_recommenders_b200 import _lib
    from generative_recommenders_b200.common import HammerKernel
    from generative_recommenders_b200.ops.hstu_attention import hstu_mha

    d, lmax, B, H = 64, 2048, 6, 2
    q, k, v, off, nt = _inputs(B, H, d, lmax, 9)
    v2 = torch.empty_like(v).uniform_(-0.5, 0.5)
    f = lambda vv: hstu_mha(lmax, 0.125, q, k, vv, off, num_targets=nt, kernel=HammerKernel.CUDA, impl=_lib.IMPL_UMMA).float()  # noqa: E731
    o1, o2, o12 = f(v), f(v2), f((v.float() + v2.float()).to(v.dtype))
    assert_rel((o1 + o2).to(torch.bfloat16), o12, "linearity in V", tol=6e-3)  # three bf16 roundings of V / O
    # permute sequences
    lens = (off[1:] - off[:-1]).tolist()
    order = [3, 0, 5, 1, 4, 2]
    rows = torch.cat([torch.arange(int(off[i]), int(off[i + 1]), device=q.device) for i in order])
    off2 = offsets_from([lens[i] for i in order], q.device)
    o_perm = hstu_mha(lmax, 0.125, q[rows], k[rows], v[rows], off2, num_targets=nt[order], kernel=HammerKernel.CUDA,
                      impl=_lib.IMPL_UMMA)
    assert torch.equal(o_perm.float(), o1[rows])
