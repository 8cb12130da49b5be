"""tcgen05 on a CTA pair: the 2-SM MMA (M = 256, each CTA holding half of B) against a torch matmul."""
import ctypes

import pytest
import torch

from mentflow_b200 import _lib

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("mode,k", [(0, 16), (1, 64)])
def test_umma_pair_half_b_tiles(mode, k):
    """cluster of 2, cta_group::2 alloc / MMA / multicast commit, remote request arrive; SWIZZLE_32B (mode 0) and
    SWIZZLE_128B (mode 1) tiles.  fp16-representable inputs with exact fp32 sums: the result is exact."""
    lib = _lib.load()
    torch.manual_seed(7 + mode)
    a = (torch.randint(-8, 9, (256, k)).float() / 8).cuda()
    b = (torch.randint(-8, 9, (64, k)).float() / 4).cuda()
    d = torch.full((256, 64), float("nan"), device="cuda")
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = lib.mfb_selftest_umma_pair(a.data_ptr(), b.data_ptr(), mode, d.data_ptr(), err.data_ptr(), st)
    assert rc == 0
    torch.cuda.synchronize()
    assert int(err.item()) == 0
    assert torch.equal(d, a @ b.T)
