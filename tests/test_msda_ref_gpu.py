"""tair_msda_forward against the reference's OWN CUDA kernel (ms_deformable_im2col_gpu_kernel,
testr/adet/layers/csrc/DeformAttn/ms_deform_im2col_cuda.cuh:237-299).  The kernel's outputs on the seeded inputs of
oracle.msda.ref_kernel_case are stored, a fixed sample of rows per case, in tests/golden/msda_ref_cases.npz
(make_golden.py msda_ref).  Where the kernel has been compiled unmodified from the reference tree into
oracle/_ref/libmsda_ref.so (oracle/build_ref.sh), the whole output is also compared live."""
import ctypes as C
import os

import pytest
import torch

pytestmark = pytest.mark.gpu
REF = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "libmsda_ref.so")


@pytest.mark.parametrize("B,Lq,shapes", [(2, 300, [(16, 16), (32, 32), (64, 64), (64, 64)]), (3, 77, [(8, 8), (4, 6), (3, 3)]),
                                         (1, 9472, [(16, 16), (32, 32), (64, 64), (64, 64)])])
def test_drop_in_forward_equals_reference_cuda_kernel(cuda_lib, golden, B, Lq, shapes):
    from oracle.msda import ref_kernel_case
    from tair_b200 import ops
    M, D, P = 8, 32, 4
    value, shp, start, loc, w = ref_kernel_case(B, Lq, shapes, M, D, P)
    out = ops.msda_forward(value, shp, start, loc, w)
    assert out.shape == (B, Lq, M * D)
    g = golden("msda_ref_cases.npz")
    key = f"B{B}_Lq{Lq}_L{len(shapes)}"
    rows = torch.from_numpy(g[key + "_rows"]).cuda()
    assert (out.reshape(B * Lq, -1)[rows].cpu() - torch.from_numpy(g[key + "_out"])).abs().max().item() <= 1e-5
    if os.path.exists(REF):
        ref = torch.empty(B, Lq, M * D, device="cuda")
        rc = C.CDLL(REF).msda_ref_forward_f32(*(C.c_void_p(t.data_ptr()) for t in (value, shp, start, loc, w, ref)),
                                              B, value.shape[1], M, D, len(shapes), Lq, P,
                                              C.c_void_p(torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        assert rc == 0 and (out - ref).abs().max().item() <= 1e-5
