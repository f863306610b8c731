"""The relatedness accumulator without a GPU: vcfx_cuda_king_create fails with VCFX_E_NO_DEVICE instead of falling back,
and api.King raises it."""
import ctypes as C

import pytest


def test_king_create_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from vcfx_b200 import api, build
    build.build_cuda()
    lib = C.CDLL(str(api.lib_path()))
    h = C.c_void_p()
    lib.vcfx_cuda_king_create.argtypes = [C.c_int, C.c_uint32, C.c_void_p, C.POINTER(C.c_void_p)]
    assert lib.vcfx_cuda_king_create(0, 10, None, C.byref(h)) == -2 and not h
    with pytest.raises(api.VcfxCudaError) as e:
        api.King(10, stream=0)
    assert e.value.code == -2
    with pytest.raises(api.VcfxCudaError):
        api.king(b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\ta\tb\n1\t1\t.\tA\tG\t.\t.\t.\tGT\t0/1\t1/1\n")
