"""The batched inverse entry points refuse a null context / pipeline with BWTC_CUDA_EARG and a message in
bwtc_cuda_global_error(), as the other entry points do.  No device needed: the handle is checked before any CUDA call."""
import ctypes

import numpy as np

import bwtc_b200 as bw

EARG = -1


def test_inverse_blocks_null_context():
    lib = bw.load_library()
    blk = np.zeros(16, np.uint8)
    ptrs = (ctypes.c_void_p * 1)(blk.ctypes.data)
    sizes = np.array([16], np.uint32)
    LF = np.zeros(256, np.uint32)
    assert lib.bwtc_cuda_inverse_blocks(None, ptrs, None, sizes.ctypes.data, 1, 0, LF.ctypes.data, None) == EARG
    assert b"null context" in lib.bwtc_cuda_global_error()


def test_pipeline_submit_inverse_null_pipeline():
    lib = bw.load_library()
    blk = np.zeros(16, np.uint8)
    ticket = ctypes.c_uint64(0)
    assert lib.bwtc_cuda_pipeline_submit_inverse(None, blk.ctypes.data, blk.ctypes.data, 16, 0, 0, None,
                                                 ctypes.byref(ticket)) == EARG
    assert b"null pipeline" in lib.bwtc_cuda_global_error()
