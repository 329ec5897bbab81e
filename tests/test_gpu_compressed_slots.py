"""Witness slots are compressible device memory (cuMemCreate with generic compression) where the device supports it: every slot
of a main-shape handle is granted compression, teardown gives all of it back, and every read path sees the same bytes."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SHAPE = (16, 4, 16, 50, 31, 2, 10 ** 19, 10 ** 20)
CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED = 107
CU_MEM_ALLOCATION_COMP_GENERIC = 1


class CUmemLocation(ctypes.Structure):
    _fields_ = [("type", ctypes.c_int), ("id", ctypes.c_int)]


class CUmemAllocFlags(ctypes.Structure):
    _fields_ = [("compressionType", ctypes.c_ubyte), ("gpuDirectRDMACapable", ctypes.c_ubyte), ("usage", ctypes.c_ushort), ("reserved", ctypes.c_ubyte * 4)]


class CUmemAllocationProp(ctypes.Structure):
    _fields_ = [("type", ctypes.c_int), ("requestedHandleTypes", ctypes.c_int), ("location", CUmemLocation),
                ("win32HandleMetaData", ctypes.c_void_p), ("allocFlags", CUmemAllocFlags)]


def _cuda_driver():
    cu = ctypes.CDLL("libcuda.so.1")
    assert cu.cuInit(0) == 0
    return cu


def _compression_supported(cu, device=0):
    dev, v = ctypes.c_int(), ctypes.c_int()
    assert cu.cuDeviceGet(ctypes.byref(dev), device) == 0
    assert cu.cuDeviceGetAttribute(ctypes.byref(v), CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, dev) == 0
    return v.value != 0


def _compression_type(cu, dptr):
    h = ctypes.c_ulonglong()
    assert cu.cuMemRetainAllocationHandle(ctypes.byref(h), ctypes.c_void_p(dptr)) == 0, "not a cuMemCreate allocation"
    try:
        prop = CUmemAllocationProp()
        assert cu.cuMemGetAllocationPropertiesFromHandle(ctypes.byref(prop), h) == 0
        return prop.allocFlags.compressionType
    finally:
        assert cu.cuMemRelease(h) == 0


def _mem_free(cu):
    free, total = ctypes.c_size_t(), ctypes.c_size_t()
    assert cu.cuMemGetInfo_v2(ctypes.byref(free), ctypes.byref(total)) == 0
    return free.value


def test_every_slot_of_a_main_shape_handle_is_compressible():
    import pob_b200
    from pob_b200 import synth
    cu = _cuda_driver()
    if not _compression_supported(cu):
        pytest.skip("the device does not support generic compression: slots are plain")
    c = pob_b200.Circuit(pob_b200.MAIN_PROOF_OF_BURN)
    try:
        n = c.desc["n_slots"]
        res = c.run_packed(synth.pack_instances(synth.make_batch(n, SHAPE, seed=31), SHAPE))
        assert (res.status == 0).all()
        ptrs = {c.witness_device_ptr(i) for i in range(n)}
        assert len(ptrs) == n
        assert all(_compression_type(cu, p) == CU_MEM_ALLOCATION_COMP_GENERIC for p in ptrs)
    finally:
        c.close()


def test_create_and_destroy_give_all_device_memory_back():
    """a leaked slot allocation would pin 6.9 GB (all of them: ~145 GB)"""
    import pob_b200
    cu = _cuda_driver()
    pob_b200.Circuit(pob_b200.MAIN_PROOF_OF_BURN).close()      # first use loads the modules
    before = _mem_free(cu)
    for _ in range(3):
        c = pob_b200.Circuit(pob_b200.MAIN_PROOF_OF_BURN)
        assert c.desc["n_slots"] >= 2
        c.close()
    assert abs(_mem_free(cu) - before) < (64 << 20)


def test_kernel_copy_engine_and_oracle_read_the_same_witness():
    """k_digest on the SMs, a D2H copy through the copy engine, and the oracle's own witness agree on one main-shape witness"""
    import pob_b200
    from pob_b200 import synth
    from oracle import oracle
    insts = synth.make_batch(1, SHAPE, seed=17)
    c = pob_b200.Circuit(pob_b200.MAIN_PROOF_OF_BURN, max_slots=2)
    try:
        res = c.run_packed(synth.pack_instances(insts, SHAPE), digest=True)
        assert res.status[0] == 0
        host = c.witness(0)
        host_digest = int(oracle.lib().pob_oracle_digest(host.ctypes.data, host.shape[0]))
        w = oracle.run(pob_b200.MAIN_PROOF_OF_BURN, synth.to_json(insts[0], SHAPE))
        try:
            assert w.ok
            assert int(res.digests[0]) == host_digest == w.digest()
            assert np.array_equal(host, w.limbs)
        finally:
            w.free()
    finally:
        c.close()
