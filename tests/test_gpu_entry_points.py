"""The four ways into the compressor walk a region batch by batch under the same rules: the region call
(phy_compress_region), the streamed call (phy_compress_region_streamed, the caller fills the region behind a `wait`
callback), the stream call (phy_compress_stream, the library pulls the region through `read` and hands each batch to
`emit`) and the resident legs (phy_upload, phy_compress_resident, phy_download).  On the same input they must return the
same subblocks: descriptors, payloads, working-region overlap, batches and launches."""
import ctypes as C

import numpy as np
import pytest

from phyngsc_b200 import api, synth

pytestmark = pytest.mark.gpu

WAIT = C.CFUNCTYPE(None, C.c_void_p, C.c_uint64)
READ = C.CFUNCTYPE(C.c_int64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64)
EMIT = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(api.SubblockDesc), C.c_uint32, C.c_void_p)
DESC_FIELDS = ("win_off", "win_len", "rec_start", "overlap", "n_records", "warnings", "bytes_consumed", "sec_len", "out_len", "status")


def _newline_free_tail(data):
    assert data[-1] == 10
    return data[:-1]


CASES = {  # name: (data, np, rank, window_bytes, max_batch_bytes, max_subblocks)
    "multi_batch_rank0": (lambda: synth.fastq("100bp", 51, target_bytes=6_000_000), 1, 0, 256 * 1024, 1 << 20, 64),
    "rank1_of_2_no_final_newline": (lambda: _newline_free_tail(synth.fastq("36bp", 52, target_bytes=6_000_000)), 2, 1, 256 * 1024, 1 << 20, 64),
    "capacity_stop": (lambda: synth.fastq("100bp", 49, target_bytes=3_000_000), 1, 0, 64 * 1024, 1 << 20, 5),
}


def region_call(ctx, region, prm):
    descs, out, res = ctx.compress_region(region, prm)
    return descs, api.payloads(descs, out), res


def streamed_call(ctx, region, prm, uptos):
    L = api.lib()
    L.phy_compress_region_streamed.restype = C.c_int
    L.phy_compress_region_streamed.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(api.RegionParams), WAIT, C.c_void_p,
                                               C.c_void_p, C.c_uint64, C.POINTER(api.SubblockDesc), C.POINTER(C.c_uint32),
                                               C.POINTER(api.RegionResult)]
    wait = WAIT(lambda user, upto: uptos.append(upto))
    out = np.empty(region.size // 2 + (1 << 20), np.uint8)
    descs = (api.SubblockDesc * 4096)()
    n = C.c_uint32(4096)
    res = api.RegionResult()
    rc = L.phy_compress_region_streamed(ctx._h, region.ctypes.data, region.size, C.byref(prm), wait, None, out.ctypes.data, out.size,
                                        descs, C.byref(n), C.byref(res))
    if rc:
        raise ctx._err(rc)
    descs = list(descs[: n.value])
    return descs, api.payloads(descs, out), res


def stream_call(ctx, region, prm):
    L = api.lib()
    L.phy_compress_stream.restype = C.c_int
    L.phy_compress_stream.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(api.RegionParams), READ, C.c_void_p, EMIT, C.c_void_p,
                                      C.POINTER(api.RegionResult)]
    descs, payloads, batches = [], [], []

    def read(user, off, dst, n):  # called from the library's reader threads
        C.memmove(dst, region.ctypes.data + off, n)
        return n

    def emit(user, d, n, base):  # called from the library's emitter thread, one batch at a time, in order
        try:
            batch = [api.SubblockDesc.from_buffer_copy(d[i]) for i in range(n)]
            descs.extend(batch)
            payloads.extend(C.string_at(base + x.out_off, x.out_len) for x in batch)
            batches.append(n)
            return 0
        except Exception:  # noqa: BLE001  (an exception must not cross the C boundary: stop the call instead)
            return 1

    read_cb, emit_cb = READ(read), EMIT(emit)
    res = api.RegionResult()
    rc = L.phy_compress_stream(ctx._h, region.size, C.byref(prm), read_cb, None, emit_cb, None, C.byref(res))
    if rc:
        raise ctx._err(rc)
    assert len(batches) == res.n_batches
    return descs, payloads, res


def resident_legs(ctx, region, prm):
    ctx.upload(region)
    descs, res = ctx.compress_resident(region.size, prm)
    out = np.empty(res.out_used, np.uint8)
    assert ctx.download(out) == res.out_used
    return descs, api.payloads(descs, out), res


def fields(descs):
    return [tuple(list(getattr(d, f)) if f == "sec_len" else getattr(d, f) for f in DESC_FIELDS) for d in descs]


@pytest.mark.parametrize("name", list(CASES))
def test_every_entry_point_returns_the_same_subblocks(name):
    make, npr, rank, win, max_batch, max_sb = CASES[name]
    data = make()
    start, _ = api.region_slice(data.size, npr, rank)
    region = np.ascontiguousarray(data[start:])
    prm = api.region_params(data.size, npr, rank, window_bytes=win)
    uptos = []
    calls = {"region": lambda c: region_call(c, region, prm), "streamed": lambda c: streamed_call(c, region, prm, uptos),
             "stream": lambda c: stream_call(c, region, prm), "resident": lambda c: resident_legs(c, region, prm)}
    got = {}
    for k, call in calls.items():  # a context of its own per entry point: no hint of an earlier call carries over
        ctx = api.Context(0, max_batch_bytes=max_batch, max_subblocks=max_sb)
        try:
            got[k] = call(ctx)
        finally:
            ctx.close()
    d0, p0, r0 = got["region"]
    assert r0.n_batches > 2 and len(d0) > 5 and all(d.status == 0 for d in d0)
    assert sum(d.bytes_consumed for d in d0) == r0.bytes_in
    for k, (d, p, r) in got.items():
        assert fields(d) == fields(d0), k
        assert p == p0, k
        assert r.wr_overlap == r0.wr_overlap, k
        assert (r.n_batches, r.kernel_launches, r.n_subblocks, r.bytes_in, r.bytes_out) == \
            (r0.n_batches, r0.kernel_launches, r0.n_subblocks, r0.bytes_in, r0.bytes_out), k
    assert uptos and all(a <= b for a, b in zip(uptos, uptos[1:])) and uptos[-1] == region.size
    if rank:
        assert r0.wr_overlap > 0 and d0[0].rec_start == r0.wr_overlap
