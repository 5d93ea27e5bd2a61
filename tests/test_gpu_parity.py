"""Parity of the CUDA path (through the C ABI) against the oracle and the reference-minted goldens."""
import json
import os

import numpy as np
import pytest

import gpu_cases
from phyngsc_b200 import api, container, synth

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def ctx(oracle):
    c = api.Context(0, max_batch_bytes=64 << 20, max_subblocks=256)
    yield c
    c.close()


@pytest.mark.parametrize("case", gpu_cases.CASES, ids=[c[0] for c in gpu_cases.CASES])
def test_payloads_bit_exact_against_oracle(case, ctx):
    probs = gpu_cases.run_case(ctx, case)
    assert not probs, "\n".join(probs[:20])


@pytest.mark.parametrize("case", json.load(open(os.path.join(GOLD, "manifest.json"))), ids=lambda c: c["file"])
def test_payloads_bit_exact_against_reference_goldens(case, ctx):
    data = synth.fastq(case["shape"], case["seed"], target_bytes=case["target_bytes"])
    ng = container.read_ngsc(os.path.join(GOLD, case["file"]))
    for r in range(case["np"]):
        start, _ = api.region_slice(data.size, case["np"], r)
        descs, out, res = ctx.compress_region(data[start:], api.region_params(data.size, case["np"], r))
        assert api.payloads(descs, out) == ng["per_rank_subblocks"][r]
        assert res.wr_overlap == ng["footer"]["overlaps"][r]


def test_multi_batch_equals_single_batch(oracle):
    """One batch of 24 subblocks against many small batches and against the oracle."""
    data = synth.fastq("100bp", 41, target_bytes=6_000_000)
    win = 256 * 1024
    prm = api.region_params(data.size, 1, 0, window_bytes=win)
    big = api.Context(0, max_batch_bytes=32 << 20, max_subblocks=64)
    small = api.Context(0, max_batch_bytes=1 << 20, max_subblocks=64)
    try:
        d1, o1, r1 = big.compress_region(data, prm)
        d2, o2, r2 = small.compress_region(data, prm)
        assert r1.n_batches == 1 and r2.n_batches > 2 and len(d1) >= 16
        assert api.payloads(d1, o1) == api.payloads(d2, o2)
        assert [(d.win_off, d.win_len, d.n_records) for d in d1] == [(d.win_off, d.win_len, d.n_records) for d in d2]
        assert api.payloads(d1, o1) == oracle.compress_rank(data, 1, 0, window_bytes=win)["subblocks"]
    finally:
        big.close(); small.close()


def test_groups_of_a_large_batch_equal_one_group_batches(ctx):
    """A 200 MB batch runs as three groups (own streams, record table and window plan of the later groups overlapping
    the statistics of the earlier ones); the same data through 64 MiB batches runs one group per batch.  Same windows,
    same payloads, payloads of all groups back to back, and every payload decodes to its input."""
    data = synth.fastq("100bp", 47, target_bytes=200_000_000)
    prm = api.region_params(data.size, 1, 0)
    big = api.Context(0, max_batch_bytes=256 << 20, max_subblocks=64)
    try:
        d1, o1, r1 = big.compress_region(data, prm)
        d2, o2, r2 = ctx.compress_region(data, prm)
        assert r1.n_batches == 1 and r2.n_batches > 2
        assert r1.kernel_launches > 2 + 3 * 3 + 12 * 2  # more than two groups' worth of launches
        assert [(d.win_off, d.win_len, d.n_records, d.bytes_consumed) for d in d1] == [(d.win_off, d.win_len, d.n_records, d.bytes_consumed) for d in d2]
        assert api.payloads(d1, o1) == api.payloads(d2, o2)
        assert all(a.out_off + ((a.out_len + 15) & ~15) == b.out_off for a, b in zip(d1, d1[1:]))
        for x in d1[::5]:
            dec = api.decode_subblock(o1[x.out_off:x.out_off + x.out_len], x.bytes_consumed + 4096)
            assert np.array_equal(dec, data[x.win_off:x.win_off + x.bytes_consumed])
    finally:
        big.close()


def test_resident_legs_match_region_call(ctx):
    data = synth.fastq("36bp", 42, target_bytes=3_000_000)
    prm = api.region_params(data.size, 1, 0, window_bytes=1 << 20)
    d1, o1, _ = ctx.compress_region(data, prm)
    ctx.upload(data)
    d2, res = ctx.compress_resident(data.size, prm)
    o2 = np.empty(res.out_used, np.uint8)
    assert ctx.download(o2) == res.out_used
    assert api.payloads(d1, o1) == api.payloads(d2, o2)
    assert res.kernel_launches >= 10 and res.kernel_ms > 0


def test_malformed_inputs_are_errors(ctx):
    good = synth.fastq("36bp", 43, target_bytes=200_000)
    prm = lambda a: api.region_params(a.size, 1, 0)  # noqa: E731
    # line 3 is not '+'
    bad = good.copy()
    plus = good.tobytes().find(b"\n+\n", 5000) + 1  # a real line 3 ('+' is also a quality character)
    bad[plus] = ord("-")
    with pytest.raises(api.PhyError) as e:
        ctx.compress_region(bad, prm(bad))
    assert e.value.code == -1
    # a title with one separator more than record 0
    txt = good.tobytes().split(b"\n")
    txt[4 * 7] = txt[4 * 7].replace(b"/2", b"/2/3")
    bad = np.frombuffer(b"\n".join(txt), np.uint8)
    with pytest.raises(api.PhyError) as e:
        ctx.compress_region(bad, prm(bad))
    assert e.value.code == -2
    # quality shorter than the sequence
    txt = good.tobytes().split(b"\n")
    txt[4 * 3 + 3] = txt[4 * 3 + 3][:-2]
    bad = np.frombuffer(b"\n".join(txt), np.uint8)
    with pytest.raises(api.PhyError) as e:
        ctx.compress_region(bad, prm(bad))
    assert e.value.code == -1
    # the ctx still works afterwards
    d, o, _ = ctx.compress_region(good, prm(good))
    assert len(d) == 1 and d[0].status == 0


def test_roundtrip_properties_at_full_window_size(ctx):
    """Size-independent checks on a 64 MB input: every desc chains to the next, record counts add up,
    the info stream's header words agree with the descriptor."""
    data = synth.fastq("150bp_paired", 44, target_bytes=64_000_000)
    d, out, res = ctx.compress_region(data, api.region_params(data.size, 1, 0))
    assert res.bytes_in == data.size and sum(x.bytes_consumed for x in d) == data.size
    pos = 0
    for x in d:
        assert x.win_off == pos and x.status == 0
        pos += x.bytes_consumed
        p = out[x.out_off:x.out_off + 19].tobytes()
        assert int.from_bytes(p[0:4], "big") == x.n_records and int.from_bytes(p[4:8], "big") == 150
        assert x.out_len == sum(x.sec_len)
    assert sum(x.n_records for x in d) == int((data == 10).sum()) // 4


@pytest.mark.parametrize("shape,mb", [("36bp", 256), ("100bp", 128)])
def test_full_size_round_trip_through_the_reference_decoder(shape, mb, ctx):
    """Encode on the GPU -> decode with the reference's own Fetch* functions (oracle/_ref/libphyref_kat.so) -> the
    input FASTQ, byte for byte, at a size the oracle encoder would need minutes for: every 8 MiB subblock of a
    multi-batch region call is decoded (one at a time: the reference's Huffman loader keeps function-static scratch).
    Where the reference's decoder is not built, every payload must equal, by digest, the oracle's for this input
    (tests/golden/reference_digests.json; the reference decoder reads the oracle's payloads back,
    test_oracle_payloads_decode_with_the_reference_decoder) and is decoded by phy_decode_subblock instead."""
    from oracle import phy_oracle as O
    data = synth.fastq(shape, 45, target_bytes=mb * 1_000_000)
    d, out, res = ctx.compress_region(data, api.region_params(data.size, 1, 0))
    assert res.n_batches > 1 and res.bytes_in == data.size
    decode = api.decode_subblock
    if os.path.exists(O.REF_KAT) and hasattr(O.ref_kat(), "ref_decode_subblock"):
        decode = O.ref_decode_subblock
    else:
        want = gpu_cases.ref_digests(f"roundtrip_{shape}_{mb}mb_seed45_np1")["subblocks"][0]
        assert [gpu_cases.digest(p) for p in api.payloads(d, out)] == want
    bad = []
    for i, x in enumerate(d):
        dec = decode(out[x.out_off:x.out_off + x.out_len], x.bytes_consumed + 4096)
        if dec.size != x.bytes_consumed or not np.array_equal(dec, data[x.win_off:x.win_off + x.bytes_consumed]):
            bad.append(i)
    assert not bad, f"subblocks that do not decode to their input: {bad[:10]}"


@pytest.mark.parametrize("shape,mb", [("36bp", 1000), ("100bp", 512), ("150bp_paired", 512), ("var50_205", 512)])
def test_baseline_size_round_trip_through_the_decoder(shape, mb, ctx):
    """Encode on the GPU -> phy_decode_subblock (host/phy_decode.hpp) -> the input FASTQ, byte for byte, at BASELINE.json
    sizes (configs[1] in full, 512 MB slices of the shapes of configs[2..4]), every subblock of a 17-batch region call."""
    from concurrent.futures import ThreadPoolExecutor
    data = synth.fastq(shape, 46, target_bytes=mb * 1_000_000)
    d, out, res = ctx.compress_region(data, api.region_params(data.size, 1, 0))
    assert res.bytes_in == data.size and sum(x.bytes_consumed for x in d) == data.size

    def check(x):
        dec = api.decode_subblock(out[x.out_off:x.out_off + x.out_len], x.bytes_consumed + 4096)
        return dec.size == x.bytes_consumed and np.array_equal(dec, data[x.win_off:x.win_off + x.bytes_consumed])

    with ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 1)) as ex:
        ok = list(ex.map(check, d))
    assert all(ok), f"subblocks that do not decode to their input: {[i for i, v in enumerate(ok) if not v][:10]}"


def test_a_bad_record_fails_only_its_subblock_in_a_grouped_batch():
    """200 MB in one batch (three groups): a '+' line damaged in the middle fails exactly the subblock that holds it
    (PHY_ERR_MALFORMED); every other subblock of every group is written and decodes to its input."""
    data = synth.fastq("36bp", 48, target_bytes=200_000_000).copy()
    mid = data.size // 2
    plus = data[mid:mid + 4096].tobytes().find(b"\n+\n") + 1
    data[mid + plus] = ord("-")
    big = api.Context(0, max_batch_bytes=256 << 20, max_subblocks=64)
    try:
        d, out, res = big.compress_region(data, api.region_params(data.size, 1, 0), check=False)
        assert res.n_batches == 1 and len(d) >= 16
        bad = [i for i, x in enumerate(d) if x.status]
        assert len(bad) == 1 and d[bad[0]].status == -1
        assert d[bad[0]].win_off <= mid + plus < d[bad[0]].win_off + d[bad[0]].bytes_consumed
        for i in (0, bad[0] - 1, bad[0] + 1, len(d) - 1):
            x = d[i]
            dec = api.decode_subblock(out[x.out_off:x.out_off + x.out_len], x.bytes_consumed + 4096)
            assert np.array_equal(dec, data[x.win_off:x.win_off + x.bytes_consumed])
    finally:
        big.close()


@pytest.mark.parametrize("shape,seed", [("36bp", 2), ("100bp", 3)])
def test_baseline_size_payloads_bit_exact_against_the_compiled_reference(shape, seed, tmp_path):
    """BASELINE.json size, not a round trip: 1 GB of the configs[1] / configs[2] shapes is compressed by the UNMODIFIED
    reference (oracle/_ref/phyNGSC_ref, np = 2, threads = 1; about 10 s) and by the CUDA path at the same partitioning,
    once with whole-region batches (a rank's 60 subblocks run as three subblock groups) and once with 64 MiB batches.
    Every subblock payload is compared keyed by (WRID, ordinal), through its digest; so are the footer's start overlaps.
    Where the reference is not built, its payloads are stood in for by tests/golden/reference_digests.json."""
    from oracle import phy_oracle as O
    data = synth.fastq(shape, seed, target_bytes=1_000_000_000)
    if O.have_reference():
        shm = "/dev/shm" if os.path.isdir("/dev/shm") else str(tmp_path)
        src, dst = os.path.join(shm, f"phy_parity_{os.getpid()}.fastq"), os.path.join(shm, f"phy_parity_{os.getpid()}.ngsc")
        data.tofile(src)
        try:
            O.run_reference(src, dst, np_ranks=2, threads=1, timeout=900)
            ref = container.read_ngsc(dst)
        finally:
            for p in (src, dst):
                if os.path.exists(p):
                    os.remove(p)
        assert ref["footer"]["fastq_size"] == data.size
        want_sb = [[gpu_cases.digest(p) for p in ref["per_rank_subblocks"][r]] for r in range(2)]
        want_ov = ref["footer"]["overlaps"]
    else:
        g = gpu_cases.ref_digests(f"baseline_{shape}_seed{seed}_np2")
        want_sb, want_ov = g["subblocks"], g["overlaps"]
    whole = api.Context(0, max_batch_bytes=(512 << 20) + (16 << 20), max_subblocks=96)
    small = api.Context(0, max_batch_bytes=64 << 20, max_subblocks=32)
    try:
        for r in range(2):
            start, _ = api.region_slice(data.size, 2, r)
            want = want_sb[r]
            for name, c in (("whole-region batch", whole), ("64 MiB batches", small)):
                descs, out, res = c.compress_region(data[start:], api.region_params(data.size, 2, r))
                got = [gpu_cases.digest(p) for p in api.payloads(descs, out)]
                assert len(got) == len(want), f"rank {r}, {name}: {len(got)} subblocks, reference wrote {len(want)}"
                bad = [i for i, (a, b) in enumerate(zip(got, want)) if a != b]
                assert not bad, f"rank {r}, {name}: payloads {bad[:8]} differ from the reference's"
                assert res.wr_overlap == want_ov[r]
                assert (res.n_batches == 1) == (c is whole)
    finally:
        whole.close(); small.close()


def test_more_windows_than_subblock_capacity_continue_in_the_same_bytes(oracle):
    """A batch holds more windows than the context's subblock capacity (small windows, max_subblocks = 5): the window chain
    stops when the capacity is used up and the next round continues in the same resident bytes -- in the final batch, in a
    single-batch region, in the middle of a multi-batch region and on the resident legs.  Same payloads as the oracle."""
    data = synth.fastq("100bp", 49, target_bytes=3_000_000)
    win = 64 * 1024
    prm = api.region_params(data.size, 1, 0, window_bytes=win)
    want = oracle.compress_rank(data, 1, 0, window_bytes=win)["subblocks"]
    one = api.Context(0, max_batch_bytes=8 << 20, max_subblocks=5)
    many = api.Context(0, max_batch_bytes=1 << 20, max_subblocks=5)
    try:
        d1, o1, r1 = one.compress_region(data, prm)
        assert r1.n_batches >= len(want) // 5 and api.payloads(d1, o1) == want
        d2, o2, r2 = many.compress_region(data, prm)
        assert r2.n_batches > r1.n_batches // 2 and api.payloads(d2, o2) == want
        for c in (one, many):  # resident legs: one batch / several batches of a region larger than max_batch_bytes
            c.upload(data)
            d3, r3 = c.compress_resident(data.size, prm)
            o3 = np.empty(r3.out_used, np.uint8)
            assert c.download(o3) == r3.out_used
            assert api.payloads(d3, o3) == want
            assert (r3.n_batches > 1)
    finally:
        one.close(); many.close()
