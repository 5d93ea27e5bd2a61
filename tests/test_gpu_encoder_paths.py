"""The encoder's per-subblock path choices against the oracle.  k_slots and run_body send a subblock through the
single-walk kernels (k_enc_qd + k_place) or the two-walk kernels (k_lengths + k_emit), with the packed quality tables in
shared memory or in global memory, and with escapes for quality codes longer than 12 bits.  Every test compares payloads,
section lengths and windows with the oracle and asserts, from the SbClass records of the call (gpu_cases.sb_paths), the
path it is about -- so that a test cannot drift onto another path without failing."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import gpu_cases as G
from phyngsc_b200 import api, synth

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def fresh():
    """A context whose first batch sizes the single-walk staging for 12-bit codes and waits for the exact packed-table size."""
    return api.Context(0, max_batch_bytes=64 << 20, max_subblocks=64)


def run(ctx, data, npr, rank, **kw):
    """One single-batch call, diffed against the oracle -> its subblocks' paths."""
    probs, descs, res = G.run_rank(ctx, data, npr, rank, **kw)
    assert not probs, "\n".join(probs[:20])
    assert res.n_batches == 1
    paths = G.sb_paths(ctx, len(descs))
    assert all(p[0] == 0 for p in paths)
    return paths


def test_sbclass_size_matches_the_device_build():
    ctx = api.Context(0, max_batch_bytes=1 << 20, max_subblocks=4)
    try:
        assert int(ctx.debug_read("sizeof", 0, 24, dtype=np.uint32)[2]) == G.sbclass_layout()[0]
    finally:
        ctx.close()


@pytest.mark.parametrize("npr", [1, 2])
@pytest.mark.parametrize("L", G.LONG_CODE_READS)
def test_long_quality_codes_on_a_fresh_context_then_the_same_context(L, npr, oracle):
    """deepq at D = 13, 16 and the deepest a window allows.  First call on a fresh context (staging for 12-bit codes):
    single-walk with escapes exactly where seg_len * D fits the staging, else the two-walk fallback -- both bit-exact.
    Second call on the same context (staging sized from the first call's longest code): single-walk with escapes."""
    for D in G.long_code_depths(L):
        data, w, cap = G.long_code_case(L, D)
        for r in range(npr):
            deps = G.window_depths(data, npr, r, w, cap)
            ctx = fresh()
            try:
                first = run(ctx, data, npr, r, window_bytes=w, record_cap=cap)
                assert len(first) == len(deps)
                for (st, fast, esc, qlen, nq), (dq, dall) in zip(first, deps):
                    assert qlen == L
                    assert fast == int(G.single_walk_fits(L, dq, L, 0)), (L, D, r, dq, fast)
                    assert esc == int(dall > 12)
                assert any(d == (D, D) for d in deps)
                second = run(ctx, data, npr, r, window_bytes=w, record_cap=cap)
                assert [p[1] for p in second] == [1] * len(second), (L, D, r)
                assert [p[2] for p in second] == [int(d[1] > 12) for d in deps]
                print(f"L={L} D={D} np={npr} rank {r}: first {G.path_counts(first)}, second {G.path_counts(second)}")
            finally:
                ctx.close()


def test_mixed_batch_places_and_emits_into_one_output(oracle):
    """One batch of 24 subblocks in three groups: shallow windows single-walk, deep ones two-walk (fresh context), the
    switch in the middle of the second group, every payload equal to the oracle's."""
    data, w, cap = G.mixed_case()
    ctx = fresh()
    try:
        paths = run(ctx, data, 1, 0, window_bytes=w, record_cap=cap)
    finally:
        ctx.close()
    assert len(paths) == G.MIXED_WINDOWS
    fast = [p[1] for p in paths]
    assert fast == [1] * G.MIXED_SWITCH + [0] * (G.MIXED_WINDOWS - G.MIXED_SWITCH)
    s0 = [G.MIXED_WINDOWS * g // 3 for g in range(4)]
    assert 0 < sum(fast[s0[1]:s0[2]]) < s0[2] - s0[1]  # both paths inside the second group
    assert all(p[2] == 1 for p in paths[G.MIXED_SWITCH:])
    print(f"mixed batch: {G.path_counts(paths)}")


def test_quality_alphabet_grows_between_calls(oracle):
    """The packed-table reservation of a later batch comes from the previous batch's alphabet (+ 8 symbols): 5 symbols,
    then 41 -> every subblock two-walk with its tables in global memory, then single-walk on the next call.  The other
    order stays single-walk."""
    small = synth.fastq("150bp_paired", 71, target_bytes=1_500_000)
    wide = G.wideq(100, 72, 1_500_000)
    w = 256 * 1024
    ctx = fresh()
    try:
        p0 = run(ctx, small, 1, 0, window_bytes=w)
        assert all(p[1] == 1 and p[4] == 5 for p in p0)
        p1 = run(ctx, wide, 1, 0, window_bytes=w)
        assert all(p[4] == 41 for p in p1) and [p[1] for p in p1] == [0] * len(p1)
        p2 = run(ctx, wide, 1, 0, window_bytes=w)
        assert [p[1] for p in p2] == [1] * len(p2)
        print(f"5 then 41 symbols: {G.path_counts(p0)} -> {G.path_counts(p1)} -> {G.path_counts(p2)}")
    finally:
        ctx.close()
    ctx = fresh()
    try:
        p0 = run(ctx, wide, 1, 0, window_bytes=w)
        p1 = run(ctx, small, 1, 0, window_bytes=w)
        assert [p[1] for p in p0 + p1] == [1] * (len(p0) + len(p1))
    finally:
        ctx.close()


@pytest.mark.parametrize("L", G.WIDEQ_READS)
def test_packed_tables_in_shared_and_in_global_memory(L, oracle):
    """41 quality symbols: 298 bp keeps the packed tables in shared memory (single-walk), 299 bp is past PK_SMEM_MAX and
    the group runs two-walk with the tables in global memory."""
    data = G.wideq(L, 60 + L, 3_000_000)
    ctx = fresh()
    try:
        paths = run(ctx, data, 1, 0, window_bytes=1 << 20)
    finally:
        ctx.close()
    assert all(p[3] == L and p[4] == 41 and p[2] == 0 for p in paths)
    assert [p[1] for p in paths] == [int(L == 298)] * len(paths)


@pytest.fixture(scope="module")
def lctx(oracle):
    c = fresh()
    yield c
    c.close()


@pytest.mark.parametrize("npr", [1, 2])
@pytest.mark.parametrize("name", sorted(G.LENMIX))
def test_read_length_switch_points(name, npr, lctx):
    """Lanes per record 1 -> 4 at 64/65 bp and 4 -> 8 at 256/257 bp, k_seqstat's 32-bit -> 16-bit counters at 126/127
    rows, 511 bp (the longest read the raw per-position table takes; records beyond the 500-byte overlap).  One context
    for all of them, each case twice: later batches reserve the packed tables from the previous alphabet plus eight
    symbols, and that reservation must not push tables that fit (511 bp: 20 480 B) out of shared memory."""
    data, w = G.lenmix_case(name)
    for r in range(npr):
        for _ in range(2):
            paths = run(lctx, data, npr, r, window_bytes=w)
            assert [(p[1], p[3] in G.LENMIX[name]) for p in paths] == [(1, True)] * len(paths)


def test_reads_of_512_bases_fail_their_subblock_and_the_context_stays_usable(lctx, oracle):
    data = G.lenmix((36,), 77, 1_500_000, long_at=(700_000, 512))
    w = 256 * 1024
    want = oracle.compress_rank(data, 1, 0, window_bytes=w)
    descs, out, res = lctx.compress_region(data, api.region_params(data.size, 1, 0, window_bytes=w), check=False)
    assert len(descs) == len(want["subblocks"])
    long_rec = re.search(rb"\n([ACGT]{512})\n", data.tobytes()).start(1)  # the 512 bp read
    bad = [i for i, d in enumerate(descs) if d.status]
    assert len(bad) == 1 and descs[bad[0]].status == -4  # PHY_ERR_UNSUPPORTED
    assert descs[bad[0]].win_off <= long_rec < descs[bad[0]].win_off + descs[bad[0]].bytes_consumed
    for i, d in enumerate(descs):
        if i != bad[0]:
            assert out[d.out_off:d.out_off + d.out_len].tobytes() == want["subblocks"][i]
    good = G.lenmix((36,), 78, 1_000_000)
    assert not G.compare_rank(lctx, good, 1, 0, window_bytes=w)


def test_forced_two_walk_encoder_is_bit_exact():
    """PHY_ENC=0 (read once per process, hence a subprocess): every oracle case, the deepq / wideq / lenmix inputs and the
    reference goldens through k_lengths + k_emit (solo variant for 36 bp, warp pairs for 100 bp and longer)."""
    env = dict(os.environ, PHY_ENC="0")
    p = subprocess.run([sys.executable, os.path.join(HERE, "gpu_two_walk_runner.py")], env=env, capture_output=True, text=True,
                       timeout=1200)
    print(p.stdout[-4000:])
    assert p.returncode == 0, p.stdout[-8000:] + p.stderr[-4000:]
    assert "two-walk runner: 0 problems" in p.stdout
