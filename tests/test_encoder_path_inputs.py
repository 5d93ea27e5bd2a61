"""CPU checks of the inputs tests/test_gpu_encoder_paths.py relies on: the longest quality code of every deepq window is
the depth the GPU test expects, the wide-alphabet inputs sit either side of the shared-memory limit of the packed tables,
the read-length mixes reach both sides of each switch point, the single-walk encoder logic (tests/mirror) reproduces the
oracle on windows with long codes, and the SbClass layout the GPU tests decode is sane."""
import ctypes as C

import numpy as np
import pytest

import gpu_cases as G


@pytest.fixture(scope="module")
def mirror():
    return G.mirror()


@pytest.mark.parametrize("L", G.LONG_CODE_READS)
def test_long_code_windows_have_the_depth_the_gpu_tests_expect(L, oracle):
    for D in G.long_code_depths(L):
        data, w, cap = G.long_code_case(L, D)
        for npr in (1, 2):
            for r in range(npr):
                deps = G.window_depths(data, npr, r, w, cap)
                m, _ = G.deepq_window(L, w)
                ref = oracle.compress_rank(data, npr, r, window_bytes=w, record_cap=cap)
                full = [i for i, n in enumerate(ref["records"]) if n == m]
                assert full, f"L={L} D={D} np={npr} rank {r}: no window holds a whole period"
                assert all(deps[i] == (D, D) for i in full), (L, D, npr, r, deps)
                assert all(d[1] <= D for d in deps)


def test_mixed_batch_windows_switch_depth_in_the_second_group(oracle):
    data, w, cap = G.mixed_case()
    deps = G.window_depths(data, 1, 0, w, cap)
    assert len(deps) == G.MIXED_WINDOWS
    assert [d[0] for d in deps] == [G.MIXED_SHALLOW] * G.MIXED_SWITCH + [G.MIXED_DEEP] * (G.MIXED_WINDOWS - G.MIXED_SWITCH)
    s0 = [G.MIXED_WINDOWS * g // 3 for g in range(4)]  # run_body's three subblock groups
    assert s0[1] < G.MIXED_SWITCH < s0[2]
    assert G.single_walk_fits(36, G.MIXED_SHALLOW, 36, 0) and not G.single_walk_fits(36, G.MIXED_DEEP, 36, 0)


def test_deepq_transfers_ambiguity_codes_in_about_one_percent_of_records():
    data = G.deepq(36, [16] * 2, 7, 1 << 19)
    recs = data.tobytes().split(b"\n")
    seqs, quals = recs[1::4], recs[3::4]
    xf = [i for i, s in enumerate(seqs) if any(c not in b"ACGT" for c in s)]
    assert 0.005 * len(seqs) < len(xf) < 0.02 * len(seqs)
    for i in xf:  # every non-ACGT base carries a quality of 33..40: the whole record is transferred
        assert all(33 <= q <= 40 for c, q in zip(seqs[i], quals[i]) if c not in b"ACGT")


@pytest.mark.parametrize("L", G.WIDEQ_READS)
def test_wide_alphabet_packed_tables_sit_either_side_of_the_shared_memory_limit(L, oracle):
    data = G.wideq(L, 60 + L, 3_000_000)
    ref = oracle.compress_rank(data, 1, 0, window_bytes=1 << 20)
    assert len(ref["subblocks"]) >= 2
    for p in ref["subblocks"]:
        max_qlen, nq = int.from_bytes(p[4:8], "big"), p[14]
        assert (max_qlen, nq) == (L, 41)
        assert (((max_qlen + 1) * nq * 2 + 15) // 16 * 16 <= G.PK_SMEM_MAX) == (L == 298)  # run_body reserves 16-byte units


@pytest.mark.parametrize("name", sorted(G.LENMIX))
def test_read_length_mixes_reach_both_sides_of_each_switch(name, oracle):
    data, w = G.lenmix_case(name)
    ref = oracle.compress_rank(data, 1, 0, window_bytes=w)
    lens = set(G.LENMIX[name])
    for (woff, wlen, rs, ov), n in zip(ref["windows"], ref["records"]):
        got = {len(x) for x in data[woff + rs:woff + wlen].tobytes().split(b"\n", 4 * n)[1:4 * n:4]}
        assert got == lens or (len(lens) > 1 and n < 100 and got <= lens)


@pytest.mark.parametrize("lanes_per_record", [1, 4, 8])
@pytest.mark.parametrize("L,D", [(36, 16), (100, 16), (150, 14)])
def test_single_walk_encoder_logic_reproduces_oracle_on_long_codes(L, D, lanes_per_record, mirror, oracle):
    """phy_fast.cuh emulated lane by lane (codes of D > 12 bits span staging words) against the oracle, one whole deepq
    period per window."""
    w = G.deepq_window_bytes(L, D)
    m, cap = G.deepq_window(L, w)
    d = G.deepq(L, [D], 90 + L, w, extra_records=50)
    want = oracle.compress_window(d, r_buffer_size=w, record_cap=cap)
    assert want["n_records"] == m
    out = np.zeros(d.size + 65536, np.uint8); sec = np.zeros(4, np.uint32); nr = C.c_uint32(); bc = C.c_uint64()
    rc = mirror.mirror_compress_window_fast(d.ctypes.data, d.size, w, 0, 500, cap, out.ctypes.data, out.size, sec.ctypes.data,
                                            C.byref(nr), C.byref(bc), lanes_per_record)
    assert rc == 0
    assert sec.tolist() == [len(s) for s in want["sections"]]
    assert out[: int(sec.sum())].tobytes() == want["payload"]
    assert (nr.value, bc.value) == (want["n_records"], want["bytes_consumed"])


def test_sbclass_layout_export():
    size, off = G.sbclass_layout()
    assert off["status"] == 0
    assert off["max_qlen"] == 5 * 4 and off["nq"] == 8 * 4  # status R nf P nnc | max_qlen max_slen nsym nq
    assert off["max_qlen"] < off["nq"] < off["qpk_esc"] < off["fast"] < size
    assert all(v % 4 == 0 for v in off.values()) and size % 8 == 0
