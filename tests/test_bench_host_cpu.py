"""Host logic of bench.py that needs no GPU: the repeated-segment file image every rank cuts its working region from, the
record statistics behind the per-kernel algorithmic bytes, and the N-rank partition of one file (phyNGSC.cpp:113-124) -- the
oracle compressing the regions rank by rank must give the same subblocks as it gives on the whole image."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from phyngsc_b200 import api, synth  # noqa: E402


def test_file_image_fill_is_the_tiled_segment(monkeypatch):
    monkeypatch.setattr(bench, "SEGMENT_MB", 1)
    img = bench.FileImage("100bp", 3)  # 3 MB image = a 1 MB segment three times
    seg = img.segment
    assert img.tiles == 3 and img.size == 3 * seg.size and seg[-1] == 10
    whole = np.tile(seg, 3)
    for start, end in ((0, 10), (seg.size - 5, seg.size + 7), (123_457, 2 * seg.size + 999), (0, img.size)):
        out = np.empty(end - start, np.uint8)
        assert np.array_equal(img.fill(start, end, out), whole[start:end])


def test_record_stats_counts_lines():
    data = np.frombuffer(b"@r1 x\nACGT\n+\nIIII\n@r2 yy\nAC\n+\nII\n", np.uint8)
    nrec, title, seq = bench.record_stats(data)
    assert (nrec, title, seq) == (2, 6 + 7, 4 + 2)


def test_port_baseline_sample_ends_on_a_record(oracle, monkeypatch):
    """Without the compiled reference the CPU baseline times the oracle port on a prefix of the sample; a prefix cut
    inside a record would be malformed input to it."""
    monkeypatch.setattr(bench, "PORT_SAMPLE_BYTES", 100_000)
    monkeypatch.setattr(oracle, "have_reference", lambda: False)
    seg = synth.fastq("100bp", 3, target_bytes=300_000)
    small = bench.whole_records(seg, 100_000)
    assert 90_000 < small.size <= 100_000 and small[-1] == 10 and int((small == 10).sum()) % 4 == 0
    r = bench.run_reference_sample(seg, 250_000)
    assert r["kind"] == "port" and r["value"] > 0 and f"first {small.size} bytes" in r["sample"]


def test_dump_outputs_writes_descriptors_result_and_seeded_payload_sample(tmp_path):
    """Payloads at 16-byte aligned offsets with junk in the gaps: the dump holds every descriptor, the result counts and
    the payload bytes laid end to end -- all of them when they fit, else a sample at positions fixed by the seed."""
    lens, offs = [37, 1000, 5], [0, 48, 1056]
    out = np.full(1072, 0xEE, np.uint8)
    rng = np.random.default_rng(1)
    descs, chunks = [], []
    for o, n in zip(offs, lens):
        out[o:o + n] = p = rng.integers(0, 200, n, dtype=np.uint8)
        chunks.append(p)
        d = api.SubblockDesc()
        d.out_off, d.out_len, d.bytes_consumed, d.n_records = o, n, 10 * n, n // 4
        descs.append(d)
    res = api.RegionResult()
    res.n_subblocks, res.n_batches, res.bytes_in, res.bytes_out, res.out_used, res.kernel_ms = 3, 1, 10 * sum(lens), sum(lens), 1072, 1.5
    whole = np.concatenate(chunks)

    bench.dump_outputs(str(tmp_path / "all"), descs, res, out, 1 << 20)
    s = np.load(tmp_path / "all" / "payload_sample.npy")
    assert s.dtype == np.float32 and np.array_equal(s, whole)
    d = np.load(tmp_path / "all" / "descs.npy")
    assert d.dtype == np.float64 and d.shape == (3, 14) and d[:, 11].tolist() == offs and d[:, 12].tolist() == lens
    assert np.load(tmp_path / "all" / "result.npy").tolist() == [3, 1, 10 * sum(lens), sum(lens), 1072, 0]

    budget = 3 * 128 + d.nbytes + 6 * 8 + 4 * 200
    for k in (1, 2):
        bench.dump_outputs(str(tmp_path / f"s{k}"), descs, res, out, budget, prefix="rank0_")
        assert sum(f.stat().st_size for f in (tmp_path / f"s{k}").iterdir()) <= budget
    a, b = (np.load(tmp_path / f"s{k}" / "rank0_payload_sample.npy") for k in (1, 2))
    pos = np.sort(np.random.default_rng(0).integers(0, whole.size, 200))
    assert a.size == 200 and np.array_equal(a, b) and np.array_equal(a, whole[pos])


def test_ranks_of_one_image_tile_the_file(oracle, monkeypatch):
    """The strong-scaling partition bench.py measures: rank r gets region_slice(size, N, r) of the one image and compresses
    it with region_params(size, N, r); decoded back, the ranks' subblocks are the file, every record exactly once."""
    monkeypatch.setattr(bench, "SEGMENT_MB", 1)
    img = bench.FileImage("36bp", 2)
    whole = np.tile(img.segment, img.tiles)
    for n in (1, 2, 3):
        text = []
        for r in range(n):
            start, end = api.region_slice(img.size, n, r, slack=4096)
            region = img.fill(start, end, np.empty(end - start, np.uint8))
            assert np.array_equal(region, whole[start:end])
            for sb in oracle.compress_rank(whole, n, r, window_bytes=256 * 1024)["subblocks"]:
                text.append(api.decode_subblock(sb).tobytes())
        assert b"".join(text) == whole.tobytes()  # every record of the file exactly once, in order
