"""Shared helpers of the GPU parity tests: run the CUDA path through the C ABI and diff it against the
oracle, reporting the first differing section / byte so that one GPU run says as much as possible."""
import hashlib
import json
import os

import numpy as np

from oracle import phy_oracle as O
from phyngsc_b200 import api, synth

SEC = ["info", "title", "quality", "dna"]
REF_DIGESTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_digests.json")


def digest(b):
    """Short content digest of one payload or block (64 bits of SHA-256)."""
    return hashlib.sha256(b).hexdigest()[:16]


def ref_digests(key):
    """Stored stand-in for a compiled-reference run (tests/golden/make_reference_digests.py)."""
    with open(REF_DIGESTS) as f:
        return json.load(f)["cases"][key]


def first_diff(a, b):
    n = min(len(a), len(b))
    x = np.frombuffer(a[:n], np.uint8) != np.frombuffer(b[:n], np.uint8)
    k = int(np.argmax(x)) if x.any() else n
    return k


def compare_rank(ctx, data, npr, rank, window_bytes=api.WINDOW_BYTES, record_cap=api.RECORD_CAP, whole_tail=True, verbose=True, threads=1):
    """-> list of problem strings (empty = parity)."""
    ref = O.compress_rank(data, npr, rank, window_bytes=window_bytes, record_cap=record_cap, threads=threads)
    start, end = api.region_slice(data.size, npr, rank)
    region = data[start:] if whole_tail else data[start:end]
    prm = api.region_params(data.size, npr, rank, window_bytes=window_bytes, record_cap=record_cap, threads=threads)
    probs = []
    try:
        descs, out, res = ctx.compress_region(region, prm, check=True)
    except api.PhyError as e:
        probs.append(f"rank {rank}: call failed: {e}")
        descs, out, res = ctx.compress_region(region, prm, check=False)
        if len(descs) > len(ref["subblocks"]) + 8:
            return probs
    if len(descs) != len(ref["subblocks"]):
        probs.append(f"subblock count {len(descs)} != {len(ref['subblocks'])}")
    if res.wr_overlap != ref["wr_overlap"]:
        probs.append(f"wr_overlap {res.wr_overlap} != {ref['wr_overlap']}")
    for i, d in enumerate(descs[: len(ref["subblocks"])]):
        woff, wlen, rs, ov = ref["windows"][i]
        tag = f"rank {rank} sb {i}"
        if d.status:
            probs.append(f"{tag}: status {d.status}")
            continue
        if (d.win_off + start, d.win_len, d.rec_start, d.overlap) != (woff, wlen, rs, ov):
            probs.append(f"{tag}: window {(d.win_off + start, d.win_len, d.rec_start, d.overlap)} != {(woff, wlen, rs, ov)}")
        if d.n_records != ref["records"][i]:
            probs.append(f"{tag}: n_records {d.n_records} != {ref['records'][i]}")
        mine = out[d.out_off:d.out_off + d.out_len].tobytes()
        want = ref["subblocks"][i]
        if list(d.sec_len) != ref["section_lens"][i]:
            probs.append(f"{tag}: section lens {list(d.sec_len)} != {ref['section_lens'][i]}")
        if mine != want:
            o = 0
            for k in range(4):
                a = mine[sum(d.sec_len[:k]):sum(d.sec_len[:k + 1])]
                b = want[o:o + ref["section_lens"][i][k]]
                o += ref["section_lens"][i][k]
                if a != b:
                    j = first_diff(a, b)
                    probs.append(f"{tag}: {SEC[k]} differs at byte {j}/{len(b)} (len {len(a)} vs {len(b)}): got {a[j:j+12].hex()} want {b[j:j+12].hex()}")
    return probs


CASES = [  # (name, shape, seed, bytes, np, window_bytes)
    ("36bp_small_windows", "36bp", 21, 1_500_000, 2, 256 * 1024),
    ("100bp_small_windows", "100bp", 22, 2_000_000, 3, 384 * 1024),
    ("100bp_huffdna", "100bp_huffdna", 23, 1_200_000, 2, 512 * 1024),
    ("150bp_paired", "150bp_paired", 24, 1_500_000, 2, 300 * 1000),
    ("var50_205", "var50_205", 25, 1_500_000, 2, 256 * 1024),
    ("var50_250_slack", "var50_250", 26, 1_500_000, 2, 256 * 1024),
    ("title_stress", "title_stress", 27, 1_200_000, 2, 400 * 1024),
    ("degrade", "degrade", 28, 300_000, 2, 128 * 1024),
    ("mixed_amb", "mixed_amb", 29, 600_000, 3, 128 * 1024),
    ("36bp_one_rank", "36bp", 30, 700_000, 1, 200 * 1024),
    ("36bp_full_window", "36bp", 31, 20_000_000, 2, 1 << 23),
    ("100bp_full_window", "100bp", 32, 20_000_000, 2, 1 << 23),
    ("mixed_amb_record_cap", "mixed_amb", 33, 12_000_000, 2, 1 << 23),
    ("long300_two_position_passes", "py:long300", 34, 3_000_000, 2, 1 << 20),
    ("odd_quality_bytes", "py:odd_qual", 35, 1_500_000, 2, 512 * 1024),
    ("tiny_reads", "py:tiny", 36, 600_000, 2, 128 * 1024),
    ("36bp_threads4_short_last_window", "36bp", 702, 40_000_000 + 846, 2, 1 << 23, 4),
    ("100bp_threads3_small_windows", "100bp", 37, 1_500_000, 2, 64 * 1024, 3),
]


def py_fastq(kind, seed, nbytes):
    """Inputs the C generator has no shape for (each exercises one path of the CUDA kernels):
    long300    300 bp reads: more read positions than the 256 rows of k_qhist's private table (second pass over the
               positions), records beyond the reference's 500-byte overlap
    odd_qual   quality bytes outside 33..127 (>= 128, < 33) in records without ambiguity codes: k_qhist's exact recount
    tiny       reads of 1..6 bases: tails of the four-bases-per-step loops, blocks with very few payload bits
    """
    rng = np.random.default_rng(seed)
    out = []
    n = 0
    i = 0
    while n < nbytes:
        i += 1
        if kind == "long300":
            L = 300
            title = f"@LR{seed}.{i} run:{i % 7}:{(i * 37) % 1000} len={L}"
        elif kind == "tiny":
            L = int(rng.integers(1, 7))
            title = f"@T.{i} {i % 3}/1"
        else:
            L = 36
            title = f"@OQ.{i} x_{(i * 13) % 500:03d}:{i % 2047}/2"
        seq = rng.choice(np.frombuffer(b"ACGT", np.uint8), L)
        qual = rng.choice(np.arange(35, 74, dtype=np.uint8), L, p=None)
        if kind == "odd_qual" and rng.random() < 0.02:
            k = int(rng.integers(0, L))
            qual[k] = int(rng.choice([200, 255, 128, 31, 9, 127]))
        if kind == "long300" and rng.random() < 0.03:
            k = int(rng.integers(0, L))
            seq[k] = ord("N"); qual[k] = 35
        rec = title.encode() + b"\n" + seq.tobytes() + b"\n+\n" + qual.tobytes() + b"\n"
        out.append(rec)
        n += len(rec)
    return np.frombuffer(b"".join(out), np.uint8).copy()


def run_case(ctx, case):
    name, shape, seed, nbytes, npr, win = case[:6]
    threads = case[6] if len(case) > 6 else 1
    data = py_fastq(shape[3:], seed, nbytes) if shape.startswith("py:") else synth.fastq(shape, seed, target_bytes=nbytes + 131)
    probs = []
    for r in range(npr):
        probs += compare_rank(ctx, data, npr, r, window_bytes=win, threads=threads)
    return probs
