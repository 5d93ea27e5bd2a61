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
    return run_rank(ctx, data, npr, rank, window_bytes=window_bytes, record_cap=record_cap, whole_tail=whole_tail, threads=threads)[0]


def run_rank(ctx, data, npr, rank, window_bytes=api.WINDOW_BYTES, record_cap=api.RECORD_CAP, whole_tail=True, threads=1):
    """One rank through the CUDA path, diffed against the oracle.  -> (problem strings, descs, result).  The call's
    SbClass records stay readable with sb_paths() (they describe the call's last batch)."""
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
            return probs, descs, res
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
    return probs, descs, res


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


# ---- which encoder path each subblock took -------------------------------------------------------------------------
MIRROR_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "mirror", "mirror.cpp")
MIRROR_LIB = os.path.join(os.path.dirname(os.path.abspath(__file__)), "mirror", "libmirror.so")
_CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "phyngsc_b200", "csrc")
_mirror = None


def mirror():
    """tests/mirror/mirror.cpp compiled with g++ (rebuilt when it or the headers it includes are newer)."""
    global _mirror
    if _mirror is not None:
        return _mirror
    import ctypes as C
    import subprocess
    import tempfile
    deps = [MIRROR_SRC] + [os.path.join(_CSRC, f) for f in ("phy_core.cuh", "phy_fast.cuh")]
    if not os.path.exists(MIRROR_LIB) or os.path.getmtime(MIRROR_LIB) < max(os.path.getmtime(p) for p in deps):
        fd, tmp = tempfile.mkstemp(suffix=".so", dir=os.path.dirname(MIRROR_LIB))
        os.close(fd)
        try:
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-x", "c++", "-fPIC", "-shared", "-o", tmp, MIRROR_SRC])
            os.replace(tmp, MIRROR_LIB)  # a concurrent loader sees the old library or the new one, never half of one
        finally:
            if os.path.exists(tmp):
                os.remove(tmp)
    L = C.CDLL(MIRROR_LIB)
    L.mirror_compress_window.restype = C.c_int
    L.mirror_compress_window.argtypes = [C.c_void_p, C.c_uint64, C.c_int64, C.c_uint32, C.c_int32, C.c_uint32, C.c_void_p,
                                         C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mirror_compress_window_fast.restype = C.c_int
    L.mirror_compress_window_fast.argtypes = L.mirror_compress_window.argtypes + [C.c_uint32]
    L.mirror_huffman.restype = C.c_uint32
    L.mirror_huffman.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
    L.mirror_sbclass_layout.restype = C.c_uint32
    L.mirror_sbclass_layout.argtypes = [C.c_void_p, C.c_uint32]
    _mirror = L
    return L


PATH_FIELDS = ("status", "fast", "qpk_esc", "max_qlen", "nq")


def sbclass_layout():
    """-> (sizeof(SbClass), {field: byte offset}) for the fields of PATH_FIELDS, from the host compile of phy_core.cuh."""
    v = np.zeros(6, np.uint32)
    mirror().mirror_sbclass_layout(v.ctypes.data, 6)
    return int(v[0]), dict(zip(PATH_FIELDS, (int(x) for x in v[1:])))


def sb_paths(ctx, n):
    """Encoder path of the first n subblocks of the context's last batch: per subblock (status, fast, qpk_esc, max_qlen, nq).
    fast = 1: single-walk kernels (k_enc_qd + k_place), 0: two-walk kernels (k_lengths + k_emit); qpk_esc = 1: some packed
    quality entry is the escape to a code longer than 12 bits."""
    size, off = sbclass_layout()
    raw = ctx.debug_read("cls", 0, n * size)
    assert raw.size == n * size
    rows = raw.reshape(n, size)
    col = lambda f: rows[:, off[f]:off[f] + 4].copy().view(np.int32 if f == "status" else np.uint32)[:, 0]  # noqa: E731
    cols = [col(f) for f in PATH_FIELDS]
    return [tuple(int(c[i]) for c in cols) for i in range(n)]


def path_counts(paths):
    """{'fast': subblocks with fast=1, 'two_walk': fast=0, 'esc': qpk_esc=1} of sb_paths()' records with status 0."""
    ok = [p for p in paths if p[0] == 0]
    return {"fast": sum(p[1] for p in ok), "two_walk": sum(1 - p[1] for p in ok), "esc": sum(p[2] for p in ok)}


# ---- inputs for the encoder's path rules ----------------------------------------------------------------------------
AMB = b"??YRWSKMDVHBNXU.-"  # ambiguity code a (2..16) -> base; a transferred quality is 112 + 8 a + (q - 33), q in 33..40
Q_FREQ = 70                 # the frequent quality symbol of deepq ('F')


def fib(k):
    a, b = 1, 1
    for _ in range(k - 1):
        a, b = b, a + b
    return a  # fib(1) = fib(2) = 1


def deepq_symbol(j):
    """Quality byte of deepq's j-th rare symbol (count fib(j) per window and read position).  The eight rarest (the longest
    codes) are bytes 143..234, which a record can also carry as an ambiguity base with a quality of 33..40 (transfer)."""
    return 130 + 13 * j if j <= 8 else 33 + j


def deepq_record_bytes(L):
    return 2 * L + 15  # "@Q.<7 digits>\n" + read + "\n+\n" + quality + "\n"


def deepq_window(L, window_bytes):
    """-> (records per window M, record_cap) for deepq reads of L bp: the record cap, not the window's bytes, ends every
    window, so every window holds M = record_cap + 1 consecutive records."""
    m = (window_bytes - 500 - 4 * deepq_record_bytes(L)) // deepq_record_bytes(L)
    return m, m - 1


def deepq_max_depth(L, window_bytes, limit=24):
    """Deepest D whose Fibonacci histogram fits a window (the frequent symbol keeps at least fib(D + 1) of the records)."""
    m, _ = deepq_window(L, window_bytes)
    d = 1
    while d < limit and fib(d + 3) - 1 + fib(d + 2) <= m:
        d += 1
    return d


def deepq(L, depths, seed, window_bytes, extra_records=0):
    """FASTQ of L bp reads whose per-position quality histograms make the longest quality code of window k exactly
    depths[k] bits.  Every M records (deepq_window) form one period: at every read position the rare symbols 1..D occur
    fib(1..D) times, shuffled per position, and the rest of the records carry Q_FREQ, so D + 1 symbols build a Huffman
    chain of depth D.  The pattern of a position repeats with period M, so any M consecutive records of a constant-D
    stretch hold exactly that histogram -- the windows of a later rank included, whatever record they start at.
    About 1 % of the records move their bytes 143..234 into transferable ambiguity codes (same quality symbols after
    the transfer).  Titles are short (one numeric field) so that a window holds many records.  extra_records more
    records of the last depth follow the last whole period."""
    m, _ = deepq_window(L, window_bytes)
    rng = np.random.default_rng(seed)
    pats = {}
    for D in sorted(set(depths)):
        assert fib(D + 2) - 1 < m, f"depth {D} needs more than {m} records per window"
        base = np.full(m, Q_FREQ, np.uint8)
        o = 0
        for j in range(1, D + 1):
            base[o:o + fib(j)] = deepq_symbol(j)
            o += fib(j)
        pats[D] = rng.permuted(np.tile(base, (L, 1)), axis=1).T.copy()  # [record of the period, position]
    n = len(depths) * m + extra_records
    q = np.empty((n, L), np.uint8)
    for k in range((n + m - 1) // m):
        c = q[k * m:(k + 1) * m]
        c[:] = pats[depths[min(k, len(depths) - 1)]][:c.shape[0]]
    s = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, (n, L))]
    hi = q >= 128
    cand = np.flatnonzero(hi.any(axis=1))
    xf = cand[rng.random(cand.size) < min(1.0, 0.01 * n / max(cand.size, 1))]
    sub = hi[xf]
    v = q[xf].astype(np.int32) - 112
    s[xf] = np.where(sub, np.frombuffer(AMB, np.uint8)[np.clip(v // 8, 0, 16)], s[xf])
    q[xf] = np.where(sub, 33 + v % 8, q[xf]).astype(np.uint8)
    return _fixed_records(b"@Q.", s, q)


def _fixed_records(prefix, s, q):
    """Records of equal read length: title prefix + (1000000 + i), read s[i], quality q[i]."""
    n, L = s.shape
    num = (1000000 + np.arange(n))[:, None] // (10 ** np.arange(6, -1, -1))[None, :] % 10 + 48
    t = len(prefix)
    rec = np.empty((n, t + 7 + 1 + L + 3 + L + 1), np.uint8)
    rec[:, :t] = np.frombuffer(prefix, np.uint8)
    rec[:, t:t + 7] = num
    o = t + 7
    rec[:, o] = 10; rec[:, o + 1:o + 1 + L] = s; o += 1 + L
    rec[:, o:o + 3] = np.frombuffer(b"\n+\n", np.uint8); rec[:, o + 3:o + 3 + L] = q; rec[:, -1] = 10
    return rec.reshape(-1)


def wideq(L, seed, nbytes, nsym=41):
    """L bp reads, qualities drawn uniformly from nsym symbols (33..33+nsym-1), bases ACGT: packed quality tables of
    (L + 1) x nsym x 2 bytes with short codes."""
    n = max(1, nbytes // (2 * L + 15))
    rng = np.random.default_rng(seed)
    s = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, (n, L))]
    q = (33 + rng.integers(0, nsym, (n, L))).astype(np.uint8)
    return _fixed_records(b"@W.", s, q)


def lenmix(lengths, seed, nbytes, long_at=None, nsym=20):
    """Reads whose lengths are drawn from `lengths` (one value: fixed length), nsym quality symbols, bases ACGT (20: the
    packed quality tables of 511 bp reads, 512 x 20 x 2 bytes, fit shared memory).  long_at =
    (byte offset, L): the first record starting at or after that offset has L bases instead."""
    rng = np.random.default_rng(seed)
    out, n, i = [], 0, 0
    acgt = np.frombuffer(b"ACGT", np.uint8)
    while n < nbytes:
        L = int(rng.choice(lengths))
        if long_at is not None and n >= long_at[0]:
            L, long_at = long_at[1], None
        rec = (b"@M.%d\n" % (1000000 + i) + acgt[rng.integers(0, 4, L)].tobytes() + b"\n+\n"
               + (33 + rng.integers(0, nsym, L)).astype(np.uint8).tobytes() + b"\n")
        out.append(rec)
        n += len(rec)
        i += 1
    return np.frombuffer(b"".join(out), np.uint8).copy()


def window_depths(data, npr, rank, window_bytes, record_cap=api.RECORD_CAP):
    """Per oracle window of the rank: (longest quality code over the read-position tables 1..max_qlen, the same over all
    tables incl. the whole-read table 0), from the window's per-position quality histograms (after the ambiguity
    transfer, phyNGSC.cpp:549-588) and oracle.huffman."""
    amb = np.zeros(256, np.int32)
    for a, c in enumerate(AMB):
        if a >= 2:
            amb[c] = a
    for c in b"ACGT":
        amb[c] = 1
    ref = O.compress_rank(data, npr, rank, window_bytes=window_bytes, record_cap=record_cap)
    out = []
    for (woff, wlen, rs, ov), nrec in zip(ref["windows"], ref["records"]):
        lines = data[woff + rs:woff + wlen].tobytes().split(b"\n", 4 * nrec)[:4 * nrec]
        seqs, quals = lines[1::4], lines[3::4]
        hist = np.zeros((max(len(x) for x in seqs) + 1) * 256, np.int64)
        for L in sorted({len(x) for x in seqs}):
            idx = [i for i, x in enumerate(seqs) if len(x) == L]
            s = np.frombuffer(b"".join(seqs[i] for i in idx), np.uint8).reshape(-1, L)
            q = np.frombuffer(b"".join(quals[i] for i in idx), np.uint8).reshape(-1, L).astype(np.int64)
            a = amb[s]
            xf = (a != 1).any(axis=1) & ((a == 1) | ((a >= 2) & (q >= 33) & (q <= 40))).all(axis=1)
            q = np.where(xf[:, None] & (a >= 2), 112 + 8 * a + q - 33, q)
            hist += np.bincount(((np.arange(L) + 1)[None, :] * 256 + q).ravel(), minlength=hist.size)
        hist = hist.reshape(-1, 256)
        syms = np.flatnonzero(hist.sum(axis=0))
        deep = max(int(O.huffman(h[syms].astype(np.uint32), True)[1].max()) for h in hist[1:])
        out.append((deep, max(deep, int(O.huffman(hist[1:, syms].sum(axis=0).astype(np.uint32), True)[1].max()))))
    return out


# ---- the encoder's path rules (k_slots, run_body) restated for the tests' expectations --------------------------------
PK_SMEM_MAX = 24 * 1024  # packed quality tables larger than this stay in global memory (phy_b200.cu)


def seg_len(L, g):
    return (L + 4 * g - 1) // (4 * g) * 4


def enc_lanes(max_len):
    """Lanes per record of k_enc_qd for a batch whose longest read is max_len."""
    g = 1 if max_len <= 64 else 4 if max_len <= 256 else 8
    while g < 8 and seg_len(max_len, g) > 64:
        g *= 2
    return g


def staging_words(max_len, qcode_hint):
    """Lane-private staging words of k_enc_qd: 12-bit codes unless the context's previous batch saw longer ones (<= 24)."""
    return (seg_len(max_len, enc_lanes(max_len)) * min(max(qcode_hint, 12), 24) + 31) // 32 + 2


def single_walk_fits(read_len, depth, max_len, qcode_hint):
    """k_slots' staging test: a lane's run of positions times the subblock's longest quality code fits the staging."""
    return seg_len(read_len, enc_lanes(max_len)) * depth <= 32 * (staging_words(max_len, qcode_hint) - 1)


def deepq_window_bytes(L, D):
    """Smallest window (a power of two, at most 8 MiB) that holds a deepq period of depth D for L bp reads."""
    w = 1 << 16
    while w < (1 << 23) and deepq_max_depth(L, w) < D:
        w *= 2
    assert deepq_max_depth(L, w) >= D, (L, D)
    return w


LONG_CODE_READS = (36, 100, 150, 300)


def long_code_depths(L):
    return (13, 16, deepq_max_depth(L, 1 << 23))


def long_code_case(L, D, seed=0):
    """-> (data, window_bytes, record_cap): four deepq periods of depth D and a third of one more."""
    w = deepq_window_bytes(L, D)
    m, cap = deepq_window(L, w)
    return deepq(L, [D] * 4, 1000 + 7 * L + D + seed, w, extra_records=m // 3), w, cap


MIXED_SHALLOW, MIXED_DEEP, MIXED_WINDOWS, MIXED_SWITCH = 8, 15, 24, 12


def mixed_case():
    """36 bp, 256 KiB windows: MIXED_SWITCH shallow windows, then deep ones, MIXED_WINDOWS in all (one rank)."""
    w = 256 * 1024
    m, cap = deepq_window(36, w)
    depths = [MIXED_SHALLOW] * MIXED_SWITCH + [MIXED_DEEP] * (MIXED_WINDOWS - MIXED_SWITCH)
    return deepq(36, depths, 4242, w), w, cap


WIDEQ_READS = (298, 299)  # (L + 1) * 41 * 2 bytes of packed tables: 24 518 and 24 600, either side of PK_SMEM_MAX
LENMIX = {  # name -> read lengths; the switch points of enc_lanes (64/65, 256/257), of k_seqstat's counters (126/127)
    "64": (64,), "65": (65,), "126": (126,), "127": (127,), "256": (256,), "257": (257,),
    "64_65": (64, 65), "126_127": (126, 127), "256_257": (256, 257), "511": (511,)}


def lenmix_case(name):
    lens = LENMIX[name]
    return lenmix(lens, 500 + max(lens) + len(lens), 1_500_000 if max(lens) < 300 else 3_000_000), 256 * 1024
