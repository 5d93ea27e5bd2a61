"""The drop-in host driver (phyngsc_b200/host/phyNGSC_b200: C++/MPI over the C ABI) end to end: same CLI as the
reference, .ngsc written with MPI_Exscan offsets + MPI_File_write_at.  Every block, keyed by rank, must equal the
oracle's / the reference golden's; the footer must describe the rank-major order actually written."""
import json
import os
import subprocess

import pytest

from gpu_cases import digest, ref_digests
from phyngsc_b200 import build, container, synth

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def run_driver(src, dst, npr, threads=1):
    exe = build.build_driver()
    env = dict(os.environ, PHY_SHIM_NP=str(npr))
    p = subprocess.run([exe, str(src), str(dst), str(threads)], env=env, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    return p.stdout


@pytest.mark.parametrize("shape,mb,npr", [("36bp", 30, 2), ("100bp", 70, 2), ("150bp_paired", 25, 3), ("var50_205", 20, 1), ("mixed_amb", 9, 4)])
def test_driver_file_matches_oracle_blocks_and_footer(shape, mb, npr, tmp_path, oracle):
    data = synth.fastq(shape, 500 + mb, target_bytes=mb * 1_000_000 + 977)
    src, dst = tmp_path / "in.fastq", tmp_path / "out.ngsc"
    data.tofile(src)
    out = run_driver(src, dst, npr)
    assert "COMP_TIME" in out
    ranks = [oracle.compress_rank(data, npr, r) for r in range(npr)]
    order = [r for r in range(npr) for _ in ranks[r]["blocks"]]
    want = b"".join(b for r in range(npr) for b in ranks[r]["blocks"])
    got = open(dst, "rb").read()
    assert got[: len(want)] == want                                   # every header and payload, rank-major
    if npr > 1:
        foot = oracle.make_footer(npr, data.size, len(order), sum(len(x["subblocks"]) for x in ranks), [x["wr_overlap"] for x in ranks],
                                  order, [x["last_block_size"] for x in ranks])
        assert got[len(want):] == foot
    ng = container.read_ngsc(got)
    assert ng["footer"]["block_order"] == order and ng["footer"]["fastq_size"] == data.size
    for r in range(npr):
        assert ng["per_rank_subblocks"][r] == ranks[r]["subblocks"]


@pytest.mark.parametrize("case", [c for c in json.load(open(os.path.join(GOLD, "manifest.json"))) if c["shape"] in ("36bp", "title_stress", "100bp_huffdna")],
                         ids=lambda c: c["file"])
def test_driver_blocks_match_reference_goldens_keyed_by_rank(case, tmp_path):
    data = synth.fastq(case["shape"], case["seed"], target_bytes=case["target_bytes"])
    src, dst = tmp_path / "in.fastq", tmp_path / "out.ngsc"
    data.tofile(src)
    run_driver(src, dst, case["np"])
    mine = container.read_ngsc(str(dst))
    ref = container.read_ngsc(os.path.join(GOLD, case["file"]))
    for r in range(case["np"]):
        assert [b["raw"] for b in mine["per_rank_blocks"][r]] == [b["raw"] for b in ref["per_rank_blocks"][r]]
    assert mine["footer"]["overlaps"] == ref["footer"]["overlaps"]
    assert mine["footer"]["n_subblocks"] == ref["footer"]["n_subblocks"]


@pytest.mark.parametrize("shape,mb,npr,stream", [("var50_205", 400, 3, "1"), ("36bp", 150, 2, "0")])
def test_compress_then_decompress_gives_the_file_back(shape, mb, npr, stream, tmp_path):
    """The whole tool chain on a file: driver (reader thread + streamed region call, or everything read first) -> .ngsc
    with several blocks per rank and subblocks split across blocks -> phyngsc_b200.decompress -> the input, byte for byte."""
    from phyngsc_b200 import decompress
    data = synth.fastq(shape, 600 + mb, target_bytes=mb * 1_000_000 + 311)
    src, dst, back = tmp_path / "in.fastq", tmp_path / "out.ngsc", tmp_path / "back.fastq"
    data.tofile(src)
    os.environ["PHY_DRIVER_STREAM"] = stream
    try:
        run_driver(src, dst, npr)
    finally:
        del os.environ["PHY_DRIVER_STREAM"]
    if stream == "1":
        n, k = decompress.decompress(str(dst), str(back), threads=8)  # Python container reader + phy_decode_subblock
        assert n == data.size and k >= npr
    else:
        p = subprocess.run([build.build_decompressor(), str(dst), str(back), "8"], capture_output=True, text=True, timeout=600)  # the C++ program
        assert p.returncode == 0, p.stdout + p.stderr
    assert open(back, "rb").read() == data.tobytes()


@pytest.mark.parametrize("threads", [2, 4])
def test_driver_threads_argument_matches_the_reference_at_the_same_thread_count(threads, tmp_path, oracle):
    """`threads` > 1: 36 bp windows hold ~69 k records (more than 100000/threads, so a whole-window cap of 100000/threads
    would cut them short), and the small final window of rank 0 keeps more records than with one thread because only the
    reference's last thread applies the stop rule (phyNGSC.cpp:261-266, 303, 315).  The driver's blocks must equal the
    oracle's at that thread count and -- keyed by rank -- the unmodified reference's (which is flaky with more than one
    thread, SURVEY.md Q16: it gets a few attempts; where it is not built, tests/golden/reference_digests.json stands in)."""
    data = synth.fastq("36bp", 702, target_bytes=40_000_000 + 977)  # seed picked so that the last window differs from the one-thread result
    src, dst, ref = tmp_path / "in.fastq", tmp_path / "out.ngsc", tmp_path / "ref.ngsc"
    data.tofile(src)
    out = run_driver(src, dst, 2, threads=threads)
    assert "WARNING" not in out
    mine = container.read_ngsc(str(dst))
    one = [oracle.compress_rank(data, 2, r, threads=1)["subblocks"] for r in range(2)]
    for r in range(2):
        assert mine["per_rank_subblocks"][r] == oracle.compress_rank(data, 2, r, threads=threads)["subblocks"]
    assert mine["per_rank_subblocks"] != one, "this input was chosen because its last window depends on the thread count"
    if oracle.have_reference():
        want = None
        for _ in range(4):
            try:
                oracle.run_reference(str(src), str(ref), np_ranks=2, threads=threads, timeout=90)
                want = container.read_ngsc(str(ref))
                break
            except Exception:  # noqa: BLE001  (hang or crash of the multi-threaded reference)
                continue
        if want is None:
            pytest.skip("the reference did not finish with this thread count")
        want_blocks = [[digest(b["raw"]) for b in want["per_rank_blocks"][r]] for r in range(2)]
        want_nsb = want["footer"]["n_subblocks"]
    else:
        g = ref_digests(f"threads{threads}_36bp_seed702_np2")
        want_blocks, want_nsb = g["blocks"], g["n_subblocks"]
    for r in range(2):
        assert [digest(b["raw"]) for b in mine["per_rank_blocks"][r]] == want_blocks[r]
    assert mine["footer"]["n_subblocks"] == want_nsb


@pytest.mark.parametrize("shape,mb,npr,threads", [("100bp", 60, 2, 1), ("36bp", 45, 3, 2)])
def test_patch_b_reference_main_over_the_c_abi_writes_the_reference_blocks(shape, mb, npr, threads, tmp_path, oracle):
    """INTEGRATION.md patch B, compiled: the reference's own phyNGSC.cpp with its loop body replaced by one phy_compress_region
    call (oracle/patch_b.py applies the edit to /root/reference where it lies and links -lphyngsc_b200; the binary travels in
    oracle/_ref/).  Block assembly, headers, the timestamp-ordered writer and the footer are still the reference's code, so the
    file it writes must hold, per rank, exactly the blocks the unmodified reference writes, and a footer with the same counts."""
    from oracle import patch_b
    exe = patch_b.build()
    if not exe or not os.path.exists(exe) or not oracle.have_reference():
        pytest.skip("oracle/_ref/phyNGSC_patchB or phyNGSC_ref not built (needs /root/reference at build time)")
    data = synth.fastq(shape, 900 + mb, target_bytes=mb * 1_000_000 + 131)
    src, dst, ref = tmp_path / "in.fastq", tmp_path / "patched.ngsc", tmp_path / "ref.ngsc"
    data.tofile(src)
    env = dict(os.environ, PHY_SHIM_NP=str(npr), OMP_NUM_THREADS=str(threads))
    p = subprocess.run([exe, str(src), str(dst), str(threads)], env=env, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    mine = container.read_ngsc(str(dst))
    want = None
    for _ in range(4):  # the multi-threaded reference is flaky (SURVEY.md Q16)
        try:
            oracle.run_reference(str(src), str(ref), np_ranks=npr, threads=threads, timeout=120)
            want = container.read_ngsc(str(ref))
            break
        except Exception:  # noqa: BLE001
            continue
    if want is None:
        pytest.skip("the reference did not finish with this thread count")
    for r in range(npr):
        assert [b["raw"] for b in mine["per_rank_blocks"][r]] == [b["raw"] for b in want["per_rank_blocks"][r]]
    for k in ("np", "fastq_size", "n_blocks", "n_subblocks"):
        assert mine["footer"][k] == want["footer"][k]
