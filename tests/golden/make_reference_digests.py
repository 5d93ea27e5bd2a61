"""Record tests/golden/reference_digests.json: what the GPU tests that compare with the compiled reference
(oracle/_ref) check against, for machines where the reference's sources are not available to build it.

    python tests/golden/make_reference_digests.py

The digests come from the oracle (oracle/phy_oracle.c), the C restatement of the reference that reproduces every
reference-minted .ngsc file in this directory byte for byte (tests/test_oracle_golden.py).  Each case lists, per rank,
64-bit SHA-256 digests of the subblock payloads or blocks, with the counts the tests compare.
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from gpu_cases import digest  # noqa: E402
from oracle import phy_oracle as O  # noqa: E402
from phyngsc_b200 import synth  # noqa: E402


def rank_digests(data, npr, threads=1):
    ranks = [O.compress_rank(data, npr, r, threads=threads) for r in range(npr)]
    return {"subblocks": [[digest(s) for s in x["subblocks"]] for x in ranks], "blocks": [[digest(b) for b in x["blocks"]] for x in ranks],
            "overlaps": [x["wr_overlap"] for x in ranks], "n_subblocks": sum(len(x["subblocks"]) for x in ranks)}


def main():
    cases = {}
    # test_gpu_parity.py::test_baseline_size_payloads_bit_exact_against_the_compiled_reference
    for shape, seed in (("36bp", 2), ("100bp", 3)):
        d = rank_digests(synth.fastq(shape, seed, target_bytes=1_000_000_000), 2)
        cases[f"baseline_{shape}_seed{seed}_np2"] = {"subblocks": d["subblocks"], "overlaps": d["overlaps"]}
    # test_gpu_parity.py::test_full_size_round_trip_through_the_reference_decoder (one region)
    for shape, mb in (("36bp", 256), ("100bp", 128)):
        d = rank_digests(synth.fastq(shape, 45, target_bytes=mb * 1_000_000), 1)
        cases[f"roundtrip_{shape}_{mb}mb_seed45_np1"] = {"subblocks": d["subblocks"]}
    # test_gpu_driver.py::test_driver_threads_argument_matches_the_reference_at_the_same_thread_count
    data = synth.fastq("36bp", 702, target_bytes=40_000_000 + 977)
    for threads in (2, 4):
        d = rank_digests(data, 2, threads)
        cases[f"threads{threads}_36bp_seed702_np2"] = {"blocks": d["blocks"], "n_subblocks": d["n_subblocks"]}
    with open(os.path.join(HERE, "reference_digests.json"), "w") as f:
        json.dump({"source": "oracle/phy_oracle.c via tests/golden/make_reference_digests.py", "cases": cases}, f, indent=0)
    print(f"wrote {len(cases)} cases")


if __name__ == "__main__":
    main()
