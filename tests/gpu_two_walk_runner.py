"""Runs with PHY_ENC=0 (test_gpu_encoder_paths.py starts it in a subprocess: the switch is read once per process):
every subblock goes through the two-walk kernels k_lengths + k_emit.  Compares every oracle case of gpu_cases.CASES, the
deepq / wideq / lenmix inputs and the reference goldens with what they must be, checks that no subblock took the
single-walk kernels, prints one line per problem and exits non-zero when there is any."""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [HERE, os.path.dirname(HERE)]

import gpu_cases as G  # noqa: E402
from oracle import phy_oracle  # noqa: E402
from phyngsc_b200 import api, container, synth  # noqa: E402


def main():
    assert os.environ.get("PHY_ENC") == "0", "run with PHY_ENC=0"
    phy_oracle.build()
    ctx = api.Context(0, max_batch_bytes=256 << 20, max_subblocks=256)  # every call below is one batch
    probs, counts = [], {"calls": 0, "subblocks": 0}

    def check(name, data, npr, window_bytes, record_cap=api.RECORD_CAP, threads=1):
        for r in range(npr):
            p, descs, res = G.run_rank(ctx, data, npr, r, window_bytes=window_bytes, record_cap=record_cap, threads=threads)
            probs.extend(f"{name} rank {r}: {x}" for x in p)
            if res.n_batches != 1:
                probs.append(f"{name} rank {r}: {res.n_batches} batches")
            fast = [i for i, x in enumerate(G.sb_paths(ctx, len(descs))) if x[1]]
            if fast:
                probs.append(f"{name} rank {r}: subblocks {fast[:8]} took the single-walk kernels")
            counts["calls"] += 1
            counts["subblocks"] += len(descs)

    for case in G.CASES:
        name, shape, seed, nbytes, npr, win = case[:6]
        data = G.py_fastq(shape[3:], seed, nbytes) if shape.startswith("py:") else synth.fastq(shape, seed, target_bytes=nbytes + 131)
        check(name, data, npr, win, threads=case[6] if len(case) > 6 else 1)
    for L, D in ((36, 16), (100, 13), (150, 16), (300, 13)):
        data, w, cap = G.long_code_case(L, D)
        check(f"deepq_{L}bp_D{D}", data, 2, w, record_cap=cap)
    data, w, cap = G.mixed_case()
    check("deepq_mixed", data, 1, w, record_cap=cap)
    for L in G.WIDEQ_READS:
        check(f"wideq_{L}bp", G.wideq(L, 60 + L, 3_000_000), 1, 1 << 20)
    for name in sorted(G.LENMIX):
        if name == "511":
            continue  # 32 records of 511 bp exceed the two-walk kernels' 24 KiB stage: PHY_ERR_UNSUPPORTED by design
        data, w = G.lenmix_case(name)
        check(f"lenmix_{name}", data, 2, w)
    gold = os.path.join(HERE, "golden")
    with open(os.path.join(gold, "manifest.json")) as f:
        manifest = json.load(f)
    for case in manifest:
        data = synth.fastq(case["shape"], case["seed"], target_bytes=case["target_bytes"])
        ng = container.read_ngsc(os.path.join(gold, case["file"]))
        for r in range(case["np"]):
            start, _ = api.region_slice(data.size, case["np"], r)
            descs, out, res = ctx.compress_region(data[start:], api.region_params(data.size, case["np"], r), check=False)
            if api.payloads(descs, out) != ng["per_rank_subblocks"][r] or res.wr_overlap != ng["footer"]["overlaps"][r]:
                probs.append(f"golden {case['file']} rank {r}: payloads differ from the reference's")
            if any(x[1] for x in G.sb_paths(ctx, len(descs))):
                probs.append(f"golden {case['file']} rank {r}: a subblock took the single-walk kernels")
            counts["calls"] += 1
            counts["subblocks"] += len(descs)
    ctx.close()
    for p in probs:
        print(p)
    print(f"two-walk runner: {len(probs)} problems in {counts['calls']} calls, {counts['subblocks']} subblocks")
    return 1 if probs else 0


if __name__ == "__main__":
    sys.exit(main())
