#!/usr/bin/env python
"""bench.py -- FASTQ compress throughput (input GB/s) of the B200-native phyNGSC subblock path.

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA path through the C ABI)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU implementation
    python bench.py --gpus 1 --dump-outputs DIR              # also writes the last timed step's outputs (see dump_outputs)

Workload (BASELINE.json configs[2], the configuration the metric's "1/2/4/8 B200" is quoted on): ONE synthetic 16 GB
FASTQ file image of 100 bp reads with N runs and a 41-symbol quality alphabet.  Strong scaling with the reference's own
partitioning (phyNGSC.cpp:113-164): with N ranks, rank r compresses the working region [r*size/N, (r+1)*size/N + 499]
of that image -- forward sync to its first record, window chaining, the final-window rule -- on its own GPU.  No
data-path collective; the only cross-rank datum is the exclusive scan of the compressed sizes that fixes the file
offsets (torch.distributed here, MPI_Exscan in the host driver).  The image is a 1 GB generated segment repeated, so
every rank can materialise exactly its own bytes of the same file.  A "step" is one pass of the hot path over the
whole image (all ranks together).

value       kernel-only: every rank's region resident in HBM, CUDA-event time of its whole kernel sequence (all batches),
            max over ranks
e2e         the same regions from pinned HOST memory through phy_compress_region: H2D + kernels + D2H of the payloads
            into pinned host memory, wall clock around the synchronous call, max over ranks
driver_e2e  file to file: the drop-in driver binary (host/phyNGSC_b200, MPI_Exscan + MPI_File_write_at + footer) on a
            tmpfs copy of the first --driver-mb of the image with N ranks; its own COMP_TIME (file open -> footer written),
            max over ranks; the .ngsc is parsed back and checked
"""
import argparse
import json
import os
import re
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {  # name -> description
    "36bp": "36 bp Illumina-style reads, ERR005195-like titles (BASELINE.json configs[1] shape)",
    "100bp": "100 bp reads with N runs and a 41-symbol quality alphabet (BASELINE.json configs[2] shape)",
    "150bp_paired": "150 bp paired-style reads (configs[3] shape)",
    "var50_205": "variable-length 50-205 bp reads, 17-field titles, skewed quality (configs[4] shape, in-domain cap)",
}
SEGMENT_MB = 1000
PORT_SAMPLE_BYTES = 64_000_000  # the oracle port is a scalar single-core loop: a larger sample only costs time
DUMP_BYTES = 64_000_000  # most bytes --dump-outputs writes, all files together


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--shape", default="100bp", choices=sorted(WORKLOADS))
    ap.add_argument("--mb", type=int, default=16000, help="size of the whole file image in MB (10^6 bytes), split over the ranks")
    ap.add_argument("--cpu-sample-mb", type=int, default=256)
    ap.add_argument("--e2e-batch-mb", type=int, default=128, help="batch size (MiB) of the pipelined end-to-end run")
    ap.add_argument("--driver-mb", type=int, default=8000, help="file size of the file-to-file driver leg (0: skip it)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-shapes", action="store_true", help="skip the 1 GB kernel-only probes of the other named shapes (N = 1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed kernel-only step returned to DIR/*.npy (see dump_outputs)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    return a


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs (the recipe's `-lms` loop, started
    before the region and stopped after it)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) >= 7:
                self.rows.append((time.perf_counter(), parts))

    def wait_first(self, timeout=5.0):
        t = time.perf_counter()
        while self.proc is not None and not self.rows and time.perf_counter() - t < timeout:
            time.sleep(0.02)

    def summary(self, t0=None, t1=None):
        if self.proc is not None:
            self.proc.terminate()
        rows = [r for (t, r) in self.rows if (t0 is None or t >= t0 - 0.11) and (t1 is None or t <= t1 + 0.11)] or [r for _, r in self.rows]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}

        def num(x):
            try:
                return float(x)
            except ValueError:
                return None
        sm = sorted(v for v in (num(r[0]) for r in rows) if v is not None)
        reasons = set()
        for r in rows:
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": num(rows[0][1]), "reasons": sorted(reasons), "samples": len(rows),
                "power_w_max": max((v for v in (num(r[2]) for r in rows) if v is not None), default=None)}


class FileImage:
    """The benchmark's FASTQ file: one generated segment of whole records repeated `tiles` times.  Any byte range of the
    file can be materialised from the segment, so N ranks see N regions of the SAME file without anyone holding all of it."""

    def __init__(self, shape, total_mb, seed=3):
        from phyngsc_b200 import synth
        seg_mb = min(SEGMENT_MB, total_mb)
        self.segment = synth.fastq(shape, seed, target_bytes=seg_mb * 1_000_000)
        self.tiles = max(1, round(total_mb / seg_mb))
        self.size = self.segment.size * self.tiles

    def fill(self, start, end, out):
        """out[0 : end - start] = file[start : end]"""
        n, seg, pos, o = end - start, self.segment.size, start, 0
        while o < n:
            k = pos % seg
            m = min(seg - k, n - o)
            out[o:o + m] = self.segment[k:k + m]
            o += m; pos += m
        return out[:n]

    def write(self, path, nbytes):
        with open(path, "wb") as f:
            left = nbytes
            while left > 0:
                m = min(left, self.segment.size)
                f.write(memoryview(self.segment[:m]))
                left -= m
        return nbytes


def record_stats(data):
    """records and title / sequence byte totals (for the per-kernel algorithmic bytes)."""
    nl = np.flatnonzero(data == 10)
    nrec = nl.size // 4
    nl = nl[: nrec * 4].reshape(nrec, 4)
    starts = np.concatenate(([0], nl[:-1, 3] + 1))
    title = int((nl[:, 0] - starts + 1).sum())
    seq = int((nl[:, 1] - nl[:, 0] - 1).sum())
    return nrec, title, seq


def whole_records(data, n):
    """data[:n] cut back to the end of its last complete four-line record."""
    nl = np.flatnonzero(data[:n] == 10)
    return data[:int(nl[(nl.size // 4) * 4 - 1]) + 1]


def dump_outputs(path, descs, res, out, budget, prefix=""):
    """Writes what one compress_resident + download returned, so that two builds can be compared output for output:
      descs.npy           float64 [n_subblocks, 14]: every descriptor field in SubblockDesc order (sec_len as four columns)
      result.npy          float64 [6]: n_subblocks, n_batches, bytes_in, bytes_out, out_used, wr_overlap
      payload_sample.npy  float32: payload bytes of the payloads laid end to end (the alignment gaps between them are not
                          outputs) -- all of them if they fit `budget`, else those at the sorted positions
                          np.random.default_rng(0).integers(0, bytes_out, n)
    Times and launch counts are left out: they are how the call ran, not what it computed."""
    rows = np.array([[d.win_off, d.win_len, d.rec_start, d.overlap, d.n_records, d.warnings, d.bytes_consumed, *d.sec_len,
                      d.out_off, d.out_len, d.status] for d in descs], np.float64).reshape(-1, 14)
    result = np.array([res.n_subblocks, res.n_batches, res.bytes_in, res.bytes_out, res.out_used, res.wr_overlap], np.float64)
    off, ln = rows[:, 11].astype(np.int64), rows[:, 12].astype(np.int64)
    ends = np.cumsum(ln)
    total = int(ends[-1]) if ln.size else 0
    n = max(0, min(total, (budget - rows.nbytes - result.nbytes - 3 * 128) // 4))  # 128: an .npy header
    pos = np.arange(total) if n == total else np.sort(np.random.default_rng(0).integers(0, total, n))
    i = np.searchsorted(ends, pos, side="right")
    sample = out[off[i] + pos - (ends[i] - ln[i])].astype(np.float32)
    os.makedirs(path, exist_ok=True)
    for name, arr in (("descs", rows), ("result", result), ("payload_sample", sample)):
        np.save(os.path.join(path, prefix + name + ".npy"), arr)


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        return os.cpu_count() or 1


def run_reference_sample(data, sample_bytes, tmpdir="/dev/shm"):
    """Times the reference's own CPU implementation (oracle/_ref/phyNGSC_ref = the unmodified sources built
    against the fork-based MPI stand-in) on the first `sample_bytes` of the image, cut at a record boundary,
    with one single-threaded rank per host core (rank scaling is the reference's effective axis, BASELINE.md).
    Falls back to the oracle port (one core) when the reference binary is not there.
    -> dict(value GB/s, cores, kind, sample, seconds)"""
    from oracle import phy_oracle as O
    sample = whole_records(data, sample_bytes)
    cut = sample.size
    cores = host_cores()
    if O.have_reference():
        npr = max(2, min(cores, 64))
        src = os.path.join(tmpdir, f"phy_bench_{os.getpid()}.fastq")
        dst = src + ".ngsc"
        sample.tofile(src)
        try:
            t = time.perf_counter()
            out = O.run_reference(src, dst, np_ranks=npr, threads=1, timeout=1200)
            wall = time.perf_counter() - t
        finally:
            for p in (src, dst):
                if os.path.exists(p):
                    os.remove(p)
        times = [float(m.group(1)) for m in re.finditer(r"^\s*\d+\s+([0-9.]+)\s+\d+\s+\d+\s*$", out, re.M)]
        secs = max(times) if times else wall
        return dict(value=cut / secs / 1e9, unit="GB/s", cores=npr, kind="reference", seconds=secs,
                    sample=f"first {cut} bytes of the file image, unmodified reference, np={npr} x threads=1 over the fork-based MPI stand-in, "
                           f"tmpfs I/O included (max COMP_TIME {secs:.3f}s, wall {wall:.3f}s)")
    O.build()
    small = whole_records(sample, PORT_SAMPLE_BYTES)  # a record cut short would be malformed input to the port
    t = time.perf_counter()
    O.compress_rank(small, 1, 0)
    secs = time.perf_counter() - t
    return dict(value=small.size / secs / 1e9, unit="GB/s", cores=1, kind="port", seconds=secs,
                sample=f"first {small.size} bytes of the file image, oracle/phy_oracle.c (scalar port), 1 core")


def run_driver_leg(image, nbytes, n_ranks, tmpdir="/dev/shm"):
    """File to file through the drop-in driver binary with n_ranks ranks (one GPU each): -> dict or None."""
    from phyngsc_b200 import build, container
    exe = build.build_driver()
    src = os.path.join(tmpdir, f"phy_bench_drv_{os.getpid()}.fastq")
    dst = src + ".ngsc"
    try:
        image.write(src, nbytes)
        env = dict(os.environ, PHY_SHIM_NP=str(n_ranks))
        env.pop("LOCAL_RANK", None)  # the driver's ranks pick GPU rank % device_count
        t = time.perf_counter()
        p = subprocess.run([exe, src, dst, "1"], env=env, capture_output=True, text=True, timeout=1800)
        wall = time.perf_counter() - t
        if p.returncode != 0:
            return {"error": (p.stdout[-300:] + p.stderr[-300:]).strip()}
        times = [float(m.group(1)) for m in re.finditer(r"^\s*\d+\s+([0-9.]+)\s+\d+\s+\d+\s*$", p.stdout, re.M)]
        secs = max(times) if times else wall
        ng = container.read_ngsc(dst)  # parses every block header, joins split subblocks, reads the footer
        ok = (ng["footer"]["fastq_size"] == nbytes and ng["footer"]["np"] == n_ranks and len(ng["footer"]["block_order"]) == ng["footer"]["n_blocks"]
              and sum(len(x) for x in ng["per_rank_subblocks"]) == ng["footer"]["n_subblocks"])
        return {"value": nbytes / secs / 1e9, "unit": "GB/s", "file_bytes": int(nbytes), "ngsc_bytes": os.path.getsize(dst), "ranks": n_ranks,
                "comp_time_s": secs, "wall_s": wall, "container_ok": bool(ok), "n_blocks": ng["footer"]["n_blocks"], "n_subblocks": ng["footer"]["n_subblocks"],
                "what": "phyNGSC_b200 in.fastq out.ngsc 1 on tmpfs: reader thread + pinned staging, GPU path, block assembly, MPI_Exscan, "
                        "MPI_File_write_at, footer; max COMP_TIME over ranks (process start-up and CUDA context creation are outside it only "
                        "as far as they precede the file open, like MPI_Init in the reference)"}
    finally:
        for q in (src, dst):
            if os.path.exists(q):
                os.remove(q)


def main():
    # stdout carries exactly one JSON line: everything libraries print (NCCL's version banner, warnings) goes to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())

    a = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    config = {"workload": f"one {a.mb} MB synthetic FASTQ file image, {WORKLOADS[a.shape]}", "shape": a.shape, "file_mb": a.mb, "window_bytes": 1 << 23,
              "partitioning": "region = size/np: rank r of N compresses the reference's working region r of the one file (phyNGSC.cpp:113-164), "
                              "forward sync and final-window rule included",
              "l2": "every rank's region (>= 2 GB) is larger than the 126 MB L2; no flush needed"}

    if a.impl == "reference":
        if rank != 0:
            return 0
        image = FileImage(a.shape, a.mb)
        data = image.segment
        sample = min(a.cpu_sample_mb * 1_000_000, data.size)
        vals = []
        for i in range(a.warmup + a.steps):
            r = run_reference_sample(data, sample)
            if i >= a.warmup:
                vals.append(r)
        secs = sum(v["seconds"] for v in vals) / len(vals)
        value = float(np.mean([v["value"] for v in vals]))
        line = {"impl": "reference", "metric": "fastq_compress_input_throughput", "value": value, "unit": "GB/s", "n_gpus": a.gpus,
                "steps": a.steps, "warmup": a.warmup, "ms_per_step": secs * 1e3, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": value, "unit": "GB/s", "cores": vals[-1]["cores"], "kind": vals[-1]["kind"], "sample": vals[-1]["sample"]},
                "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        emit(line)
        return 0

    import torch
    import torch.distributed as dist
    from phyngsc_b200 import api
    from phyngsc_b200 import dist as pdist
    if not torch.cuda.is_available():
        print("bench.py: no CUDA device -- the product path has no CPU fallback", file=sys.stderr)
        return 2
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- this rank's working region of the one file ------------------------------------------------------------
    image = FileImage(a.shape, a.mb)
    slack = 64 * 1024  # bytes read past p_wr_end: records longer than the overlap (SURVEY.md Q4)
    start, end = api.region_slice(image.size, world, rank, slack=slack)
    pin_in = api.pinned_array(end - start + 8192)
    region = image.fill(start, end, pin_in.array)
    pin_out = api.pinned_array(region.size // 2 + (1 << 20))
    prm = api.region_params(image.size, world, rank)
    max_descs = region.size // (4 << 20) + 64
    ctx = api.Context(local)  # defaults: batches of 1 GiB + 16 MiB, 192 subblocks per batch

    # ---- kernel-only ---------------------------------------------------------------------------------------
    ctx.upload(region)
    for _ in range(a.warmup):
        descs, res = ctx.compress_resident(region.size, prm, max_descs=max_descs)
    sampler = ClockSampler(local)
    sampler.wait_first()
    barrier()
    k_ms, launches = 0.0, 0
    t0 = time.perf_counter()
    t_region0 = t0
    for _ in range(a.steps):
        descs, res = ctx.compress_resident(region.size, prm, max_descs=max_descs)
        k_ms += res.kernel_ms
        launches += res.kernel_launches
    barrier()
    wall_k = time.perf_counter() - t0
    ms_per_step = max_over_ranks(k_ms / a.steps)
    bytes_in, bytes_out, n_batches = res.bytes_in, res.bytes_out, res.n_batches
    total_in = sum_over_ranks(float(bytes_in))
    total_out = sum_over_ranks(float(bytes_out))
    value = total_in / (ms_per_step * 1e-3) / 1e9
    if a.dump_outputs:  # the payloads of the last timed step are still in device memory; pin_out is free until the e2e leg
        ctx.download(pin_out.array)
        dump_outputs(a.dump_outputs, descs, res, pin_out.array, DUMP_BYTES // world, f"rank{rank}_" if world > 1 else "")

    # ---- end to end from pinned host memory ---------------------------------------------------------------------
    # a second context with small batches: upload of batch b+1, kernels of batch b and download of batch b-1 overlap
    ctx_e = api.Context(local, max_batch_bytes=a.e2e_batch_mb << 20, max_subblocks=(a.e2e_batch_mb << 20) // (4 << 20) + 16)
    ctx_e.compress_region(region, prm, out=pin_out.array, max_descs=max_descs)
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        d2, o2, r2 = ctx_e.compress_region(region, prm, out=pin_out.array, max_descs=max_descs)
        _offset, _total = pdist.exscan_bytes(r2.bytes_out, device="cuda")  # file offsets (MPI_Exscan in the host driver)
    barrier()
    e2e_s = max_over_ranks((time.perf_counter() - t0) / a.steps)
    clocks = sampler.summary(t_region0, time.perf_counter())
    h2d_total, d2h_total = sum_over_ranks(float(region.size)), sum_over_ranks(float(r2.out_used))
    e2e = {"value": total_in / e2e_s / 1e9, "unit": "GB/s", "h2d_bytes_per_step": int(h2d_total), "d2h_bytes_per_step": int(d2h_total),
           "ms_per_step": e2e_s * 1e3, "batches_per_rank": int(r2.n_batches), "batch_mb": a.e2e_batch_mb, "h2d_ms_sum_rank0": r2.h2d_ms,
           "kernel_ms_sum_rank0": r2.kernel_ms, "d2h_ms_sum_rank0": r2.d2h_ms,
           "overlap": "upload / kernels / download of consecutive batches run on three streams"}
    assert r2.bytes_out == bytes_out and r2.bytes_in == bytes_in, "pipelined and resident runs disagree"
    ctx_e.close()
    # what the box's host <-> device path can move with no kernels at all (all ranks copying at once): the e2e leg's ceiling
    ceil = pdist.copy_ceiling(1.0, float(r2.out_used) / max(1, region.size))
    e2e["copy_ceiling"] = {"input_gbs_while_payloads_flow_back": ceil["both"]["aggregate_gbs"], "h2d_alone_gbs": ceil["h2d"]["aggregate_gbs"],
                           "d2h_alone_gbs": ceil["d2h"]["aggregate_gbs"], "per_rank_min_gbs": ceil["both"]["per_rank_gbs_min"],
                           "what": "copy-only probe on this box, all ranks at once: 1 GB per rank host -> device plus the payload fraction device -> host, "
                                   "pinned memory, 64 MiB pieces, two streams (phyngsc_b200.dist.copy_ceiling)"}
    e2e["frac_of_copy_ceiling"] = e2e["value"] / max(1e-9, ceil["both"]["aggregate_gbs"])

    # ---- per-kernel times -> roofline of the dominant kernel ---------------------------------------------------------
    ctx.profile(True)
    for _ in range(2):
        ctx.compress_resident(region.size, prm, max_descs=max_descs)
    stages = {k: v * n_batches for k, v in ctx.profile_read().items()}  # ms per step of this rank (mean per batch x batches)
    ctx.profile(False)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy, read+write)"
    else:
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    line = None
    if rank == 0:
        nrec_s, title_s, seq_s = record_stats(image.segment)
        f = bytes_in / image.segment.size  # this rank's share, in segments
        nrec, title_b, seq_b = nrec_s * f, title_s * f, seq_s * f
        # algorithmic bytes per step of each stage on this rank (DESIGN.md section 3): what it must read + must write
        # (stat2 / enc_title read the parsed title rows k_stat1 left, not the title bytes: the title bytes are an upper bound for them)
        alg = {"nl_count": bytes_in + bytes_in / 8, "nl_emit": bytes_in / 8 + 12 * nrec, "stat1": title_b + 4 * nrec, "seqstat": 2 * seq_b + 2 * nrec,
               "stat2": title_b + 8 * nrec, "enc_title": title_b + 0.12 * bytes_out, "enc_qd": 2 * seq_b + 0.88 * bytes_out, "place": 2 * bytes_out,
               "lengths": bytes_in + 8 * nrec, "emit": bytes_in + bytes_out}
        dom = max((k for k in stages if k in alg), key=lambda k: stages[k])
        ach = alg[dom] / (stages[dom] * 1e-3) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tpath):  # one ncu --set full capture, scaled to this region by algorithmic bytes
            tj = json.load(open(tpath)).get("k_" + dom)
            if tj:
                traffic = int(tj["traffic"] * alg[dom] / tj["algorithmic"])
        roofline = {"bound": "hbm", "kernel": "k_" + dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                    "traffic_source": "profiles/ncu_traffic.json (ncu --set full capture, scaled by algorithmic bytes)" if traffic else None,
                    "peak_source": peak_src, "algorithmic_bytes": int(alg[dom]), "kernel_ms": stages[dom],
                    "pipeline": {"algorithmic_bytes": int(bytes_in + bytes_out), "achieved": (bytes_in + bytes_out) / (k_ms / a.steps * 1e-3) / 1e9,
                                 "frac": (bytes_in + bytes_out) / (k_ms / a.steps * 1e-3) / 1e9 / peak, "note": "rank 0: (region bytes in + payload bytes out) / its kernel-leg time"},
                    "stage_ms": {k: round(v, 4) for k, v in stages.items()}}
        cpu = None
        if world == 1 and not a.no_cpu_baseline:
            cpu = run_reference_sample(image.segment, a.cpu_sample_mb * 1_000_000)
            cpu.pop("seconds", None)
        line = {"metric": "fastq_compress_input_throughput", "value": value, "unit": "GB/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": config, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
                "compression": {"bytes_in": int(total_in), "bytes_out": int(total_out), "ratio": total_in / max(1.0, total_out)},
                "wall_ms_per_step_kernel_loop": wall_k / a.steps * 1e3, "batches_per_rank_resident": int(n_batches)}
    # ---- the other named shapes, kernel-only on 1 GB each (one GPU only) -------------------------------------------------
    if world == 1 and not a.no_other_shapes and line is not None:
        from phyngsc_b200 import synth
        other = {}
        for shp, seed in (("36bp", 2), ("150bp_paired", 4), ("var50_205", 5)):
            if shp == a.shape:
                continue
            dat = synth.fastq(shp, seed, target_bytes=1_000_000_000)
            ctx.upload(dat)
            p1 = api.region_params(dat.size, 1, 0)
            for _ in range(2):
                ctx.compress_resident(dat.size, p1)
            ms = []
            for _ in range(3):
                _d, rr = ctx.compress_resident(dat.size, p1)
                ms.append(rr.kernel_ms)
            m = float(np.median(ms))
            other[shp] = {"what": f"1 GB of {WORKLOADS[shp]}, one region, kernel-only", "value": rr.bytes_in / (m * 1e-3) / 1e9, "unit": "GB/s", "ms": m,
                          "ratio": rr.bytes_in / max(1, rr.bytes_out), "pipeline_frac": (rr.bytes_in + rr.bytes_out) / (m * 1e-3) / 1e9 / peak}
        line["other_shapes"] = other
    ctx.close()
    pin_in.free(); pin_out.free()
    barrier()
    if world > 1:
        dist.destroy_process_group()  # the other ranks are done: nothing of theirs may keep a GPU busy during the driver leg
    # ---- file to file through the drop-in driver binary (rank 0 starts it; its N ranks take the N GPUs) -------------------------
    if a.driver_mb and line is not None:
        try:
            nbytes = max(1, min(a.driver_mb * 1_000_000, image.size) // image.segment.size) * image.segment.size
            line["driver_e2e"] = run_driver_leg(image, nbytes, world)
        except Exception as e:  # noqa: BLE001
            line["driver_e2e"] = {"error": f"{type(e).__name__}: {e}"}
    if line is not None:
        emit(line)
    return 0


if __name__ == "__main__":
    sys.exit(main())
