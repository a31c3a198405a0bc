#!/usr/bin/env python
"""bench.py — the Decoder hot path on B200: log lines/s and GB/s parsed, with roofline + CPU baseline.

    python bench.py --gpus N --steps K --warmup W [--format rfc5424|ltsv|gelf|rfc3164|mixed] [--lines L] [--impl reference]
                    [--dump-outputs DIR]

A "step" is one pass of the parse kernel over one synthetic batch that is already resident in HBM
(BASELINE.json configs[1]: 10 M RFC5424 lines, mean 180 B, per GPU).  `e2e` is the same metric through
the reference-facing C-ABI call fg_decode_batch() with HOST buffers (pinned H2D + kernels + D2H inside
the timed region).  For N>1 every rank owns one GPU and an independent shard of lines (weak scaling,
no collective on the parse path); time is the max over ranks.  `--impl reference` times the CPU
restatement of the reference decoders (oracle/) on the host cores for the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

FORMATS = {"rfc5424": 0, "ltsv": 1, "gelf": 2, "rfc3164": 3}
SEEDS = {"rfc5424": 5424, "ltsv": 1757, "gelf": 0x6E1F, "rfc3164": 3164}
RFC3164_YEAR = 2026  # the year timestamps without one belong to: fixed, so that a run is reproducible
# generator parameter that lands the ACTUAL mean line length on the BASELINE.json shape
GEN_MEAN = {"rfc5424": 169.2, "ltsv": 420.0, "gelf": 466.0, "rfc3164": 140.0}
TARGET_MEAN = {"rfc5424": 180, "ltsv": 420, "gelf": 512, "rfc3164": 127}
DEFAULT_LINES = {"rfc5424": 10_000_000, "ltsv": 4_000_000, "gelf": 3_500_000, "rfc3164": 10_000_000}  # int32 offsets cap a batch at 2 GiB
DUMP_BYTES = 60 << 20  # --dump-outputs writes at most this much array data (stays under 64 MB with the .npy headers)
DUMP_SEED = 0
DUMP_BLOCK = 64  # --dump-outputs samples blocks of this many consecutive lines


def env_int(name: str, default: int) -> int:
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def hbm_peak() -> tuple[float, str]:
    p = REPO / "MEASURED_PEAKS.json"
    try:
        return float(json.loads(p.read_text())["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device = device
        self.rows: list[list[str]] = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.device)], stdout=subprocess.PIPE, text=True)
        except Exception:
            self.proc = None
            return
        def pump():
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = [r for r in self.rows if len(r) >= 9]
        # samples taken while the GPU was drawing load power (the sampler runs from before the warm-ups to after the
        # timed regions; idle samples between phases would dilute the median)
        def watts(r):
            try:
                return float(r[3])
            except ValueError:
                return 0.0
        peak_w = max([watts(r) for r in rows], default=0.0)
        loaded = [r for r in rows if watts(r) >= 0.6 * peak_w] or rows
        sm = sorted(int(float(r[1])) for r in loaded if r[1].replace(".", "").isdigit())
        mx = [int(float(r[2])) for r in rows if r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) < 9:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_total": len(rows), "power_w_max": peak_w,
                "window": "from before the warm-ups to after the e2e region (50 ms period); median over samples at >= 60 % of the peak power"}



def bind_to_gpu_numa_node(local: int) -> str:
    """Pin this rank (and therefore its first-touch pinned host buffers) to the CPUs of the NUMA node its GPU hangs off,
    so that H2D/D2H traffic of 8 ranks does not cross sockets. Best effort: any failure leaves the affinity alone."""
    try:
        import torch
        p = torch.cuda.get_device_properties(local)
        bus = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(Path(f"/sys/bus/pci/devices/{bus}/numa_node").read_text().strip())
        if node < 0:
            return "numa: unknown"
        cpus = set()
        for part in Path(f"/sys/devices/system/node/node{node}/cpulist").read_text().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, cpus)
        return f"numa node {node} ({len(cpus)} cpus)"
    except Exception as e:  # noqa: BLE001
        return f"numa: not bound ({type(e).__name__})"


def make_batch(fb, fmt_name: str, lines: int, rank: int):
    fmt = FORMATS[fmt_name]
    nthreads = min(os.cpu_count() or 8, 32)
    data, offs = fb.generate(fmt, SEEDS[fmt_name], lines, first_index=rank * lines, mean_len=GEN_MEAN[fmt_name],
                             bad_frac=0.005, nthreads=nthreads)
    return data, offs


LTSV_SCHEMA = {"counter": "u64", "score": "i64", "mean": "f64", "done": "bool"}
LTSV_SUFFIXES = {"u64": "_u64", "i64": "_i64", "f64": "_f64", "bool": "_bool"}


def ltsv_kwargs(fmt_name: str, typed: bool = False) -> dict:
    """format-specific decoder configuration"""
    if fmt_name == "ltsv" and typed:
        return {"ltsv_schema": LTSV_SCHEMA, "ltsv_suffixes": LTSV_SUFFIXES}
    if fmt_name == "rfc3164":
        return {"rfc3164_year": RFC3164_YEAR}
    return {}


def oracle_config(pyoracle, fmt_name: str, typed: bool):
    if fmt_name == "ltsv" and typed:
        return pyoracle.LtsvConfig(LTSV_SCHEMA, LTSV_SUFFIXES)
    if fmt_name == "rfc3164":
        return pyoracle.Rfc3164Config(RFC3164_YEAR)
    return None


def dump_outputs(decoded: dict, out_dir: str, budget: int) -> None:
    """--dump-outputs: the Records of decoded batches ({file name prefix: (BatchDecoder, BatchResult, bytes, offsets)}) as
    the product's host library materialises them for a caller, in the canonical dump format of oracle/oracle.cpp (every
    field, ts as its bits).  The raw result arrays are not written: the kernels fill their side tables in a different order
    from run to run.  For each prefix, in `out_dir`:
        <prefix>line.npy            float64 [k]    the line numbers dumped, ascending
        <prefix>record_offsets.npy  float64 [k+1]  record i is record_bytes[offsets[i]:offsets[i+1]]
        <prefix>record_bytes.npy    float32        the dump text, one byte per element
    The lines are blocks of DUMP_BLOCK consecutive lines, taken in a seeded order until the prefix's share of `budget`
    (bytes of array data) is used."""
    import numpy as np
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    share = budget // max(len(decoded), 1) - 8
    for prefix, (dec, res, data, offsets) in decoded.items():
        blocks, used = [], 0
        for lo in np.random.default_rng(DUMP_SEED).permutation(-(-res.n // DUMP_BLOCK)) * DUMP_BLOCK:
            lo = int(lo)
            hi = min(res.n, lo + DUMP_BLOCK)
            text, offs = dec.dump(res, data, offsets, nthreads=1, lo=lo, hi=hi)
            cost = 4 * len(text) + 16 * (hi - lo)  # float32 per byte, float64 line number and offset per line
            if used + cost > share:
                break
            blocks.append((lo, hi, text, offs))
            used += cost
        blocks.sort(key=lambda b: b[0])
        lines = [np.arange(lo, hi) for lo, hi, _, _ in blocks]
        lengths = [np.diff(offs) for _, _, _, offs in blocks]
        rec_offs = np.zeros(sum(len(x) for x in lines) + 1)
        np.cumsum(np.concatenate(lengths) if lengths else [], out=rec_offs[1:])
        np.save(out / f"{prefix}line.npy", np.concatenate(lines).astype(np.float64) if lines else np.zeros(0))
        np.save(out / f"{prefix}record_offsets.npy", rec_offs)
        np.save(out / f"{prefix}record_bytes.npy", np.frombuffer(b"".join(b[2] for b in blocks), np.uint8).astype(np.float32))


def run_reference(args) -> None:
    """CPU arm: the restated reference decoders (oracle/) on the host cores, same workload shape."""
    rank = env_int("RANK", 0)
    if rank != 0:
        return
    import flowgger_b200 as fb
    sys.path.insert(0, str(REPO / "oracle"))
    import pyoracle
    fmt_name = args.format
    fmt = FORMATS[fmt_name]
    cores = os.cpu_count() or 1
    sample = args.lines  # the same lines the GPU arm parses (same generator, seed and count)
    data, offs = make_batch(fb, fmt_name, sample, 0)
    nbytes = int(offs[-1])
    ocfg = oracle_config(pyoracle, fmt_name, args.ltsv_typed)
    for _ in range(max(args.warmup, 1)):
        pyoracle.decode_bench(fmt, data, offs, ocfg, nthreads=cores)
    t = 0.0
    for _ in range(args.steps):
        s, _ok = pyoracle.decode_bench(fmt, data, offs, ocfg, nthreads=cores)
        t += s
    ms = 1e3 * t / args.steps
    value = sample / (t / args.steps)
    line = {
        "impl": "reference", "metric": "log lines/sec parsed (%s)" % fmt_name.upper(), "value": value, "unit": "lines/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "gb_per_s": nbytes / (t / args.steps) / 1e9,
        "config": {"workload": workload_name(fmt_name, args.lines), "lines_per_gpu": sample, "bytes_per_gpu": nbytes,
                   "mean_line_bytes": round(nbytes / sample, 2)},
        "cpu_baseline": {"value": value, "unit": "lines/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} lines of the same generator/seed, all {cores} host threads over contiguous line shards; "
                                   "restated reference decoder (Rust toolchain unavailable), owned Record per line"},
        "e2e": {"value": value, "unit": "lines/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)



def run_mixed(args) -> None:
    """BASELINE.json configs[4]: mixed RFC5424+GELF stream (50/50 in runs of 4096 lines), contiguous line shard per GPU.
    A Decoder instance is single-format (mod.rs:413-422), so the host demultiplexes the runs into one RFC5424 batch and
    int32-offset GELF sub-batches per GPU; a step parses all of them (device-resident)."""
    import numpy as np
    import torch
    import flowgger_b200 as fb

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce(x, op):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local}")
        dist.all_reduce(t, op=op)
        return float(t.item())

    RUN = 4096
    n5 = (args.lines // 2) // RUN * RUN
    ng = (args.lines - n5) // RUN * RUN
    sub = 3_200_000 // RUN * RUN
    parts = [("rfc5424", n5, rank * n5)]
    done = 0
    while done < ng:
        k = min(sub, ng - done)
        parts.append(("gelf", k, rank * ng + done))
        done += k
    decs = []
    nthreads = min(os.cpu_count() or 8, 32)
    tot_lines = tot_bytes = 0
    b_read = {"rfc5424": 0, "gelf": 0}
    for fmt_name, n, first in parts:
        fmt = FORMATS[fmt_name]
        data, offs = fb.generate(fmt, SEEDS[fmt_name], n, first_index=first, mean_len=GEN_MEAN[fmt_name], bad_frac=0.005, nthreads=nthreads)
        nb = int(offs[-1])
        dec = fb.BatchDecoder(fmt, device=local, max_batch_bytes=nb + (1 << 20), max_batch_lines=n, chunk_lines=1 << 19)
        hb = dec.host_alloc(nb)
        ho = dec.host_alloc(offs.nbytes, dtype=np.int32)
        hb[:] = data
        ho[:] = offs
        del data
        dec.upload(hb, ho)
        decs.append((fmt_name, dec, hb, ho, n, nb))
        tot_lines += n
        tot_bytes += nb
        b_read[fmt_name] += nb + 4 * (n + 1)
    for _ in range(max(args.warmup, 3)):
        for _, dec, *_ in decs:
            dec.parse_resident()
    launches0 = sum(d[1].kernel_launches() for d in decs)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    t0 = time.perf_counter()
    kms = {"rfc5424": 0.0, "gelf": 0.0}
    for fmt_name, dec, *_ in decs:
        kms[fmt_name] += dec.parse_resident_many(args.steps)
    barrier()
    wall = reduce(time.perf_counter() - t0, torch.distributed.ReduceOp.MAX if dist else None)
    clocks = sampler.stop() if rank == 0 else None
    launches = sum(d[1].kernel_launches() for d in decs) - launches0
    if args.dump_outputs:  # before the e2e decodes below overwrite the results of the last timed step
        rank_prefix = f"rank{rank}." if world > 1 else ""
        dump_outputs({f"{rank_prefix}{k}.{f}.": (dec, dec.download(), hb, ho) for k, (f, dec, hb, ho, *_) in enumerate(decs)},
                     args.dump_outputs, DUMP_BYTES // world)
    per_gpu = tot_lines / (wall / args.steps)
    total_lines = reduce(float(tot_lines), torch.distributed.ReduceOp.SUM if dist else None)
    total_bytes = reduce(float(tot_bytes), torch.distributed.ReduceOp.SUM if dist else None)
    value = total_lines / (wall / args.steps)
    for d in decs:
        d[1].decode(d[2], d[3])
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        for _, dec, hb, ho, *_ in decs:
            dec.decode(hb, ho)
    barrier()
    e2e_wall = reduce(time.perf_counter() - t0, torch.distributed.ReduceOp.MAX if dist else None)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sys.path.insert(0, str(REPO / "oracle"))
        import pyoracle
        cores = os.cpu_count() or 1
        t = 0.0
        ns = 0
        for fmt_name, dec, hb, ho, n, nb in decs[:2]:
            sample = min(n, 1_000_000)
            so = np.ascontiguousarray(ho[: sample + 1])
            sb = hb[: int(so[-1])]
            pyoracle.decode_bench(FORMATS[fmt_name], sb, so, None, nthreads=cores)
            sec, _ = pyoracle.decode_bench(FORMATS[fmt_name], sb, so, None, nthreads=cores)
            t += sec
            ns += sample
        cpu = {"value": ns / t, "unit": "lines/s", "cores": cores, "kind": "port",
               "sample": f"{ns} lines (equal RFC5424/GELF halves of the GPU batches), {cores} host threads; restated reference decoders"}
    if rank == 0:
        peak, peak_kind = hbm_peak()
        g_ms = kms["gelf"] / args.steps
        achieved = (b_read["gelf"] / 1e9) / (g_ms / 1e3)
        line = {
            "metric": "log lines/sec parsed (mixed RFC5424+GELF stream)", "value": value, "unit": "lines/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": 1e3 * wall / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "gb_per_s": total_bytes / (wall / args.steps) / 1e9, "per_gpu_lines_per_s": per_gpu,
            "config": {"workload": f"Mixed RFC5424+GELF stream, runs of {RUN} lines, {tot_lines} lines per GPU ({n5} RFC5424 + {ng} GELF), "
                                   f"{world} GPU(s) (BASELINE.json configs[4] = 100 M lines over 8 GPUs)",
                       "lines_per_gpu": tot_lines, "bytes_per_gpu": tot_bytes, "sub_batches": [(f, n) for f, _, _, _, n, _ in decs],
                       "parallelism": f"line shards x{world}, no collective", "l2": "every sub-batch >> 126 MB L2"},
            "kernel_ms": {k: v / args.steps for k, v in kms.items()},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "of": peak_kind,
                         "traffic": None, "kernel": "parse_gelf_kernel + post_gelf_kernel (dominant: %.1f of %.1f ms/step)" % (g_ms, (kms["gelf"] + kms["rfc5424"]) / args.steps)},
            "e2e": {"value": total_lines / (e2e_wall / args.e2e_steps), "unit": "lines/s", "h2d_bytes_per_step": b_read["gelf"] + b_read["rfc5424"],
                    "d2h_bytes_per_step": None, "steps": args.e2e_steps, "api": "fg_decode_batch (pinned host buffers)"},
            "gpu_launches": launches, "clocks": clocks,
        }
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    for d in decs:
        d[1].close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def workload_name(fmt_name: str, lines: int) -> str:
    if fmt_name == "rfc3164":
        return (f"RFC3164 batch: {lines} synthetic BSD-syslog lines per GPU, mean {TARGET_MEAN[fmt_name]} B (SURVEY.md 8(f) N3; not a "
                "BASELINE.json config)")
    if fmt_name != "rfc5424":
        return (f"{fmt_name.upper()} batch: {lines}-line int32-offset sub-batch per GPU of the 10 M-line workload, mean "
                f"{TARGET_MEAN[fmt_name]} B (BASELINE.json configs[{ {'gelf': 2, 'ltsv': 3}[fmt_name] }])")
    return f"{fmt_name.upper()} batch: {lines} synthetic lines per GPU, mean {TARGET_MEAN[fmt_name]} B (BASELINE.json configs[{ {'rfc5424': 1, 'gelf': 2, 'ltsv': 3}[fmt_name] }])"


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--format", default="rfc5424", choices=list(FORMATS) + ["mixed"])
    ap.add_argument("--lines", type=int, default=0, help="lines per GPU (default: the BASELINE.json config)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--split", action="store_true", help="also time fg_split_decode (device-side framing + UTF-8 validation, N1)")
    ap.add_argument("--ltsv-typed", action="store_true", help="LTSV with the 4-entry typed schema + suffixes (C4, second run)")
    ap.add_argument("--encode", action="store_true", help="also time fg_decode_encode_gelf (decode + GELF encode fused on the device, N2)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the Records of the last step to DIR/<name>.npy (a seeded sample of "
                         "lines, 60 MiB at most; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU decoder's outputs; --impl reference has none")
    if args.format == "mixed":
        if args.lines <= 0:
            args.lines = 12_500_000
        if args.impl == "reference":
            args.format = "rfc5424"  # the CPU arm reports per format; the mixed line carries its own cpu_baseline
            args.lines = DEFAULT_LINES["rfc5424"]
            run_reference(args)
            return
        run_mixed(args)
        return
    if args.lines <= 0:
        args.lines = DEFAULT_LINES[args.format]
    args.warmup = max(args.warmup, 0)
    if args.impl == "reference":
        run_reference(args)
        return

    import numpy as np
    import torch
    import flowgger_b200 as fb

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: flowgger_b200 has no CPU fallback")
    torch.cuda.set_device(local)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x: float) -> float:
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local}")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    fmt_name = args.format
    fmt = FORMATS[fmt_name]
    numa = bind_to_gpu_numa_node(local) if world > 1 else "numa: single rank, not bound"
    data, offs = make_batch(fb, fmt_name, args.lines, rank)
    n = args.lines
    nbytes = int(offs[-1])
    b_read = nbytes + 4 * (n + 1)  # algorithmic bytes per launch: every input byte + offset read once

    dec = fb.BatchDecoder(fmt, device=local, max_batch_bytes=nbytes + (1 << 20), max_batch_lines=n,
                          chunk_lines=env_int("FG_CHUNK_LINES", 1 << 19), **ltsv_kwargs(fmt_name, args.ltsv_typed))
    # pinned host arenas, as a batching splitter would fill them
    h_bytes = dec.host_alloc(nbytes)
    h_offs = dec.host_alloc(offs.nbytes, dtype=np.int32)
    h_bytes[:] = data
    h_offs[:] = offs
    del data

    # ---- device-resident: the kernel against the HBM roofline -------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # runs through warm-ups, the timed region and the e2e region (>= 5 samples even for a 20 ms region)
    dec.upload(h_bytes, h_offs)
    for _ in range(max(args.warmup, 3)):
        dec.parse_resident()
    # keep the GPU under the same load for a moment so that the clock record covers it (untimed)
    dec.parse_resident_many(max(args.steps, 20) * 4)
    launches0 = dec.kernel_launches()
    barrier()
    t0 = time.perf_counter()
    # K passes enqueued back to back on the launch stream, CUDA events around them, ONE host sync (per-step host syncs
    # cost ~1 ms each when 8 ranks share the host and would be charged to the GPUs)
    kernel_ms = [dec.parse_resident_many(args.steps) / args.steps]
    barrier()
    wall = time.perf_counter() - t0
    gpu_launches = dec.kernel_launches() - launches0
    wall = max_over_ranks(wall)
    k_avg_ms = max_over_ranks(sum(kernel_ms) / len(kernel_ms))
    total_lines = sum_over_ranks(float(n))
    total_bytes = sum_over_ranks(float(nbytes))
    ms_per_step = 1e3 * wall / args.steps
    value = total_lines / (wall / args.steps)

    # the dominant kernel alone (RFC5424: parse5424_kernel, without post5424_kernel), CUDA events around it, single steps
    dom = []
    for _ in range(args.steps):
        dec.parse_resident()
        dom.append(dec.last_dominant_kernel_ms())
    dom_ms = max_over_ranks(sum(dom) / len(dom))
    res = dec.download()
    n_err = int((res.status != 0).sum())
    n_entries = res.n_entries
    if fmt == 0:
        # compact results: 32-byte row per line + 8-byte side-table rows + the arena of unescaped values (+ rare wide rows)
        n_entries = int(res.raw.n_entries8)
        b_write = n * 32 + n_entries * 8 + int(res.raw.arena_bytes) + int(res.raw.n_wide) * 72 + int(res.n_entries) * 17
    else:
        b_write = n * (12 + 8 * 4) + n_entries * 17 + (int(res.raw.arena_bytes) if fmt == 3 else 0)
    d2h_bytes = b_write
    if args.dump_outputs:  # the last timed step's results, before the e2e decodes below overwrite them
        dump_outputs({f"rank{rank}." if world > 1 else "": (dec, res, h_bytes, h_offs)}, args.dump_outputs, DUMP_BYTES // world)

    # ---- end to end through the C ABI with host buffers -----------------------------------------
    dec.decode(h_bytes, h_offs)  # warm-up
    barrier()
    t0 = time.perf_counter()
    e2e_kernel_ms = 0.0
    for _ in range(args.e2e_steps):
        r = dec.decode(h_bytes, h_offs)
        e2e_kernel_ms += r.kernel_ms
    barrier()
    e2e_wall = max_over_ranks(time.perf_counter() - t0)
    e2e_value = total_lines / (e2e_wall / args.e2e_steps)
    clocks = sampler.stop() if rank == 0 else None

    # ---- bytes -> owned Records: fg_decode_batch + the host materialiser (what the reference's decode() returns) ------
    barrier()
    t0 = time.perf_counter()
    r = dec.decode(h_bytes, h_offs)
    mat_s = dec.materialize_seconds(r, h_bytes, h_offs, nthreads=max(1, (os.cpu_count() or 8) // max(world, 1)))
    barrier()
    rec_wall = max_over_ranks(time.perf_counter() - t0)
    e2e_record = {"value": total_lines / rec_wall, "unit": "lines/s", "materialize_s": mat_s,
                  "api": "fg_decode_batch + CudaBatchDecoder::materialize of every line (owned Record per line, host threads = cores / ranks)"}

    # ---- optional: bytes in -> encoded GELF records out (decode + encode fused on the device, N2) ---------------------
    encode = None
    if args.encode and fmt == 0:
        _, eo, es, ek = dec.decode_encode_gelf(h_bytes, h_offs, copy=False)  # warm-up (sizes the output buffer)
        out_bytes = int(eo[-1])
        barrier()
        t0 = time.perf_counter()
        ek = 0.0
        for _ in range(args.e2e_steps):
            _, eo, es, k1 = dec.decode_encode_gelf(h_bytes, h_offs, copy=False)
            ek += k1
        barrier()
        ew = max_over_ranks(time.perf_counter() - t0)
        encode = {"value": total_lines / (ew / args.e2e_steps), "unit": "lines/s", "h2d_bytes_per_step": b_read,
                  "d2h_bytes_per_step": out_bytes + 9 * n + 8, "json_bytes_per_gpu": out_bytes,
                  "kernel_ms_per_step": ek / args.e2e_steps, "records": int((np.asarray(es) == 0).sum()),
                  "api": "fg_decode_encode_gelf (pinned host lines in, GELF JSON records + offsets + status out; the decoder's rows never leave the device)"}

    # ---- optional: raw newline-terminated stream, framing + UTF-8 validation on the device (N1) -------
    split = None
    if args.split:
        sdata, soffs = fb.generate(fmt, SEEDS[fmt_name], n, first_index=rank * n, mean_len=GEN_MEAN[fmt_name], bad_frac=0.005,
                                   nthreads=min(os.cpu_count() or 8, 32), terminated=True)
        sdec = fb.BatchDecoder(fmt, device=local, max_batch_bytes=len(sdata) + (1 << 20), max_batch_lines=n + 64,
                               **ltsv_kwargs(fmt_name, args.ltsv_typed))
        hs = sdec.host_alloc(len(sdata))
        hs[:] = sdata
        del sdata
        sdec.split_decode(hs)
        barrier()
        t0 = time.perf_counter()
        sk = 0.0
        for _ in range(args.e2e_steps):
            r = sdec.split_decode(hs)
            sk += sdec.last_split_ms()
        barrier()
        sw = max_over_ranks(time.perf_counter() - t0)
        split = {"value": total_lines / (sw / args.e2e_steps), "unit": "lines/s", "stream_bytes_per_gpu": int(len(hs)),
                 "framing_stage_ms": sk / args.e2e_steps,
                 "api": "fg_split_decode (pinned raw stream in, 64 MiB chunks: H2D -> count/scan/fill offsets + UTF-8 check -> parse -> D2H; "
                        "framing_stage_ms spans the first to the last framing kernel, i.e. it includes waiting for the H2D chunks)"}
        sdec.close()

    # ---- CPU baseline on this box's host cores (rank 0, N=1 only) -----------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sys.path.insert(0, str(REPO / "oracle"))
        import pyoracle
        cores = os.cpu_count() or 1
        sample = min(n, 2_000_000)
        so = np.ascontiguousarray(h_offs[: sample + 1])
        sb = h_bytes[: int(so[-1])]
        ocfg = oracle_config(pyoracle, fmt_name, args.ltsv_typed)
        pyoracle.decode_bench(fmt, sb, so, ocfg, nthreads=cores)
        s_all, _ = pyoracle.decode_bench(fmt, sb, so, ocfg, nthreads=cores)
        s_one, _ = pyoracle.decode_bench(fmt, sb[: int(so[sample // 8])], np.ascontiguousarray(so[: sample // 8 + 1]), ocfg, nthreads=1)
        cpu = {"value": sample / s_all, "unit": "lines/s", "cores": cores, "kind": "port",
               "single_thread_lines_per_s": (sample // 8) / s_one,
               "sample": f"first {sample} lines of the GPU batch, {cores} host threads over contiguous line shards "
                         f"(+ {sample // 8} lines on 1 thread); restated reference decoder (oracle/, Rust toolchain unavailable)"}

    if rank == 0:
        peak, peak_kind = hbm_peak()
        achieved = (b_read / 1e9) / (dom_ms / 1e3)
        # dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel per launch, from the committed ncu capture of
        # THIS kernel build (profiles/traffic.json names the build it was taken from); scaled to this run's line count
        traffic = None
        tp = REPO / "profiles" / "traffic.json"
        if tp.exists():
            try:
                t = json.loads(tp.read_text()).get(fmt_name)
                if t and t.get("build") == fb.build_info():
                    traffic = int(t["dram_bytes_per_line"] * n)
            except Exception:
                traffic = None
        line = {
            "metric": "log lines/sec parsed (%s)" % fmt_name.upper(), "value": value, "unit": "lines/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "gb_per_s": total_bytes / (wall / args.steps) / 1e9,
            "config": {"workload": workload_name(fmt_name, n), "lines_per_gpu": n, "bytes_per_gpu": nbytes,
                       "mean_line_bytes": round(nbytes / n, 2), "error_rows": n_err, "sd_entries": n_entries,
                       "parallelism": f"line shards x{world}, no collective", "host_affinity_rank0": numa,
                       "l2": "input per step (%.2f GB) >> 126 MB L2, no flush needed" % (nbytes / 1e9)},
            "kernel_ms": k_avg_ms,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "of": peak_kind, "traffic": traffic,
                         "kernel": {0: "parse5424_kernel", 1: "parse_ltsv_kernel", 2: "parse_gelf_kernel + post_gelf_kernel", 3: "parse3164_kernel"}[fmt],
                         "kernel_ms": dom_ms, "step_ms": k_avg_ms, "step_frac": (b_read / 1e9) / (k_avg_ms / 1e3) / peak,
                         "note": "achieved = algorithmic bytes / CUDA-event time of the dominant kernel alone (single steps); "
                                 "step_* = the same over every kernel of a step (RFC5424: + post5424_kernel), which is what `value` counts",
                         "algorithmic_bytes_per_launch": b_read, "written_bytes_per_launch": b_write},
            "e2e": {"value": e2e_value, "unit": "lines/s", "h2d_bytes_per_step": b_read, "d2h_bytes_per_step": d2h_bytes,
                    "steps": args.e2e_steps, "gb_per_s": total_bytes / (e2e_wall / args.e2e_steps) / 1e9,
                    "kernel_ms_per_step": e2e_kernel_ms / args.e2e_steps, "api": "fg_decode_batch (pinned host buffers)"},
            "e2e_record": e2e_record,
            "gpu_launches": gpu_launches,
            "clocks": clocks,
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if split is not None:
            line["split_e2e"] = split
        if encode is not None:
            line["encode_e2e"] = encode
        print(json.dumps(line), flush=True)
    dec.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
