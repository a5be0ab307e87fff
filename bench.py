#!/usr/bin/env python
"""bench.py -- measures the association hot path on B200(s) and prints ONE JSON line (rank 0).

Headline (`value`): pairwise SNP x SNP tests per second on BASELINE.json configs[3] -- exhaustive epistasis screen
(computeBoost's pair loop: 3x3x2 contingency table + KSA statistic, threshold 30) on 5 000 cases / 5 000 controls x
500 000 SNPs = 124 999 750 000 pairs -- STRONG scaling: the same problem on N = 1, 2, 4, 8 GPUs. One process per GPU
(torchrun), the store replicated, the tile-pair schedule cut into one shard per rank inside the library, hit records
combined with NCCL all_gather inside the timed region. A step = one pass over all pairs; device-timed with CUDA events,
max over ranks. roofline: bound "tensor" (the screen counts with tcgen05 int8 MMAs); peak = the int8 rate this device
sustains with the kernel's own MMA instruction on resident operands (gwasdev_i8_peak, measured in this process), and the
north star's integer-popcount view of the same launch in roofline.int_popc.

`e2e`: the reference's computeBoost call surface through the C-ABI with HOST buffers, every step: case/control masks from
host memory -> selection -> margins -> tensor-core operands -> screen -> fp64 re-score -> sort -> hits to host -> G-test
of every hit, results to host. N = 1: gwasdev_select_case_control + gwasdev_pairwise_scan + gwasdev_gtest on one store.
N > 1: ONE process (rank 0; the other ranks wait on a CPU barrier) drives all N GPUs through the library's own
multi-device driver -- gwasdev_pairwise_scan_multi (host thread per device, ncclAllGather of the hit records) and
gwasdev_gtest_multi -- which is what a C++ caller of the reference's single function would use.

Nested sections: `marginal` (configs[1], marginal-scan GB/s against the HBM roofline, with its own e2e variants),
`pairwise_configs2` (configs[2]), `pairwise_missing_calls`, `biobank` (configs[4]), `configs0_file_to_statistics`.

--impl reference: the reference's own CPU implementation (oracle/_ref, the unmodified sources) of the same metric:
compute(computeBoost) on all host cores (one process per core), each step a bounded sample of configs[3]'s shape.

--dump-outputs DIR: after the timed steps, the headline's hit list of its last step (i, j, statistic; every rank's hits
merged) as DIR/hit_*.npy. The cohort comes from a fixed seed, so two builds run with the same arguments can be compared
file by file.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 20121127
MARGINAL = dict(n_snps=500_000, n_samples=10_000, n_case=5_000)       # BASELINE.json configs[1]
PAIRWISE = dict(n_snps=50_000, n_samples=4_000, n_case=2_000)         # BASELINE.json configs[2]
PAIRWISE_CFG3 = dict(n_snps=500_000, n_samples=10_000, n_case=5_000)  # BASELINE.json configs[3]: the headline
# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full captures (valid for these shapes only)
NCU_TRAFFIC = {
    ("marginal_scan_kernel", 500_000, 10_000): (1.2930e9, "profiles/r1k_marginal_scan_full.md"),
    ("pair_screen_mma_kernel", 50_000, 4_000): (5.19e9, "profiles/r2w_pair_screen_mma_cfg2_full.md"),
    ("pair_screen_mma_kernel", 500_000, 10_000): (1.843e12, "profiles/r2w_pair_screen_mma_cfg3_whole_metrics.md"),
}
CPU_MARGINAL_SAMPLE_SNPS = 2_000
CPU_PAIRWISE_SAMPLE_SNPS = 1_500     # per process and step in the reference arm: 1 124 250 pairs
CPU_BASELINE_SAMPLE_SNPS = 4_000     # cpu_baseline of the GPU arm (one core, ~15 s): 7 998 000 pairs
DUMP_BYTES = 64_000_000             # --dump-outputs budget, .npy headers included


def dump_outputs(out_dir, columns):
    """--dump-outputs: equal-length columns of one result as out_dir/<name>.npy in float64, plus row_count.npy (the full
    length). A result larger than DUMP_BYTES keeps a seeded sample of its rows, in order, and their indices (rows.npy), so
    that the files of two builds run with the same arguments can be compared one by one."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(next(iter(columns.values())))
    out = {name: np.asarray(col, np.float64) for name, col in columns.items()}
    keep = (DUMP_BYTES - 4096) // (8 * (len(out) + 1))
    if n > keep:
        rows = np.sort(np.random.default_rng(SEED).choice(n, keep, replace=False))
        out = {name: col[rows] for name, col in out.items()}
        out["rows"] = rows.astype(np.float64)
    out["row_count"] = np.array([n], np.float64)
    for name, col in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), col)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel, M, N):
    t = NCU_TRAFFIC.get((kernel, M, N))
    return (t[0], t[1]) if t else (None, None)


class ClockSampler:
    """SM clock, power and clock-event (throttle) reasons sampled DURING the timed region (B200_PROFILING.md recipe).
    Timed regions here run from milliseconds to a minute; `nvidia-smi -lms` cannot resolve the short ones, so the same
    NVML counters nvidia-smi prints are polled in-process (pynvml, ~1 ms period); nvidia-smi is the fallback."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, gpu_index: int, uuid: str | None = None):
        self.idx, self.uuid, self.rows, self.proc, self.nvml, self.source = gpu_index, uuid, [], None, None, None
        self._stop = threading.Event()

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            if self.uuid:
                try:
                    h = pynvml.nvmlDeviceGetHandleByUUID(self.uuid if self.uuid.startswith("GPU-") else "GPU-" + self.uuid)
                except Exception:
                    h = None
            if h is None:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
                ids = [v for v in vis.split(",") if v.strip().isdigit()]
                h = pynvml.nvmlDeviceGetHandleByIndex(int(ids[self.idx]) if self.idx < len(ids) else self.idx)
            self.nvml, self.handle, self.source = pynvml, h, "nvml"
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            threading.Thread(target=self._poll, daemon=True).start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi"
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _poll(self):
        nv, h = self.nvml, self.handle
        reasons_fn = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self._stop.is_set():
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                mask = int(reasons_fn(h))
                watts = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                self.rows.append((time.perf_counter(), [str(self.idx), sm, self.max_sm, watts, mask]))
            except Exception:
                pass
            time.sleep(0.001)

    def _pump(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            try:
                mask = sum(bit for (bit, _), v in zip(self.REASONS, f[4:8]) if v.lower().startswith("active"))
                self.rows.append((time.perf_counter(), [f[0], float(f[1]), float(f[2]), float(f[3]), mask]))
            except (ValueError, IndexError):
                pass

    def window(self, t0, t1):
        rows = [r for t, r in self.rows if t0 <= t <= t1]
        where = "timed region"
        if not rows:   # region shorter than one sampling period: the nearest samples around it
            rows = [r for _, r in sorted(self.rows, key=lambda tr: abs(tr[0] - 0.5 * (t0 + t1)))[:3]]
            where = "nearest samples to the timed region"
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(r[1] for r in rows)
        mask = 0
        for r in rows:
            mask |= r[4]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": rows[0][2], "reasons": sorted(n for b, n in self.REASONS if mask & b),
                "samples": len(rows), "power_w_max": round(max(r[3] for r in rows), 1), "source": self.source, "window": where}

    def stop(self):
        self._stop.set()
        if self.proc:
            self.proc.terminate()


def bind_to_gpu_numa_node(torch, local):
    """One process per GPU: run this rank's host thread on the CPUs next to its GPU (NVML's ideal affinity), so that the
    pinned host buffers of the e2e paths land on that NUMA node instead of wherever torchrun started the process."""
    try:
        import pynvml
        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(local).uuid)
        h = pynvml.nvmlDeviceGetHandleByUUID(uuid if uuid.startswith("GPU-") else "GPU-" + uuid)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return sorted(os.sched_getaffinity(0))
    except Exception:
        return None


class Ctx:
    """Per-process handles shared by the sections."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        import libgwaspp_b200 as gw
        self.args, self.torch, self.dist, self.gw = args, torch, dist, gw
        self.rank = int(os.environ.get("RANK", 0))
        self.world = int(os.environ.get("WORLD_SIZE", 1))
        self.local = int(os.environ.get("LOCAL_RANK", 0))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU arm)")
        torch.cuda.set_device(self.local)
        self.numa = bind_to_gpu_numa_node(torch, self.local)
        self.cpu_group = None
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.cpu_group = dist.new_group(backend="gloo")      # waits that must not occupy a GPU (single-process e2e on rank 0)
        self.stream = torch.cuda.current_stream()
        self.peaks, self.peak_src = measured_peaks()
        try:
            uuid = str(torch.cuda.get_device_properties(self.local).uuid)
        except Exception:
            uuid = None
        self.sampler = ClockSampler(self.local, uuid)
        if self.rank == 0:
            self.sampler.start()
        # roofline denominators measured once, on the idle device, before any section has warmed it up
        self.i8_burst, self.i8_sustained = gw.i8_peak(self.local)
        self.l2_read = {mb: gw.l2_read_peak(self.local, mb << 20, 12800 // mb) for mb in (16, 48)}   # GB/s, L2-resident buffers
        self.popc_peak, self.popc_clk = gw.popc_peak(self.local)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def cpu_barrier(self):
        if self.world > 1:
            self.dist.barrier(group=self.cpu_group)

    def reduce(self, x: float, op: str) -> float:
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return float(t.item())

    def clocks(self, t0, t1):
        return self.sampler.window(t0, t1) if self.rank == 0 else None


# ---------------------------------------------------------------------------------------------------
# pairwise screen (headline on configs[3]; nested on configs[2])
# ---------------------------------------------------------------------------------------------------
def pairwise_section(cx: Ctx, shape, K, W, label, headline):
    torch, gw, rank, world, local = cx.torch, cx.gw, cx.rank, cx.world, cx.local
    from libgwaspp_b200 import multi_gpu as mg
    M, N, NCASE = shape["n_snps"], shape["n_samples"], shape["n_case"]
    st = gw.GenoStore(M, N, device=local)
    st.set_stream(cx.stream.cuda_stream)
    st.simulate(SEED)                                          # the store is replicated on every rank
    pheno = gw.simulate_phenotype(SEED, N, NCASE)
    case_mask, ctrl_mask = gw.stream_masks(pheno)
    st.select_case_control(case_mask=case_mask, ctrl_mask=ctrl_mask)
    cap = 1 << 21
    d_hits = torch.empty((cap, 2), dtype=torch.int64, device="cuda")     # 16-byte gwasdev_hit records

    def step():
        n, stats = st.pairwise_scan(30.0, shard=rank, n_shards=world, capacity=cap, hits=d_hits, on_device=True)
        gathered = None
        if world > 1:   # hit gather over NCCL: counts, then the padded hit buffers (one collective each)
            counts = mg.gather_counts(int(n), world, torch.device("cuda", local))
            gathered = (counts, mg.gather_records(d_hits[:max(1, max(counts))], world))
            n = int(sum(counts))
        return n, stats, gathered

    for _ in range(W):
        step()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cx.barrier()
    l0, t0 = gw.launch_count(), time.perf_counter()
    ev0.record(cx.stream)
    screen_ms, pairs, cells, n_hits, cand, engine, tiles = [], 0, 0, 0, 0, 0, 0
    for _ in range(K):
        n_hits, s, gathered = step()
        screen_ms.append(s.screen_ms)
        pairs, cells, cand, engine, tiles = s.pairs_tested, s.word_cells, s.candidates, s.engine, s.tiles
    ev1.record(cx.stream)
    cx.barrier()
    t1, launches = time.perf_counter(), gw.launch_count() - l0
    if headline and cx.args.dump_outputs and rank == 0:
        if gathered is None:
            hits = np.ascontiguousarray(d_hits[:n_hits].cpu().numpy()).view(gw.HIT_DTYPE).reshape(-1)
        else:
            counts, recs = gathered
            hits = mg.merge_hits([mg.tensor_to_hits(recs[r], c) for r, c in enumerate(counts)])
        dump_outputs(cx.args.dump_outputs, {"hit_i": hits["i"], "hit_j": hits["j"], "hit_stat": hits["stat"]})
    ms_per_step = cx.reduce(ev0.elapsed_time(ev1), "max") / K
    total_pairs = cx.reduce(float(pairs), "sum")
    value = total_pairs / (ms_per_step * 1e-3)
    k_ms = float(np.mean(screen_ms))
    clocks = cx.clocks(t0, t1)
    # rooflines of the dominant kernel (this rank's launch): int8 MACs against the measured tensor peak, and the north
    # star's popcount view (4 AND+POPC word-cells per 32 samples per pair)
    macs = float(pairs) * 4.0 * N
    tops = 2.0 * macs / (k_ms * 1e-3) / 1e12
    burst, sustained = cx.i8_burst, cx.i8_sustained
    # a kernel timed inside a long step is held against the sustained figure, a short launch timed alone against the burst
    peak = sustained if k_ms > 50.0 else burst
    peak_cells, clk = cx.popc_peak, cx.popc_clk
    traffic, traffic_src = ncu_traffic("pair_screen_mma_kernel", M, N) if (engine == 2 and world == 1) else (None, None)
    kernel = {2: "pair_screen_mma_kernel (tcgen05.mma cta_group::2 kind::i8)", 1: "pair_screen_kernel<false> (AND+POPC)"}.get(engine, "?")
    roofline = {
        "bound": "tensor", "achieved": round(tops, 1), "peak": round(peak, 1), "unit": "TOP/s (int8, 2 ops per MAC)",
        "frac": round(tops / peak, 4), "traffic": traffic, "traffic_source": traffic_src, "kernel": kernel, "kernel_ms": round(k_ms, 3),
        "peak_source": f"gwasdev_i8_peak in this process: the kernel's own tcgen05.mma.cta_group::2.kind::i8 (M 256, N 256, K 32) on operands resident "
                       f"in shared memory; burst {burst:.0f}, sustained {sustained:.0f} TOP/s (nominal dense int8 4 500; 2 x MEASURED_PEAKS bf16 = "
                       f"{2 * float(cx.peaks.get('bf16_tflops', 0)):.0f})",
        "algorithmic_macs_per_launch": int(macs),
        "int_popc": {"achieved": round(cells / (k_ms * 1e-3) / 1e12, 4), "peak": round(peak_cells / 1e12, 4),
                     "unit": "T word-cells/s (32-bit AND+POPC)", "frac": round(cells / (k_ms * 1e-3) / peak_cells, 4),
                     "algorithmic_word_cells_per_launch": int(cells),
                     "peak_source": f"register-only __popc microbenchmark in this process (clock attr {clk:.0f} MHz); nominal 148 x 16 x 1.965 GHz = 4.65",
                     "note": "north star's popcount roofline; above 1 because the counting runs as an int8 GEMM on the tensor cores"},
    }
    if engine == 2:
        # what the kernel actually runs into: every tile pulls 2 x 256 operand rows from L2 (128 MAC per byte, 18.6 TB/s at the full tensor
        # rate); the cap is what plain 128-bit loads past L1 get out of an L2-resident buffer on this device (gwasdev_l2_read_peak)
        kb = (N + 127) // 128 * 128
        cap = max(cx.l2_read.values()) / 1e3
        l2 = float(tiles) * 512.0 * kb / (k_ms * 1e-3) / 1e12
        roofline["l2_to_sm"] = {"achieved": round(l2, 2), "cap": round(cap, 2), "frac": round(l2 / cap, 4), "unit": "TB/s",
                                "operand_bytes_per_launch": int(tiles) * 512 * kb,
                                "cap_source": "gwasdev_l2_read_peak in this process (ld.global.cg.v4 over L2-resident buffers, one launch of many passes): "
                                              + ", ".join(f"{mb} MiB {v / 1e3:.2f} TB/s" for mb, v in cx.l2_read.items()),
                                "note": "operand bytes TMA moves from L2 to shared memory per launch / kernel time"}
    res = {
        "metric": "pairwise SNP x SNP tests/sec", "value": round(value, 1), "unit": "pairs/s", "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": round(ms_per_step, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "int8 one-hot operands, int32 counts (tcgen05), fp32 screen, fp64 re-score", "data": "synthetic",
        "hits": int(n_hits), "candidates": int(cand),
        "config": {"workload": f"{label}: exhaustive pairwise epistasis {NCASE}/{N - NCASE} samples x {M} SNPs "
                               f"({M * (M - 1) // 2} pairs), 3x3x2 contingency + KSA statistic, threshold 30, hit list sorted by (i, j)",
                   "generator": "simulate_data.cpp restated, affy6 panel of maf_spectrum.tab, seed 20121127",
                   "engine": {2: "tensor cores", 1: "AND+POPC"}.get(engine, "?"),
                   "l2": f"inputs larger than L2 ({2.0 * M * ((NCASE + 127) // 128 + (N - NCASE + 127) // 128) * 128 / 1e6:.0f} MB operand matrix streamed "
                         "many times per step vs 126 MB L2)",
                   "parallelism": f"128x128 SNP tile pairs dealt in runs of 64 over {world} rank(s); NCCL all_gather of the hit records"},
        "roofline": roofline, "gpu_launches": int(launches), "clocks": clocks,
    }
    # ---- e2e: computeBoost call surface with host buffers
    e2e_steps = 3 if headline else max(3, min(K, 5))
    res["e2e_torchrun"] = None
    if world == 1:
        for it in range(1 + e2e_steps):
            if it == 1:
                cx.barrier()
                te0 = time.perf_counter()
            st.select_case_control(case_mask=case_mask, ctrl_mask=ctrl_mask)
            hits, s = st.pairwise_scan(30.0)
            if len(hits):
                st.gtest(hits["i"], hits["j"])
        cx.barrier()
        e2e_s = (time.perf_counter() - te0) / e2e_steps
        res["e2e"] = {"value": round(total_pairs / e2e_s, 1), "unit": "pairs/s", "ms_per_step": round(e2e_s * 1e3, 2),
                      "h2d_bytes_per_step": int(2 * 2 * st.P + 8 * len(hits)), "d2h_bytes_per_step": int(32 * len(hits)), "steps": e2e_steps,
                      "hits": int(len(hits)),
                      "what": "gwasdev_select_case_control(host masks) + gwasdev_pairwise_scan (margins, operand build, screen, fp64 re-score, "
                              "sort; hits to host) + gwasdev_gtest (host pairs in, statistic and z out): computeBoost's surface"}
        st.close()
    else:
        # (a) every rank its shard, torch.distributed gather -- the per-rank form of the same surface
        for it in range(1 + e2e_steps):
            if it == 1:
                cx.barrier()
                te0 = time.perf_counter()
            st.select_case_control(case_mask=case_mask, ctrl_mask=ctrl_mask)
            hits, s = st.pairwise_scan(30.0, shard=rank, n_shards=world)
            if len(hits):
                st.gtest(hits["i"], hits["j"])
            mg.gather_hits(hits)
        cx.barrier()
        e2e_s = cx.reduce((time.perf_counter() - te0) / e2e_steps, "max")
        res["e2e_torchrun"] = {"value": round(total_pairs / e2e_s, 1), "unit": "pairs/s", "ms_per_step": round(e2e_s * 1e3, 2), "steps": e2e_steps,
                               "what": "per rank: select + pairwise_scan(shard) + gtest of its own hits, host buffers; all_gather of the hit lists"}
        st.close()
        del d_hits
        torch.cuda.empty_cache()
        # (b) ONE process, all GPUs, through the library's multi-device driver (rank 0; the others wait on a CPU barrier)
        cx.cpu_barrier()
        e2e = None
        if rank == 0:
            try:
                e2e = single_process_e2e(cx, shape, e2e_steps, total_pairs, case_mask, ctrl_mask)
            except Exception as exc:                   # keep the line; say what happened
                e2e = dict(res["e2e_torchrun"], h2d_bytes_per_step=0, d2h_bytes_per_step=0,
                           error=f"single-process multi-device e2e failed: {exc!r}; value is the per-rank form")
        cx.cpu_barrier()
        res["e2e"] = e2e
    return res


def single_process_e2e(cx: Ctx, shape, steps, total_pairs, case_mask, ctrl_mask):
    gw, world = cx.gw, cx.world
    M, N = shape["n_snps"], shape["n_samples"]
    t_setup = time.perf_counter()
    first = gw.GenoStore(M, N, device=0)
    first.simulate(SEED)
    stores = [first] + [first.replicate(d) for d in range(1, world)]      # the table travels device to device
    t_setup = time.perf_counter() - t_setup
    hits = None
    for it in range(1 + steps):
        if it == 1:
            for s in stores:
                s.synchronize()
            t0 = time.perf_counter()
        for s in stores:
            s.select_case_control(case_mask=case_mask, ctrl_mask=ctrl_mask)
        hits, _ = gw.pairwise_scan_multi(stores, 30.0, capacity=1 << 21)
        if len(hits):
            gw.gtest_multi(stores, hits["i"], hits["j"])
    e2e_s = (time.perf_counter() - t0) / steps
    for s in stores:
        s.close()
    return {"value": round(total_pairs / e2e_s, 1), "unit": "pairs/s", "ms_per_step": round(e2e_s * 1e3, 2), "steps": steps,
            "h2d_bytes_per_step": int(world * 2 * 2 * first.P + 8 * len(hits)), "d2h_bytes_per_step": int(32 * len(hits)), "hits": int(len(hits)),
            "replication_s": round(t_setup, 3),
            "what": f"ONE host process, {world} GPUs: gwasdev_select_case_control on every device (host masks) + gwasdev_pairwise_scan_multi "
                    "(host thread per device: margins, operands, its shard of the screen, re-score, sort; ncclAllGather of the hit records; "
                    "merge on device 0; hits to host) + gwasdev_gtest_multi: computeBoost's surface as a C++ caller reaches it"}


def plant_interactions(gw, st, pheno, n_pairs):
    """Case-only dependencies between a few pairs of common SNPs, so that a screen at threshold 30 has hits: the case
    columns of SNP b are overwritten with those of SNP a (the construction of tests/helpers.planted_cohort, on packed rows)."""
    whole = st.counts(0)
    common = np.flatnonzero((whole[:, 2] > 0.04 * st.n_samples) & (whole[:, 0] > 0.04 * st.n_samples))[: 2 * n_pairs]
    case_mask, _ = gw.stream_masks(pheno)
    P = st.P
    for k in range(len(common) // 2):
        a, b = int(common[2 * k]), int(common[2 * k + 1])
        ra, rb = st.get_rows(a, 1)[0], st.get_rows(b, 1)[0]
        for pl in range(2):
            sl = slice(1 + pl * P, 1 + (pl + 1) * P)
            rb[sl] = (rb[sl] & ~case_mask) | (ra[sl] & case_mask)
        rb[0] = ra[0]                                        # same labels as the source row
        st.put_rows(rb[None, :], b)
    return len(common) // 2


def pairwise_missing_gpu(cx: Ctx):
    """configs[2] with 1 % of the calls missing (what real genotype data looks like): every 64-SNP block has missing calls,
    so the whole screen takes the reference's 9-cell branch -- here the four-plane tensor-core kernel; the 9-cell AND+POPC
    kernel it replaces is timed beside it. Threshold 30 as everywhere; the cohort carries planted case-only dependencies
    so that the candidate / re-score path has work."""
    gw, local = cx.gw, cx.local
    M, N, NCASE = PAIRWISE["n_snps"], PAIRWISE["n_samples"], PAIRWISE["n_case"]
    res = {"workload": f"configs[2] shape with 1 % missing calls: {NCASE}/{N - NCASE} samples x {M} SNPs ({M * (M - 1) // 2} pairs), "
                       "9-cell tables (compressed_genotype_table5.cpp:1000-1067) + KSA statistic, threshold 30"}
    with gw.GenoStore(M, N, device=local) as st:
        st.set_stream(cx.stream.cuda_stream)
        st.simulate(SEED, missing_rate=0.01)
        pheno = gw.simulate_phenotype(SEED, N, NCASE)
        res["planted_pairs"] = plant_interactions(gw, st, pheno, 16)
        st.select_case_control(pheno)
        for name, engine in (("tensor_cores_four_planes", 0), ("and_popc_nine_cells", 1)):
            st.set_pair_engine(engine)
            ms, hits = [], None
            for it in range(4):
                hits, s = st.pairwise_scan(30.0)
                if it:
                    ms.append(s.screen_ms)
            k_ms = float(np.mean(ms))
            res[name] = {"value": round(s.pairs_tested / (k_ms * 1e-3), 1), "unit": "pairs/s", "kernel_ms": round(k_ms, 3),
                         "tiles_with_missing_calls": int(s.tiles_nine_cell), "candidates": int(s.candidates), "hits": int(len(hits))}
        cells = 9 * ((NCASE + 31) // 32 + (N - NCASE + 31) // 32)
        peak = cx.popc_peak
        res["and_popc_nine_cells"]["frac_of_popc_roofline"] = round(res["and_popc_nine_cells"]["value"] * cells / peak, 4)
        res["tensor_cores_four_planes"]["x_popc_roofline"] = round(res["tensor_cores_four_planes"]["value"] * cells / peak, 4)
        res["same_hits"] = res["and_popc_nine_cells"]["hits"] == res["tensor_cores_four_planes"]["hits"]
        # the four-plane kernel's own bound: 256 A rows + 192 B rows (three of the four planes) per 64 x 64-SNP tile from L2
        t4 = res["tensor_cores_four_planes"]
        kb = (N + 127) // 128 * 128
        byts = float(t4["tiles_with_missing_calls"]) * (256 + 192) * kb
        cap = max(cx.l2_read.values()) / 1e3
        t4["l2_to_sm"] = {"achieved": round(byts / (t4["kernel_ms"] * 1e-3) / 1e12, 2), "cap": round(cap, 2), "unit": "TB/s",
                          "frac": round(byts / (t4["kernel_ms"] * 1e-3) / 1e12 / cap, 4), "operand_bytes_per_launch": int(byts),
                          "mma_floor_ms": round(t4["tiles_with_missing_calls"] / 74.0 * (kb // 32) * 96 / 1.965e6, 2),
                          "note": "cap = gwasdev_l2_read_peak in this process; mma_floor_ms = tiles / 74 CTA pairs x (row bytes / 32) MMAs x 96 clk "
                                  "(M 256, N 192, K 32) at 1 965 MHz"}
    return res


# ---------------------------------------------------------------------------------------------------
# marginal scan (configs[1]); weak scaling: every rank scans its own 500 000-SNP shard
# ---------------------------------------------------------------------------------------------------
def marginal_section(cx: Ctx, K, W):
    torch, gw, rank, world, local = cx.torch, cx.gw, cx.rank, cx.world, cx.local
    args = cx.args
    M, N, NCASE = args.snps or MARGINAL["n_snps"], args.samples or MARGINAL["n_samples"], args.cases or MARGINAL["n_case"]
    st = gw.GenoStore(M, N, device=local)
    st.set_stream(cx.stream.cuda_stream)
    st.simulate(SEED + rank)                                   # each rank owns a different 500k-SNP shard
    pheno = gw.simulate_phenotype(SEED, N, NCASE)
    case_mask, ctrl_mask = gw.stream_masks(pheno)
    d_counts = torch.empty((M, 8), dtype=torch.int32, device="cuda")
    d_stats = torch.empty((M, 8), dtype=torch.float64, device="cuda")
    bytes_per_step = M * N / 4.0                               # algorithmic bytes (2 bits per genotype)

    def timed(fn, steps, warm):
        for _ in range(warm):
            fn()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        cx.barrier()
        l0, t0 = gw.launch_count(), time.perf_counter()
        ev0.record(cx.stream)
        for _ in range(steps):
            fn()
        ev1.record(cx.stream)
        cx.barrier()
        t1 = time.perf_counter()
        return cx.reduce(ev0.elapsed_time(ev1), "max") / steps, gw.launch_count() - l0, (t0, t1)

    def kernel_ms(fn, reps=10):
        out = []
        for _ in range(reps):
            fn()
            out.append(st.last_scan_ms())
        return float(np.mean(out))

    def scan():
        st.marginal_scan_into(0, M, counts=d_counts, stats=d_stats)

    res = {"workload": f"configs[1]: {NCASE} cases / {N - NCASE} controls x {M} SNPs per GPU, marginal allelic + genotypic chi-square scan "
                       "(counts + statistics written)", "scaling": "weak", "n_gpus": world,
           "l2": f"inputs larger than L2 ({bytes_per_step / 1e6:.0f} MB streamed per step vs 126 MB L2)"}
    # (1) K1 on the compacted rows (K0 run once, eagerly): the reference's pre-selected overload
    st.set_select_mode(True)
    st.select_case_control(case_mask=case_mask, ctrl_mask=ctrl_mask)
    ms, launches, win = timed(scan, K, W)
    k_ms = kernel_ms(scan)
    achieved = bytes_per_step / (k_ms * 1e-3) / 1e9
    traffic, traffic_src = ncu_traffic("marginal_scan_kernel", M, N)
    res["compacted"] = {
        "value": round(world * bytes_per_step / (ms * 1e-3) / 1e9, 1), "unit": "GB/s", "ms_per_step": round(ms, 4), "steps": K, "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": cx.peaks["hbm_gbs"], "unit": "GB/s", "frac": round(achieved / cx.peaks["hbm_gbs"], 4),
                     "traffic": traffic, "traffic_source": traffic_src, "kernel": "marginal_scan_kernel", "kernel_ms": round(k_ms, 4),
                     "peak_source": cx.peak_src, "algorithmic_bytes_per_launch": bytes_per_step},
        "clocks": cx.clocks(*win)}
    ref_counts = d_counts.clone()
    # (2) K1' on the raw rows: selection fused into the scan, row totals cached per table (what a re-selection runs; no K0)
    st.set_select_mode(False)
    st.select_case_control(case_mask=case_mask, ctrl_mask=ctrl_mask)
    scan()                                                     # first scan of the table writes the row totals
    def reselect_scan():
        st.select_case_control(case_mask=case_mask, ctrl_mask=ctrl_mask)
        scan()
    ms2, launches2, _ = timed(reselect_scan, K, W)
    k_ms2 = kernel_ms(reselect_scan)
    ach2 = bytes_per_step / (k_ms2 * 1e-3) / 1e9
    assert torch.equal(d_counts, ref_counts), "masked scan differs from the compacted scan"
    res["fused_select_scan"] = {
        "value": round(world * bytes_per_step / (ms2 * 1e-3) / 1e9, 1), "unit": "GB/s", "ms_per_step": round(ms2, 4), "gpu_launches": int(launches2),
        "what": "gwasdev_select_case_control (masks from host) + marginal_scan_masked_kernel MODE 2 on the raw rows, device outputs",
        "roofline": {"bound": "hbm", "achieved": round(ach2, 1), "peak": cx.peaks["hbm_gbs"], "unit": "GB/s", "frac": round(ach2 / cx.peaks["hbm_gbs"], 4),
                     "kernel": "marginal_scan_masked_kernel<MODE 2>", "kernel_ms": round(k_ms2, 4)}}
    # (3) e2e: select_cc_maf's call surface with HOST buffers, three output forms
    h_counts = torch.empty((M, 8), dtype=torch.int32, pin_memory=True)
    h_stats = torch.empty((M, 8), dtype=torch.float64, pin_memory=True)
    h_compact = torch.empty((M, 4), dtype=torch.int64, pin_memory=True)        # 32-byte gwasdev_snp_compact records
    h_sig = torch.empty((1 << 16, 6), dtype=torch.int64, pin_memory=True)      # 48-byte gwasdev_sig_snp records
    e2e_steps = max(3, min(K, 10))

    def e2e(fn):
        for it in range(2 + e2e_steps):
            if it == 2:
                cx.barrier()
                t0 = time.perf_counter()
            st.select_case_control(case_mask=case_mask, ctrl_mask=ctrl_mask)
            fn()
        cx.barrier()
        return cx.reduce((time.perf_counter() - t0) / e2e_steps, "max")

    n_sig = [0]
    t_full = e2e(lambda: st.marginal_scan_into(0, M, counts=h_counts, stats=h_stats, on_device=False))
    t_compact = e2e(lambda: n_sig.__setitem__(0, st.marginal_scan_compact_into(0, M, records=h_compact, p_threshold=5e-8, sig=h_sig,
                                                                                  sig_capacity=1 << 16, on_device=False)))
    t_sig = e2e(lambda: st.marginal_scan_compact_into(0, M, records=None, p_threshold=5e-8, sig=h_sig, sig_capacity=1 << 16, on_device=False))
    assert torch.equal(h_counts, ref_counts.cpu()) and int(h_counts[:, :4].sum(1).min()) == NCASE
    rec = h_compact.numpy().view(gw.COMPACT_DTYPE).reshape(-1)
    assert np.array_equal(rec["cases"].astype(np.int32), h_counts.numpy()[:, :4]) and np.array_equal(rec["controls"].astype(np.int32), h_counts.numpy()[:, 4:])
    h2d = int(16 * ((st.P // 2 + 3) // 4 * 4))               # the four class masks as 32-bit words
    host = (f"{cx.numa[0]}-{cx.numa[-1]} ({len(cx.numa)}, NVML affinity of the GPU)" if cx.numa else "unbound")

    def e2e_obj(t, d2h, what):
        return {"value": round(world * bytes_per_step / t / 1e9, 2), "unit": "GB/s", "ms_per_step": round(t * 1e3, 3), "steps": e2e_steps,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(d2h), "what": what}
    res["e2e"] = e2e_obj(t_compact, M * 32 + 48 * n_sig[0],
                         "gwasdev_select_case_control(host masks) + gwasdev_marginal_scan_compact(pinned host outputs): 32 bytes per SNP (u16 genotype "
                         "counts of both classes + allelic / genotypic chi-square and p-value in fp32) and the SNPs with p < 5e-8 in fp64; pieces' D2H "
                         "copies overlap the next piece's scan")
    res["e2e"]["significant_snps"] = int(n_sig[0])
    res["e2e"]["host_cpus"] = host
    res["e2e_full_records"] = e2e_obj(t_full, M * 96, "the same with 96 bytes per SNP: u32 counts + gwasdev_snp_stats in fp64 (round 1's e2e)")
    res["e2e_significant_only"] = e2e_obj(t_sig, 48 * n_sig[0], "the same returning only the SNPs with p < 5e-8 (48-byte fp64 records)")
    st.close()
    del d_counts, d_stats, h_counts, h_stats, h_compact, h_sig, ref_counts
    torch.cuda.empty_cache()
    return res


def configs0_file_to_statistics(gw, local):
    """BASELINE configs[0] -- 1 000 cases / 1 000 controls x 10 000 SNPs, the case the reference runs on a CPU -- from the
    genotype FILE to the per-SNP statistics on the host: 80 MB of TPED text -> device loader -> selection -> scan -> host
    results, next to the reference doing the same with its own reader and select_cc_maf on one host core (oracle/_ref)."""
    import tempfile
    import oracle
    M, N, NCASE = 10_000, 2_000, 1_000
    pheno = gw.simulate_phenotype(SEED, N, NCASE)
    with gw.GenoStore(M, N, device=local) as st:            # the cohort: device generator -> rows -> text
        st.simulate(SEED)
        rows = st.get_rows()
        st.select_case_control(pheno)
        want = st.marginal_scan(mi=False)["counts"]
    P = (rows.shape[1] - 1) // 2
    p1 = np.unpackbits(np.ascontiguousarray(rows[:, 1:1 + P]).view(np.uint8), axis=1, bitorder="little")[:, :N]
    p2 = np.unpackbits(np.ascontiguousarray(rows[:, 1 + P:]).view(np.uint8), axis=1, bitorder="little")[:, :N]
    lut = np.array([np.frombuffer(t, np.uint8).view(np.uint32)[0] for t in (b"0\t0\t", b"A\tA\t", b"A\tC\t", b"C\tC\t")], np.uint32)
    code = p1 + 2 * p2
    d = tempfile.mkdtemp()
    tped, tfam = os.path.join(d, "c0.tped"), os.path.join(d, "c0.tfam")
    with open(tped, "wb") as f:
        for r in range(M):
            f.write(b"0\trs%d\t0\t%d\t" % (r, r) + lut[code[r]].view(np.uint8).tobytes()[:-1] + b"\n")
    with open(tfam, "w") as f:
        for i, ph in enumerate(pheno):
            f.write(f"F{i}\tI{i}\t0\t0\t1\t{int(ph)}\n")
    res = {"workload": f"configs[0]: {NCASE} cases / {N - NCASE} controls x {M} SNPs, {os.path.getsize(tped) / 1e6:.1f} MB TPED file (page cache) "
                       "-> per-SNP case/control counts + statistics on the host"}
    best = None
    for _ in range(3):
        t0 = time.perf_counter()
        with gw.GenoStore.from_tped(tped, device=local) as st:     # table sized and loaded in one pass over the file
            t2 = time.perf_counter()
            st.select_case_control(pheno)
            got = st.marginal_scan(mi=False)
            t3 = time.perf_counter()
        cur = {"create_load_ms": round(1e3 * (t2 - t0), 2), "select_scan_ms": round(1e3 * (t3 - t2), 2),
               "total_ms": round(1e3 * (t3 - t0), 2)}
        if best is None or cur["total_ms"] < best["total_ms"]:
            best = cur
    assert np.array_equal(got["counts"], want), "counts from the loaded file differ from the generated cohort's"
    res["b200"] = best
    if oracle.have_ref():
        t0 = time.perf_counter()
        R = oracle.Ref(tped=tped, tfam=tfam, level=5)
        t1 = time.perf_counter()
        R.run("select_cc_maf")
        t2 = time.perf_counter()
        ref_counts = np.stack([R.cc_dist(r, 1)[0] for r in range(0, M, 101)])
        assert np.array_equal(ref_counts, want[::101]), "the reference's counts differ"
        res["reference"] = {"load_ms": round(1e3 * (t1 - t0), 1), "select_cc_maf_ms": round(1e3 * (t2 - t1), 1),
                            "total_ms": round(1e3 * (t2 - t0), 1), "cores": 1, "kind": "reference",
                            "what": "TpedGenotypeFile + TfamAnnotationFile readers, compute(select_cc_maf) at --comp-level 5"}
    for fn in (tped, tfam):
        os.remove(fn)
    os.rmdir(d)
    return res


def biobank_gpu(cx: Ctx):
    """BASELINE configs[4]: 200 000 samples x 1 000 000 SNPs. (a) HBM-resident: one scan launch over the whole 50 GB table,
    through the masks on the raw rows (no second copy of the table) and on the compacted rows. (b) streamed in sample
    blocks: raw rows of one block at a time from pinned host memory -> H2D -> counts added into a device accumulator,
    statistics from the summed counts at the end; bounded to --bb-stream-snps SNPs so that the pinned host copy stays small
    (the streamed rate is PCIe-bound and scales linearly in SNPs)."""
    args, gw, torch, local = cx.args, cx.gw, cx.torch, cx.local
    t_section = time.perf_counter()
    N, NCASE, M = 200_000, 100_000, args.bb_snps
    res = {"workload": f"configs[4]: {NCASE} cases / {N - NCASE} controls x {M} SNPs"}
    pheno = gw.simulate_phenotype(SEED, N, NCASE)
    with gw.GenoStore(M, N, device=local) as st:
        st.set_stream(cx.stream.cuda_stream)
        st.simulate(SEED)
        d_counts = torch.empty((M, 8), dtype=torch.int32, device="cuda")
        d_stats = torch.empty((M, 8), dtype=torch.float64, device="cuda")

        def run(reps=8):
            kms = []
            for it in range(reps):
                st.marginal_scan_into(0, M, counts=d_counts, stats=d_stats)
                if it >= 3:
                    kms.append(st.last_scan_ms())
            k = float(np.mean(kms))
            g = M * N / 4.0 / (k * 1e-3) / 1e9
            return {"value": round(g, 1), "unit": "GB/s", "kernel_ms": round(k, 3), "bytes": M * N / 4.0,
                    "frac_of_hbm_peak": round(g / cx.peaks["hbm_gbs"], 4), "peak_source": cx.peak_src}
        st.select_case_control(pheno)
        res["resident_raw_rows"] = dict(run(), kernel="marginal_scan_masked_kernel<MODE 2> (row totals cached; 50 GB resident, no compacted copy)")
        masked_counts = d_counts[: args.bb_stream_snps].clone()
        st.set_select_mode(True)
        st.select_case_control(pheno)
        res["resident"] = dict(run(), kernel="marginal_scan_kernel on the compacted rows (a second 50 GB copy)")
        assert torch.equal(masked_counts, d_counts[: args.bb_stream_snps]), "masked and compacted scans differ"
        ref_counts = d_counts[: args.bb_stream_snps].cpu().numpy().view(np.uint32)
        del d_counts, d_stats, masked_counts
    torch.cuda.empty_cache()
    # streamed: host copy of the first Ms SNPs, block by block
    Ms, B = args.bb_stream_snps, args.bb_block
    blocks = [(s0, min(B, N - s0)) for s0 in range(0, N, B)]
    host = []
    for s0, nb in blocks:                                   # setup (untimed): generate each block, keep its raw rows pinned
        with gw.GenoStore(Ms, nb, device=local) as st:
            st.simulate_block(SEED, s0, N)
            rows = torch.from_numpy(st.get_rows()).pin_memory()
            host.append(rows)
    acc = torch.zeros((Ms, 8), dtype=torch.int32, device="cuda")
    stores = {nb: gw.GenoStore(Ms, nb, device=local) for nb in {nb for _, nb in blocks}}
    times = []
    for rep in range(3):
        acc.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for (s0, nb), rows in zip(blocks, host):
            st = stores[nb]
            st.put_rows(rows.numpy())
            st.select_case_control(pheno[s0:s0 + nb])
            st.marginal_accumulate(acc, on_device=True)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    for st in stores.values():
        st.close()
    assert np.array_equal(acc.cpu().numpy().view(np.uint32), ref_counts), "streamed counts differ from the resident scan"
    t = min(times)
    h2d = sum(int(r.numel()) * 2 for r in host)
    res["streamed"] = {"value": round(Ms * N / 4.0 / t / 1e9, 2), "unit": "GB/s of 2-bit genotypes, end to end from pinned host memory",
                       "snps": Ms, "sample_blocks": len(blocks), "block_samples": B, "seconds": round(t, 4),
                       "h2d_bytes": h2d, "h2d_gbs": round(h2d / t / 1e9, 2),
                       "check": "summed counts bit-identical to the resident scan"}
    res["section_s"] = round(time.perf_counter() - t_section, 1)
    return res


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------
def gpu_arm(args):
    cx = Ctx(args)
    K, W = args.steps, args.warmup
    shape = dict(PAIRWISE_CFG3)
    label = "configs[3]"
    if args.pw_snps:                       # reduced shapes for development runs; the line says so
        shape = dict(n_snps=args.pw_snps, n_samples=args.pw_samples or shape["n_samples"], n_case=args.pw_cases or (args.pw_samples or shape["n_samples"]) // 2)
        label = "REDUCED development shape (not BASELINE configs[3])"
    out = pairwise_section(cx, shape, K, W, label, headline=True)
    if not args.headline_only:
        out["marginal"] = marginal_section(cx, max(K, 10), max(W, 3))
        out["pairwise_configs2"] = pairwise_section(cx, PAIRWISE, max(1, min(K, 10)), 3, "configs[2]", headline=False)
        if cx.world == 1:
            out["pairwise_missing_calls"] = pairwise_missing_gpu(cx)
            if not args.no_biobank:
                try:
                    out["biobank"] = biobank_gpu(cx)
                except Exception as exc:
                    out["biobank"] = {"error": repr(exc)}
    if cx.rank == 0:
        if cx.world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline_pairwise(shape["n_samples"], shape["n_case"], CPU_BASELINE_SAMPLE_SNPS)
            if not args.headline_only:
                out["marginal"]["cpu_baseline"] = cpu_baseline_marginal(MARGINAL["n_samples"], MARGINAL["n_case"], threads=1, steps=3)
                out["pairwise_configs2"]["cpu_baseline"] = cpu_baseline_pairwise(PAIRWISE["n_samples"], PAIRWISE["n_case"], CPU_PAIRWISE_SAMPLE_SNPS)
                out["configs0_file_to_statistics"] = configs0_file_to_statistics(cx.gw, cx.local)
        cx.sampler.stop()
        print(json.dumps(out))
    if cx.world > 1:
        cx.dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------
# CPU baselines (the reference itself when oracle/_ref is present, else the C port)
# ---------------------------------------------------------------------------------------------------
def _ref_marginal_sample(seed, n_snps, N, NCASE):
    import oracle
    O = oracle.Oracle()
    codes, pheno = O.simulate(seed, n_snps, N, NCASE)
    if oracle.have_ref():
        R = oracle.Ref(n_snps, N, 5)
        R.add_codes(codes)
        R.set_case_control(pheno)
        return "reference", R, None
    rows = O.pack_codes(codes)
    return "port", O, (rows, pheno, N)


def _marginal_step(kind, obj, extra):
    """one select_cc_maf-equivalent pass: (t_select, t_scan) seconds."""
    if kind == "reference":
        return obj.time_phase(0, 1), obj.time_phase(2, 1)
    rows, pheno, N = extra
    t0 = time.perf_counter()
    sel, nca, nco = obj.select(rows, N, pheno)
    t1 = time.perf_counter()
    obj.cc_counts_selected(sel, nca, nco)
    return t1 - t0, time.perf_counter() - t1


def cpu_baseline_marginal(N, NCASE, threads=1, steps=3):
    kind, obj, extra = _ref_marginal_sample(SEED, CPU_MARGINAL_SAMPLE_SNPS, N, NCASE)
    _marginal_step(kind, obj, extra)
    ts = [_marginal_step(kind, obj, extra) for _ in range(steps)]
    t_sel, t_scan = float(np.median([t[0] for t in ts])), float(np.median([t[1] for t in ts]))
    b = CPU_MARGINAL_SAMPLE_SNPS * N / 4.0
    return {"value": round(b / (t_sel + t_scan) / 1e9, 5), "unit": "GB/s", "cores": threads, "kind": kind,
            "sample": f"{CPU_MARGINAL_SAMPLE_SNPS} SNPs x {N} samples of the same cohort: selectCaseControl ({t_sel * 1e3:.1f} ms) + pre-selected per-SNP "
                      f"counts + MinorAlleleFrequency ({t_scan * 1e3:.1f} ms), i.e. select_cc_maf without its per-SNP timer / stream writes",
            "scan_only_value": round(b / t_scan / 1e9, 4)}


def _pairwise_sample(seed, n, N, NCASE):
    import oracle
    O = oracle.Oracle()
    codes, pheno = O.simulate(seed, n, N, NCASE)
    if oracle.have_ref():
        R = oracle.Ref(n, N, 5)
        R.add_codes(codes)
        R.set_case_control(pheno)
        return "reference", R, None
    return "port", O, (O.pack_codes(codes), pheno, N)


def _pairwise_step(kind, obj, extra):
    """one compute(computeBoost)-equivalent pass over the sample; seconds."""
    if kind == "reference":
        return obj.time_phase(3, 1)
    rows, pheno, N = extra
    t0 = time.perf_counter()
    sel, nca, nco = obj.select(rows, N, pheno)
    mar = obj.margins(sel, nca, nco)
    obj.boost_screen(sel, mar, nca, nco)
    return time.perf_counter() - t0


def cpu_baseline_pairwise(N, NCASE, n):
    kind, obj, extra = _pairwise_sample(SEED, n, N, NCASE)
    t = _pairwise_step(kind, obj, extra)
    pairs = n * (n - 1) // 2
    what = ("compute(computeBoost): selectCaseControl + computeMargins + pre-screen of every pair + G-test of the hits" if kind == "reference"
            else "oracle select + margins + boost_screen")
    return {"value": round(pairs / t, 1), "unit": "pairs/s", "cores": 1, "kind": kind,
            "sample": f"first {n} SNPs x {N} samples of the same cohort ({pairs} pairs): {what}, {t:.2f} s"}


# ---------------------------------------------------------------------------------------------------
# reference arm: the reference's CPU implementation of the headline metric on all host cores
# ---------------------------------------------------------------------------------------------------
def _ref_worker(widx, N, NCASE, n, warmup, steps, start_evt, q):
    kind, obj, extra = _pairwise_sample(SEED + 1000 + widx, n, N, NCASE)
    for _ in range(warmup):
        _pairwise_step(kind, obj, extra)
    q.put(("ready", widx, kind))
    start_evt.wait()
    t0 = time.perf_counter()
    for _ in range(steps):
        _pairwise_step(kind, obj, extra)
    q.put(("done", widx, time.perf_counter() - t0))


def reference_arm(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    import multiprocessing as mp
    import oracle
    oracle.build_oracle()
    shape = PAIRWISE_CFG3
    N, NCASE, n = args.pw_samples or shape["n_samples"], args.pw_cases or shape["n_case"], args.ref_snps or CPU_PAIRWISE_SAMPLE_SNPS
    cores = args.ref_procs or len(os.sched_getaffinity(0))
    warmup = args.warmup                  # a step costs ~2 s per process at this sample size
    ctx = mp.get_context("fork")
    q, evt = ctx.Queue(), ctx.Event()
    procs = [ctx.Process(target=_ref_worker, args=(w, N, NCASE, n, warmup, args.steps, evt, q)) for w in range(cores)]
    for p in procs:
        p.start()
    kind = "port"
    for _ in range(cores):
        _, _, kind = q.get()
    t0 = time.perf_counter()
    evt.set()
    times = [q.get()[2] for _ in range(cores)]
    wall = time.perf_counter() - t0
    for p in procs:
        p.join()
    pairs = n * (n - 1) // 2
    value = cores * args.steps * pairs / max(times)
    sample = (f"each of {cores} processes: {args.steps} steps of compute(computeBoost) -- selectCaseControl + computeMargins + pre-screen of every "
              f"pair + G-test of the hits -- over its own {n} SNPs x {N} samples ({pairs} pairs per step and process) of configs[3]'s shape")
    line = {
        "impl": "reference", "metric": "pairwise SNP x SNP tests/sec", "value": round(value, 1), "unit": "pairs/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": warmup,
        "ms_per_step": round(max(times) / args.steps * 1e3, 3), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u64 words + LUT popcount, fp64 statistic (reference)", "data": "synthetic",
        "config": {"workload": f"configs[3] shape: {NCASE} cases / {N - NCASE} controls, bounded sample of {n} SNPs ({pairs} pairs) per process and step; "
                               "the reference has no threads: one process per host core"},
        "cpu_baseline": {"value": round(value, 1), "unit": "pairs/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": round(value, 1), "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": round(wall, 2),
    }
    if not args.headline_only:
        line["marginal"] = {"impl": "reference", **cpu_baseline_marginal(MARGINAL["n_samples"], MARGINAL["n_case"], threads=1, steps=3)}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5,
                    help="timed passes of the headline (the nested sections keep their own counts: marginal max(steps, 10), "
                         "configs[2] min(steps, 10), fixed repetitions elsewhere)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--snps", type=int, default=0, help="marginal section: SNPs (default configs[1])")
    ap.add_argument("--samples", type=int, default=0)
    ap.add_argument("--cases", type=int, default=0)
    ap.add_argument("--pw-snps", type=int, default=0, help="development only: a reduced headline shape (the line is labelled as such)")
    ap.add_argument("--pw-samples", type=int, default=0)
    ap.add_argument("--pw-cases", type=int, default=0)
    ap.add_argument("--headline-only", action="store_true", help="skip the nested sections")
    ap.add_argument("--no-biobank", action="store_true", help="N = 1: skip the configs[4] biobank-scale section (needs ~110 GB of HBM, ~1 min)")
    ap.add_argument("--bb-snps", type=int, default=1_000_000)
    ap.add_argument("--bb-stream-snps", type=int, default=50_000)
    ap.add_argument("--bb-block", type=int, default=16_384)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-procs", type=int, default=0)
    ap.add_argument("--ref-snps", type=int, default=0, help="reference arm: SNPs per process and step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the hit list of the headline's last step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the GPU headline's results; --impl reference has none")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        reference_arm(args)
    else:
        gpu_arm(args)


if __name__ == "__main__":
    main()
