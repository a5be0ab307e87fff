"""Times windowed LD (gwasdev_ld_window) at 500 000 SNPs x 10 000 samples, windows 64 / 1 000 / 10 000, complete and with 1 %
missing calls, against gwasdev_i8_peak measured in the same process; the operand build; the same pairs through gwasdev_ld_pairs
and through a torch fp16 banded matmul of the decoded, standardised dosages (the baselines a user would otherwise write); and
the cost of the list output on an LD-structured table where many pairs qualify.
Algorithmic int8 TOP/s count 2 operations per multiply-accumulate the contract needs: pairs x 32 Wr sample bytes x (1 product
without missing calls, 6 with).
usage: python tools/time_ld.py [--windows 64,1000,10000] [--reps 3]"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import libgwaspp_b200 as gw  # noqa: E402

M, N = 500_000, 10_000


def gpu_name():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True).stdout.strip()
    except OSError:
        return "unknown"


def dosages(st, r0, n):
    rows = st.get_rows(r0, n)
    P = st.P
    bits = lambda b: np.unpackbits(b.view(np.uint8), axis=-1, bitorder="little")[:, :N].astype(bool)
    p1, p2 = bits(np.ascontiguousarray(rows[:, 1:1 + P])), bits(np.ascontiguousarray(rows[:, 1 + P:]))
    return (p2 & ~p1).astype(np.float32) + 2 * (p1 & p2), p1 | p2


def torch_banded(st, window, n_snps=20_000, blk=2048):
    """fp16 matmul of standardised dosages (missing calls set to the mean), blocks of `blk` A-SNPs against their window."""
    import torch
    x, c = dosages(st, 0, n_snps)
    mu = (x * c).sum(1, keepdims=True) / np.maximum(c.sum(1, keepdims=True), 1)
    z = np.where(c, x, mu) - mu
    z /= np.maximum(np.sqrt((z * z).sum(1, keepdims=True)), 1e-12)
    Z = torch.from_numpy(z).to("cuda", torch.float16)
    def run():
        for i0 in range(0, n_snps, blk):
            r = Z[i0:i0 + blk] @ Z[i0:min(n_snps, i0 + blk + window)].T
            (r * r).float()
    run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run()
    e1.record()
    torch.cuda.synchronize()
    w = min(window, n_snps - 1)
    return e0.elapsed_time(e1), (n_snps - w) * w + w * (w - 1) // 2


def mosaic_table(M2, seed=5, founders=8, switch=0.01):
    rng = np.random.default_rng(seed)
    F = (rng.random((founders, M2)) < rng.uniform(0.05, 0.95, M2)).astype(np.int8)
    G = np.zeros((M2, N), np.int8)
    for h in range(2):
        src = rng.integers(0, founders, N)
        for m in range(M2):
            sw = rng.random(N) < switch
            src = np.where(sw, rng.integers(0, founders, N), src)
            G[m] += F[src, m]
    code = np.array([0, 2, 3], np.uint8)[G]
    q = code.reshape(M2, -1, 4)
    return (q[..., 0] | (q[..., 1] << 2) | (q[..., 2] << 4) | (q[..., 3] << 6)).astype(np.uint8)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", default="64,1000,10000")
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    burst, sustained = gw.i8_peak(0)
    print(f"# {gpu_name()} | gwasdev_i8_peak burst {burst:.0f} sustained {sustained:.0f} TOP/s")
    kbytes = 32 * ((gw.plane_blocks(N) // 2 + 3) // 4 * 4)
    print("| missing | window | rows/SNP | pairs | GEMM ms | call ms | pairs/s | algorithmic int8 TOP/s | share of sustained peak |")
    print("|---|---|---|---|---|---|---|---|---|")
    stores = {}
    build = {}
    for missing in (0.0, 0.01):
        st = gw.GenoStore(M, N)
        st.simulate(20121127, missing_rate=missing)
        stores[missing] = st
        _, _, first = st.ld_window(64, 0.5)                     # builds the resident operand
        _, _, warm = st.ld_window(64, 0.5)
        build[missing] = (first.total_ms, warm.total_ms)
        for w in [int(x) for x in a.windows.split(",")]:
            best = None
            for _ in range(a.reps):
                _, _, s = st.ld_window(w, 0.5)
                if best is None or s.gemm_ms < best.gemm_ms:
                    best = s
            prod = 1 if best.rows_per_snp == 1 else 6
            tops = 2.0 * best.pairs_tested * kbytes * prod / (best.gemm_ms * 1e-3) / 1e12
            print(f"| {missing:.0%} | {w} | {best.rows_per_snp} | {best.pairs_tested:.3g} | {best.gemm_ms:.2f} | {best.total_ms:.2f} | "
                  f"{best.pairs_tested / best.gemm_ms * 1e3:.3g} | {tops:.0f} | {tops / sustained:.2f} |", flush=True)
    for missing, (f, w) in build.items():
        print(f"# operand build ({missing:.0%} missing): first call {f:.2f} ms, repeated call {w:.2f} ms (window 64)")

    st = stores[0.0]
    # baselines on the first 20 000 SNPs: the CUDA-core pair path and a torch fp16 banded matmul
    for w in (64, 1000):
        n_snps = 20_000
        I = np.concatenate([np.arange(0, n_snps - d) for d in range(1, w + 1)]).astype(np.uint32)
        J = (I + np.concatenate([np.full(n_snps - d, d) for d in range(1, w + 1)])).astype(np.uint32)
        cap = min(len(I), 2_000_000)
        st.ld_pairs(I[:1000], J[:1000])
        t0 = time.perf_counter()
        st.ld_pairs(I[:cap], J[:cap])
        dt = time.perf_counter() - t0
        _, _, s = st.ld_window(w, 0.5, 0, n_snps)
        tms, tp = torch_banded(st, w, n_snps)
        print(f"# window {w}, SNPs [0, {n_snps}): ld_window GEMM {s.gemm_ms:.2f} ms ({s.pairs_tested / s.gemm_ms * 1e3:.3g} pairs/s); "
              f"ld_pairs {cap / dt:.3g} pairs/s (host call incl. copies, {cap} pairs); torch fp16 banded matmul {tms:.2f} ms "
              f"({tp / tms * 1e3:.3g} pairs/s)", flush=True)
    for s_ in stores.values():
        s_.close()

    # list output on an LD-structured table
    M2 = 50_000
    ld = gw.GenoStore(M2, N)
    ld.put_bed(mosaic_table(M2))
    for w in (100, 1000):
        _, _, s0 = ld.ld_window(w, 0.5, pairs=False)
        for thr in (2.0, 0.5, 0.0):
            best = None
            for _ in range(a.reps):
                p, _, s = ld.ld_window(w, thr, capacity=w * M2 + 1)
                if best is None or s.total_ms < best.total_ms:
                    best = s
            print(f"# LD table {M2} x {N}, window {w}, threshold {thr}: {best.pairs_kept:.3g} of {best.pairs_tested:.3g} pairs listed, "
                  f"GEMM {best.gemm_ms:.2f} ms, call {best.total_ms:.2f} ms", flush=True)
    ld.close()


if __name__ == "__main__":
    main()
