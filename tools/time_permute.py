"""Times the permutation test (gwasdev_marginal_permute) at configs[1] (500 000 SNPs x 10 000 samples, 5 000 cases) against the
re-selection loop (select + K1' scan per permutation), with P in {256, 1 024, 4 096}, complete and with 1 % missing calls.
Achieved int8 TOP/s count 2 operations per multiply-accumulate of the GEMM as run (planes x 32 Wr sample bytes per SNP and
256-padded permutation blocks) against gwasdev_i8_peak measured in the same process.
usage: python tools/time_permute.py [--perms 256,1024,4096] [--loop 64]"""
import argparse
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import libgwaspp_b200 as gw  # noqa: E402

M, N, NCASE = 500_000, 10_000, 5_000


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--perms", default="256,1024,4096")
    ap.add_argument("--loop", type=int, default=64, help="permutations of the timed re-selection loop")
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    try:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True).stdout.strip()
    except OSError:
        gpu = "unknown"
    burst, sustained = gw.i8_peak(0)
    print(f"# {gpu} | gwasdev_i8_peak burst {burst:.0f} sustained {sustained:.0f} TOP/s")
    pheno = gw.simulate_phenotype(20121127, N, NCASE)
    cm, tm = gw.stream_masks(pheno)
    kbytes = 32 * ((gw.plane_blocks(N) // 2 + 3) // 4 * 4)
    print("| missing | P | planes | GEMM ms | total ms | ms / 1000 perm | int8 TOP/s | share of sustained peak | loop ms / 1000 perm | speed-up |")
    print("|---|---|---|---|---|---|---|---|---|---|")
    for missing in (0.0, 0.01):
        st = gw.GenoStore(M, N)
        st.simulate(20121127, missing_rate=missing)
        st.select_case_control(case_mask=cm, ctrl_mask=tm)
        # re-selection loop: select a permuted phenotype + K1' scan per permutation (device outputs)
        import torch
        d_stats = torch.empty((M, 8), dtype=torch.float64, device="cuda")
        masks = gw.permutation_masks(N, cm, tm, 1, 0, a.loop)
        sel = cm | tm
        st.select_case_control(case_mask=masks[0], ctrl_mask=sel & ~masks[0])
        st.marginal_scan_into(0, M, stats=d_stats)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k in range(a.loop):
            st.select_case_control(case_mask=masks[k], ctrl_mask=sel & ~masks[k])
            st.marginal_scan_into(0, M, stats=d_stats)
        torch.cuda.synchronize()
        loop_ms = 1e3 * (time.perf_counter() - t0) / a.loop * 1000
        st.select_case_control(case_mask=cm, ctrl_mask=tm)
        for P in [int(x) for x in a.perms.split(",")]:
            st.marginal_permute(P, seed=7)        # warm-up (builds the resident SNP planes the first time)
            best = None
            for r in range(a.reps):
                s = st.marginal_permute(P, seed=7 + r, first_perm=P * r)["stats"]
                if best is None or s.total_ms < best.total_ms:
                    best = s
            ops = 2.0 * ((P + 255) // 256 * 256) * M * best.planes * kbytes
            tops = ops / (best.gemm_ms * 1e-3) / 1e12
            print(f"| {missing:.0%} | {P} | {best.planes} | {best.gemm_ms:.2f} | {best.total_ms:.2f} | {best.total_ms / P * 1000:.2f} | "
                  f"{tops:.0f} | {tops / sustained:.2f} | {loop_ms:.1f} | {loop_ms / (best.total_ms / P * 1000):.1f}x |", flush=True)
        st.close()


if __name__ == "__main__":
    main()
