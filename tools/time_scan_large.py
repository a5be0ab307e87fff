"""Times the marginal scan of a cohort whose masks exceed shared memory: 1 000 000 cases and 900 000 controls (a 237 KB
mask, read from global memory; K0 cannot compact this selection), next to 800 000 / 800 000 (a 200 KB mask in shared memory).
First scan (mode 1: three masked and three plain popcount streams, row totals written) and later scans (mode 2: row
totals cached), device outputs, CUDA-event kernel time; the rate is the raw rows' bytes over that time."""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import libgwaspp_b200 as gw

M = 20_000
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip(), flush=True)
for n_case, n_ctrl in ((800_000, 800_000), (1_000_000, 900_000)):
    N = n_case + n_ctrl
    with gw.GenoStore(M, N) as st:
        st.simulate(20121127)
        pheno = gw.simulate_phenotype(20121127, N, n_case)
        counts = torch.empty((M, 8), dtype=torch.int32, device="cuda")
        stats = torch.empty((M, 8), dtype=torch.float64, device="cuda")
        raw_gb = M * 2 * gw.plane_blocks(N) * 2 / 1e9
        for rep in range(3):
            st.select_case_control(pheno)
            times = []
            for k in range(4):
                st.marginal_scan_into(0, M, counts=counts, stats=stats)
                times.append(st.last_scan_ms())
            print(f"{n_case} cases / {n_ctrl} controls, {M} SNPs, {raw_gb:.2f} GB of raw rows, rep {rep}: first scan {times[0]:.2f} ms "
                  f"({raw_gb / times[0] * 1e3:.0f} GB/s), later scans " + ", ".join(f"{t:.2f}" for t in times[1:]) +
                  f" ms ({raw_gb / min(times[1:]) * 1e3:.0f} GB/s); compacted: {st.is_compacted()}", flush=True)
