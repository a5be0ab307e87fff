"""Times the pair screens over SNP sets (GenoStore.pairwise_scan_sets) at 500 000 SNPs x 10 000 samples (5 000 / 5 000, or
--snps / --samples), complete and with 1 % missing calls, next to the whole-table screen in the same process:
  set-by-all   the --top SNPs with the smallest marginal genotypic p-value against every SNP
  within       a set of --within SNPs (every (M / within)-th SNP, as a thinned table would leave them)
  set-by-set   two disjoint sets of --sets SNPs each
For each: total_ms (whole call), screen_ms (screen kernels), their difference (gather, selection, margins, operands, fp64 re-score
and sort; at threshold 30 the re-score and sort take well under a millisecond), screen-phase pairs/s, and the whole-table
screen's pairs/s. Prints the device name and power limit first."""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import libgwaspp_b200 as gw

ap = argparse.ArgumentParser()
ap.add_argument("--snps", type=int, default=500_000)
ap.add_argument("--samples", type=int, default=10_000)
ap.add_argument("--top", type=int, default=1000)
ap.add_argument("--within", type=int, default=100_000)
ap.add_argument("--sets", type=int, default=20_000)
ap.add_argument("--reps", type=int, default=2)
ap.add_argument("--missing", type=float, nargs="*", default=[0.0, 0.01])
a = ap.parse_args()

try:
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip(), flush=True)
except (OSError, subprocess.SubprocessError) as e:
    print(f"nvidia-smi unavailable: {e}", flush=True)

M, N = a.snps, a.samples
for miss in a.missing:
    with gw.GenoStore(M, N) as st:
        st.simulate(20121127, missing_rate=miss)
        st.select_case_control(gw.simulate_phenotype(20121127, N, N // 2))
        st.pairwise_scan(30.0)                                   # warm-up: margins, operands, modules
        _, whole = st.pairwise_scan(30.0)
        whole_rate = whole.pairs_tested / whole.screen_ms * 1e3
        print(f"missing {miss:g}: whole table {M} SNPs: screen {whole.screen_ms:.1f} ms total {whole.total_ms:.1f} ms "
              f"pairs {whole.pairs_tested} -> {whole_rate / 1e9:.1f} G pairs/s", flush=True)
        rec, _ = st.marginal_scan_compact()
        top = np.sort(np.argsort(rec["p_genotypic"], kind="stable")[:a.top]).astype(np.uint32)
        rng = np.random.default_rng(7)
        perm = rng.permutation(M)
        work = {
            f"set-by-all ({a.top} x all)": (top, np.ones(M, bool)),
            f"within ({a.within})": (np.arange(0, M, M // a.within, dtype=np.uint32)[:a.within], None),
            f"set-by-set ({a.sets} x {a.sets})": (np.sort(perm[:a.sets]).astype(np.uint32), np.sort(perm[a.sets:2 * a.sets]).astype(np.uint32)),
        }
        for name, (sa, sb) in work.items():
            st.pairwise_scan_sets(sa, sb, 30.0)                  # warm-up of the SETS kernels
            for r in range(a.reps):
                hits, s = st.pairwise_scan_sets(sa, sb, 30.0)
                rate = s.pairs_tested / s.screen_ms * 1e3
                print(f"  {name:28s} rep {r}: total {s.total_ms:8.1f} ms  screen {s.screen_ms:8.1f} ms  other {s.total_ms - s.screen_ms:7.1f} ms  "
                      f"pairs {s.pairs_tested:.4g} tiles {s.tiles} (four-plane {s.tiles_nine_cell}) -> {rate / 1e9:6.1f} G pairs/s "
                      f"({rate / whole_rate:.2f} of whole), hits {len(hits)}", flush=True)
