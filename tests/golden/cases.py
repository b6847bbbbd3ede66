"""Golden-fixture cases: reduced shapes the reference/oracle finish in seconds on CPU, plus the full
Charades configuration (BASELINE.json configs[0], the reference's own CPU-runnable case)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from vmrframe_b200.synth import Workload, small_workload  # noqa: E402

CASES = {
    # name: workload                      (B, L, Tmax, C, config_id)
    "charades_small": small_workload("charades_small", 4, 64, 10, 10, 101),
    "anet_small": small_workload("anet_small", 3, 100, 25, 12, 102),
    "tacos_small": small_workload("tacos_small", 2, 256, 19, 10, 103),
    "edge_b1": small_workload("edge_b1", 1, 64, 3, 4, 104),
    "charades_full": Workload("charades_full", 105, 32, 64, 10, 10, num_words=200),
}
# cases whose hooked intermediate tensors are stored (kept to one to bound the fixture size)
TAPPED = {"charades_small"}
# taps of a TAPPED case stored in <case>_taps.npz instead of <case>.npz: all of them in one file would exceed 1 MB
LATE_TAPS = ("t2v", "v2t", "fuse", "fep_s", "fep_e")
