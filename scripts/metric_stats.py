"""Work counters of the summary path on a reduced C-sweep bundle (fo_metric_stats).
usage: python scripts/metric_stats.py [n_traj] [n_agents] [n_states]"""
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from frenetix_occlusion_b200 import synthetic as S  # noqa: E402
from frenetix_occlusion_b200.engine import AgentSet, MetricEngine  # noqa: E402

n, a, t = (int(x) for x in (sys.argv[1:4] + ["100000", "256", "51"][len(sys.argv) - 1:]))
case = S.make_case(n, a, t)
eng = MetricEngine(case["vehicle"], case["dt"], case["activated_metrics"], case["thresholds"])
eng.set_agents(AgentSet.from_case(case["agents"]))
ego = torch.from_numpy(case["ego"].astype("float32")).cuda()
st = eng.work_stats(ego)
evals = n * a * (t - 1)
print({k: v for k, v in st.items()}, "evals", evals)
for k in ("obb", "lr4s", "cp"):
    print(k, "per visited evaluation:", st[k] / max(st["visited"], 1))
print("be pairs per pair:", st["be"] / (n * a), "probes per be:", st["be_probes"] / max(st["be"], 1))
# the BE tree walks (one per warp and agent tile with colliding pairs): nodes visited and re-timed ego-path chunks
# computed, per trajectory -- scripts/be_tree_count.py gives the float64 count model of the same walk
print("be tree nodes per trajectory:", st["be_nodes"] / n, "ego-path chunks per trajectory:", st["be_path_chunks"] / n)
if st.get("windows"):
    print("window filter: kept", st["windows_kept"] / st["windows"], "of", st["windows"], "(agent, window) items;",
          "visited", st["visited"] / evals, "of the evaluations")
