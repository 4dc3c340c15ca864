"""Re-time every chain shape of PN2_CLS on this GPU and print the plan table entries (to regenerate
s4g_release_b200/tuned_plans.json):   python profiles/dump_tuned_plans.py > gpurun_out/tuned_plans_run.json"""
import json
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench import seeded_model  # noqa: E402
from s4g_release_b200 import engine  # noqa: E402

t0 = time.time()
if "--edge" in sys.argv:  # the chains of EDGEPN2D at its default arguments (the table keeps its two edge chains, in_mode 6)
    from bench_global import seeded  # noqa: E402
    from s4g_release_b200.network_models.models.EdgePointNet2Down import EdgePointNet2Down  # noqa: E402
    eng = engine.FusedEdgePointNet2Down(seeded(EdgePointNet2Down).cuda(), autotune="force")
elif "--edge-downup" in sys.argv:  # EDGEPN2DU at its default arguments (the table keeps its edge propagation chains)
    from bench_global import seeded  # noqa: E402
    from s4g_release_b200.network_models.models.EdgePointNet2DownUp import EdgePointNet2DownUp  # noqa: E402
    eng = engine.FusedEdgePointNet2DownUp(seeded(EdgePointNet2DownUp).cuda(), autotune="force")
else:
    eng = engine.FusedPointNet2(seeded_model().cuda(), autotune="force")
torch.cuda.synchronize()
out = engine.export_tuned_plans()
out["_seconds"] = round(time.time() - t0, 2)
print(json.dumps(out, indent=1))
