"""Golden fixture for the PN2_LOCAL sibling model and the Avg / MSG set-abstraction modules from the REFERENCE's own
classes (build container only): network_models/models/PointNet2_local.py::PointNet2 / PointNet2Loss / PointNet2Metric and
pointnet2_utils/modules.py::PointNetSAAvgModule / PointNetSAModuleMSG, run on torch-CPU with the C restatement of the
operators injected as pn2_ext (like tests/golden/make_golden.py).  -> tests/golden/pn2_local.npz"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
from make_golden import array_digest, import_reference, seed_reference_weights  # noqa: E402

import_reference()
from grasp_proposal.network_models.models.PointNet2_local import PointNet2, PointNet2Loss, PointNet2Metric  # noqa: E402
from grasp_proposal.network_models.models.pointnet2_utils.modules import PointNetSAAvgModule, PointNetSAModuleMSG  # noqa: E402

CFG = dict(score_classes=3, num_centroids=(256, 64, 16, 0), radius=(0.1, 0.2, 0.4, -1.0), num_neighbours=(16, 16, 8, -1),
           sa_channels=((16, 16, 32), (32, 32, 64), (64, 64, 128), (128, 128, 256)),
           fp_channels=((64, 64), (64, 32), (32, 32), (32, 32, 16)), num_fp_neighbours=(0, 3, 3, 3), seg_channels=(32,),
           dropout_prob=0.5)
torch.manual_seed(0)
net = seed_reference_weights(PointNet2(**CFG))
torch.nn.init.normal_(net.t_logit.weight, std=0.05)  # the zero init would hide the translation head
net.eval()
rs = np.random.RandomState(7)
points = torch.from_numpy(rs.rand(2, 3, 1024).astype(np.float32))
n_frames, n_search = 40, 6
frames = torch.from_numpy(rs.randn(2, 12, n_frames, n_search).astype(np.float32))
fix = {"points": points.numpy(), "frames": frames.numpy().copy()}
with torch.no_grad():
    out_self = net({"scene_points": points})                                      # "real experiments" branch
    out_given = net({"scene_points": points, "local_search_frame": frames})       # candidates given (modifies `frames`)
fix["frames_after"] = frames.numpy().copy()
labels = {"scored_grasp_labels": torch.from_numpy(rs.randint(0, 3, (2, n_frames, n_search))),
          "scene_movable_labels": torch.from_numpy(rs.randint(0, 2, (2, 1024))),
          "best_frame_R": torch.from_numpy(np.linalg.qr(rs.randn(2, n_frames, 3, 3))[0].reshape(2, n_frames, 9)
                                           .transpose(0, 2, 1).astype(np.float32).copy()),
          "best_frame_t": torch.from_numpy(rs.rand(2, 3, n_frames).astype(np.float32))}
loss = PointNet2Loss()(out_given, labels)
metric = PointNet2Metric()(out_given, labels)
# the model's weights as digests (keeps the file under 1 MB): tests/test_pn2_local.py rebuilds them from the same seeds
fix["sd_keys"] = np.array(list(net.state_dict()))
fix["sd_sha256"] = np.array([array_digest(v) for v in net.state_dict().values()])
fix.update({"self/" + k: v.numpy() for k, v in out_self.items()})
fix.update({"given/" + k: v.numpy() for k, v in out_given.items()})
fix.update({"label/" + k: v.numpy() for k, v in labels.items()})
fix.update({"loss/" + k: v.numpy() for k, v in loss.items()})
fix.update({"metric/" + k: v.numpy() for k, v in metric.items()})

# the two extra set-abstraction modules on a 24-channel feature map
feat = torch.from_numpy(rs.randn(2, 24, 1024).astype(np.float32))
fix["feat"] = feat.numpy()
torch.manual_seed(1)
avg = seed_reference_weights(PointNetSAAvgModule(24, (32, 48), 128, 0.15, 16, True)).eval()
msg = seed_reference_weights(PointNetSAModuleMSG(24, ((16, 32), (32, 64)), 128, (0.1, 0.2), (8, 16), True)).eval()
with torch.no_grad():
    ax, af = avg(points, feat)
    mx, mf = msg(points, feat)
fix.update({"avg_sd/" + k: v.numpy() for k, v in avg.state_dict().items()})
fix.update({"msg_sd/" + k: v.numpy() for k, v in msg.state_dict().items()})
fix.update({"avg/xyz": ax.numpy(), "avg/feature": af.numpy(), "msg/xyz": mx.numpy(), "msg/feature": mf.numpy()})

# EdgeConv variants: set abstraction on edge features, feature propagation over the 3 interpolation neighbours
from grasp_proposal.network_models.models.pointnet2_utils.modules import EdgeFPModule, EdgeSAModule  # noqa: E402
import types  # noqa: E402
import grasp_proposal.network_models.functions.gather_knn as ref_gather_knn  # noqa: E402
# the compiled dgcnn_ext is absent here; its forward is a plain gather (gather_knn_kernel.cu:27-49): out[b,c,m,k] =
# feature[b,c,index[b,m,k]] — restated for the generator only
ref_gather_knn.dgcnn_ext = types.SimpleNamespace(gather_knn_forward=lambda feature, index: torch.gather(
    feature.unsqueeze(2).expand(-1, -1, index.size(1), -1), 3, index.unsqueeze(1).expand(-1, feature.size(1), -1, -1)))
torch.manual_seed(2)
esa = seed_reference_weights(EdgeSAModule(24, (32, 48), 128, 0.15, 16, True)).eval()
efp = seed_reference_weights(EdgeFPModule(2 * 48 + 24, (64, 32), 3)).eval()
with torch.no_grad():
    ex, ef = esa(points, feat)
    back = efp(points, ex, feat, ef)
fix.update({"esa_sd/" + k: v.numpy() for k, v in esa.state_dict().items()})
fix.update({"efp_sd/" + k: v.numpy() for k, v in efp.state_dict().items()})
fix.update({"esa/xyz": ex.numpy(), "esa/feature": ef.numpy(), "efp/feature": back.numpy()})
np.savez_compressed(os.path.join(HERE, "pn2_local.npz"), **fix)
print({k: v.shape for k, v in fix.items() if "sd/" not in k})
