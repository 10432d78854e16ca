"""Run by tests/test_cuda_frame_parity.py::test_unchanged_reference_tracker_runs_fused in a fresh process:
the reference's UNMODIFIED utils/tracker.py (oracle/_ref) on top of the install()ed drop-in classes.

Checks that its query_feature -> Decoder.sdf -> get_gradient sequence (utils/tracker.py:297-335) is served by the
fused K1 kernel through the lazy feature handles (few launches, no eager gathers) and returns the values of the
repo's own fused Tracker path.

What that unmodified caller returned is stored in tests/golden/unchanged_caller.npz, so the fused path is compared
with it also where oracle/_ref is not vendored.  `--save PATH` records that file (needs oracle/_ref and a GPU)."""
import argparse
import json
import os
import sys
from unittest.mock import MagicMock

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from pin_slam_b200 import install, ops  # noqa: E402
from pin_slam_b200.config import HotPathConfig  # noqa: E402
from pin_slam_b200.model import Decoder  # noqa: E402
from pin_slam_b200.synthetic import build_map, surface_queries  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden", "unchanged_caller.npz")
GOLDEN_ROWS = 2048  # stored queries per workload (the queries are random surface samples: the first rows are a fair sample)
# the compared outputs of Tracker.query_source_points, in its return order (None: not compared)
FIELDS = ("sdf", "grad", "color", "color_grad", None, "mask", "certainty", None)

ap = argparse.ArgumentParser()
ap.add_argument("--save", default=None, help="write the unmodified caller's outputs to this .npz")
args = ap.parse_args()

have_ref = os.path.isfile(os.path.join(ROOT, "oracle", "_ref", "utils", "tracker.py"))
assert have_ref or args.save is None, "--save needs the reference's own tracker.py under oracle/_ref"
install.install()  # model.neural_points / model.decoder -> the drop-ins
if have_ref:
    for m in ["open3d", "matplotlib", "matplotlib.cm", "matplotlib.pyplot", "roma", "wandb", "natsort", "skimage",
              "skimage.measure", "pypose", "gtsam", "dtyper", "pyquaternion", "laspy", "evo", "dataset",
              "dataset.slam_dataset"]:
        sys.modules.setdefault(m, MagicMock())
    sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))
    from utils.tracker import Tracker as RefTracker  # noqa: E402  (the reference's own file)

    assert "oracle/_ref/utils/tracker.py" in RefTracker.query_source_points.__code__.co_filename.replace(os.sep, "/")
golden = dict(np.load(GOLDEN)) if os.path.isfile(GOLDEN) and args.save is None else None

out, saved = {}, {}
for name, cfg in (("replica_colour", HotPathConfig.replica(device="cuda", feature_std=0.1, buffer_size=200003)),
                  ("cfg2", HotPathConfig.cfg2(device="cuda", feature_std=0.1, local_map_radius=1e4))):
    cfg.buffer_size = 200003
    npm = build_map(cfg, n_surface=150000, seed=3, extent=20.0 if name == "replica_colour" else 40.0)
    torch.manual_seed(1)
    sdf_mlp = Decoder(cfg, cfg.geo_mlp_hidden_dim, cfg.geo_mlp_level, 1)
    color_mlp = Decoder(cfg, cfg.color_mlp_hidden_dim, cfg.color_mlp_level, cfg.color_channel) if cfg.color_on else None
    for d in (sdf_mlp, color_mlp):
        if d is not None:
            for p_ in d.parameters():
                p_.requires_grad_(False)  # what pin_slam.py's freeze_decoders does once the map is initialised
    q = surface_queries(npm, 6000, seed=2)
    colour = color_mlp is not None
    if have_ref:
        trk = RefTracker(cfg, npm, {"sdf": sdf_mlp, "semantic": None, "color": color_mlp})
        n0 = ops.launch_count()
        res = trk.query_source_points(q.clone(), cfg.infer_bs, True, True, colour, colour, False, True, True, True)
        torch.cuda.synchronize()
        launches = ops.launch_count() - n0
    o = npm.query_sdf(q, sdf_mlp, need_grad=True, color_decoder=color_mlp, color_grad=colour)
    torch.cuda.synchronize()
    r = {"grad_scale": float(o["grad"].abs().mean())}
    if golden is not None:
        # the fused path against what the unmodified caller returned when the fixture was recorded
        # (relative to the largest stored value for sdf / gradients / colour; absolute for the certainty)
        g = lambda k: torch.from_numpy(golden[f"{name}.{k}"]).cuda()  # noqa: E731
        n = g("sdf").shape[0]
        rel = lambda k, got: float((g(k) - got[:n]).abs().max() / g(k).abs().max().clamp_min(1e-12))  # noqa: E731
        r["golden_sdf_err"] = rel("sdf", o["sdf"])
        r["golden_grad_err"] = rel("grad", o["grad"])
        r["golden_cert_err"] = float((g("certainty") - o["certainty"][:n]).abs().max())
        r["golden_mask_equal"] = bool(torch.equal(g("mask"), o["nn_count"][:n] >= 4))
        if colour:
            r["golden_color_err"] = rel("color", o["color"])
            r["golden_cgrad_err"] = rel("color_grad", o["color_grad"])
    if have_ref:
        sdf, grad, col, cgrad, _, mask, cert, std = res
        r.update({"launches": launches, "sdf_err": float((sdf - o["sdf"]).abs().max()),
                  "grad_err": float((grad - o["grad"]).abs().max()),
                  "cert_err": float((cert - o["certainty"]).abs().max()),
                  "mask_equal": bool(torch.equal(mask, o["nn_count"] >= 4))})
        if colour:
            r["color_err"] = float((col - o["color"]).abs().max())
            r["cgrad_err"] = float((cgrad - o["color_grad"]).abs().max())
        for k, v in zip(FIELDS, res):
            if k is not None and v is not None:
                saved[f"{name}.{k}"] = v[:GOLDEN_ROWS].detach().cpu().numpy()
        # the eager (materialising) path of the same unchanged caller, for reference
        type(npm).FUSED_QUERY_FEATURE = False
        n0 = ops.launch_count()
        res2 = trk.query_source_points(q.clone(), cfg.infer_bs, True, True, colour, colour, False, True, True, True)
        torch.cuda.synchronize()
        r["launches_eager"] = ops.launch_count() - n0
        r["eager_vs_fused_sdf"] = float((res2[0] - sdf).abs().max())
        r["eager_vs_fused_grad"] = float((res2[1] - grad).abs().max())
        type(npm).FUSED_QUERY_FEATURE = True
    out[name] = r
if args.save:
    np.savez_compressed(args.save, **saved)
print("RESULT " + json.dumps(out))
