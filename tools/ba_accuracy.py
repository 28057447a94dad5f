"""metric-size BA (E=512, 72 frames, 2 iterations) against the fp64 oracle: max abs error of poses / depths (run on the GPU box)"""
import os, sys, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT)
import droid_slam_b200
from droid_slam_b200 import synth
import oracle
be = droid_slam_b200.install()
s = synth.make_scene(synth.CONFIGS["metric"])
dev = "cuda"
args = [s[k].to(dev) for k in ("intrinsics", "disps_sens", "targets", "weights", "eta", "ii", "jj")]
P, D = s["poses"].to(dev), s["disps"].to(dev)
be.ba(P, D, *args, s["t0"], s["t1"], 2, s["lm"], s["ep"], False)
P, D = P.cpu().double(), D.cpu().double()
P64, D64 = s["poses"].double(), s["disps"].double()
oracle.ba(P64, D64, s["intrinsics"], s["disps_sens"], s["targets"], s["weights"], s["eta"], s["ii"], s["jj"], s["t0"], s["t1"], 2, s["lm"], s["ep"], False, dtype=torch.float64)
print("pose err %.3e disp err %.3e" % (float((P - P64).abs().max()), float((D - D64).abs().max())))
