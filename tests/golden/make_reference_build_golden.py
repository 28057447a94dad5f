"""Golden vectors for tests/test_vs_reference_build_gpu.py: the UNMODIFIED reference CUDA build (oracle/_ref/droid_backends_ref,
built by oracle/build_ref.sh with the Eigen stand-in) run on a B200 at BASELINE's full sizes.

    python tests/golden/make_reference_build_golden.py OUT.pt      (GPU; then copy OUT.pt to tests/golden/reference_build.pt)

Inputs are regenerated from seeds by the case functions below, which the test shares.  The full outputs run to hundreds of MB, so
the file keeps, per reference output:
  * ops compared bit for bit (lookups, geometry): the SHA-256 of the whole tensor (negative zeros folded into +0, so that equal
    hashes mean torch.equal) and a seeded sample of its values, which locates a mismatch;
  * ba: the full poses and a seeded sample of the inverse depths, held to the same relative criteria as the live comparison.
Before anything is written, our kernels are compared with the reference on the same tensors by the test's own criteria, and the
criteria are evaluated on the stored samples as well; the script fails if either does not hold."""
import hashlib
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from droid_slam_b200 import synth  # noqa: E402

DEV = "cuda"
EXACT_SAMPLE = 512        # values kept per bit-exact output (the hash carries the rest)
DISP_SAMPLE = 8192        # inverse-depth pixels kept per ba case
CHUNK = 128               # the reference's 32-bit accessors cannot address a 512-edge level-0 volume at once


# ---- fingerprints ------------------------------------------------------------------------------------------------------------------
def sample_index(numel, n, seed):
    return torch.randint(0, numel, (min(n, numel),), generator=torch.Generator().manual_seed(seed))


def fingerprint(t, seed, n=EXACT_SAMPLE):
    """sha256 of the whole tensor (with -0.0 folded into +0.0) + a seeded sample of its values"""
    t = t.detach().contiguous().cpu()
    if t.is_floating_point():
        t = t + 0.0
    flat = t.reshape(-1)
    return dict(sha256=hashlib.sha256(t.numpy().tobytes()).hexdigest(), shape=tuple(t.shape), dtype=str(t.dtype), seed=seed,
                sample=flat[sample_index(flat.numel(), n, seed)].clone())


def mismatch(t, fp):
    """None when `t` is bit-identical to the tensor `fp` was taken from, else a description of the difference"""
    got = fingerprint(t, fp["seed"], fp["sample"].numel())
    if got["shape"] != fp["shape"] or got["dtype"] != fp["dtype"]:
        return "shape/dtype %s %s, reference %s %s" % (got["shape"], got["dtype"], fp["shape"], fp["dtype"])
    if got["sha256"] == fp["sha256"]:
        return None
    return "not bit-identical: %d of %d sampled values differ" % (int((got["sample"] != fp["sample"]).sum()), fp["sample"].numel())


def disp_sample(D, seed, n=DISP_SAMPLE):
    D = D.detach().cpu().reshape(-1)
    return D[sample_index(D.numel(), n, seed)].clone()


# ---- ba criteria (BASELINE.json: 1e-4 relative) ---------------------------------------------------------------------------------------
def pose_rel(P, Pr):
    """every translation component relative to the pose's translation norm, quaternion components absolute"""
    P, Pr = P.double().cpu(), Pr.double().cpu()
    et = (P[:, :3] - Pr[:, :3]).abs() / Pr[:, :3].norm(dim=1, keepdim=True).clamp(min=1e-2)
    eq = (P[:, 3:] - Pr[:, 3:]).abs()
    return float(torch.cat([et, eq], 1).max())


def disp_rel(D, Dr, q=0.9999):
    """(q-quantile of the elementwise relative error, max abs error / max |reference|)"""
    D, Dr = D.double().cpu().flatten(), Dr.double().cpu().flatten()
    rel = torch.sort((D - Dr).abs() / Dr.abs()).values
    return float(rel[min(rel.numel() - 1, int(q * rel.numel()))]), float((D - Dr).abs().max() / Dr.abs().max())


def ba_ok(P, D, Pr, Dr):
    ep, (eq, ea) = pose_rel(P, Pr), disp_rel(D, Dr)
    return (ep < 1e-4 and eq < 1e-4 and ea < 1e-4), (ep, eq, ea)


# ---- cases (shared with the test) ----------------------------------------------------------------------------------------------------
def corr_metric_case():
    """512 edges x 48x64 f16 volumes, all four levels (CorrBlock.__call__, modules/corr.py:40-50): (volume, coords) per level"""
    s = synth.make_scene("metric")
    pyr, coords, _ = synth.make_corr_inputs(s, dtype=torch.float16, device=DEV)
    return [(vol, (coords / 2 ** lvl).contiguous()) for lvl, vol in enumerate(pyr)]


def corr_c2_case():
    """config 2 (fp32 volumes), 96 of its 128 edges: (volume, coords, grad or None) per level, gradients for levels 2 and 3"""
    s = synth.make_scene("c2_frontend")
    sub = dict(s); sub["ii"] = s["ii"][:96]; sub["jj"] = s["jj"][:96]; sub["coords_gt"] = s["coords_gt"][:96]; sub["cfg"] = dict(s["cfg"], E=96)
    pyr, coords, _ = synth.make_corr_inputs(sub, dtype=torch.float32, device=DEV)
    g = torch.Generator(device=DEV).manual_seed(3)
    out = []
    for lvl, vol in enumerate(pyr):
        grad = torch.randn(96, 7, 7, 48, 64, device=DEV, generator=g) if lvl >= 2 else None
        out.append((vol, (coords / 2 ** lvl).contiguous(), grad))
    return out


def altcorr_case():
    """AltCorrBlock.__call__ (modules/corr.py:104-117) on 48x64 f16 feature maps, 4 levels, a chunk of 24 edges: call args per level"""
    g = torch.Generator().manual_seed(5)
    N, M = 8, 24
    fmaps = torch.randn(1, N, 128, 48, 64, generator=g).half().to(DEV)
    s = synth.make_scene(dict(E=M, N=N, ht=48, wd=64, stereo=False, itrs=1, lm=1e-4, ep=0.1), seed=3)
    coords = (s["coords_gt"] + 2 * torch.rand(M, 48, 64, 2, generator=g) - 1).permute(0, 3, 1, 2)[None].contiguous().to(DEV)
    ii, jj = s["ii"].to(DEV), s["jj"].to(DEV)
    out, f = [], fmaps[0]
    for lvl in range(4):
        out.append((fmaps, f[None].contiguous(), (coords / 2 ** lvl).contiguous(), ii, jj, 3))
        f = torch.nn.functional.avg_pool2d(f, 2, stride=2)
    return out


def geometry_case():
    s = synth.make_scene("metric")
    P, D, K, ii, jj = [s[k].to(DEV) for k in ("poses", "disps", "intrinsics", "ii", "jj")]
    ix = torch.arange(72, device=DEV); th = torch.full((72,), 0.05, device=DEV)
    a, b = torch.meshgrid(torch.arange(72), torch.arange(72), indexing="ij")       # all pairs, like DepthVideo.distance
    return (P, D, K, ii, jj), (ix, th), (a.reshape(-1).to(DEV), b.reshape(-1).to(DEV))


# name -> (scene, make_scene kwargs, iterations, motion_only)
BA_CASES = {
    "metric": ("metric", {}, 2, False),                       # 512 edges, 72 keyframes
    "c4_stereo": ("c4_stereo", {}, 2, False),                 # 256 edges incl. one (i,i) edge per frame
    "c2_rgbd": ("c2_frontend", dict(rgbd=True), 2, False),
    "c2_rgbd_motion_only": ("c2_frontend", dict(rgbd=True), 2, True),
    "c3_global": ("c3_global", {}, 10, False),                # 2048 edges / 400 keyframes, lm=1e-5, ep=1e-2; 6P = 2394
}


def run_ba(be, name, scene=None):
    """ba on the case's scene through module `be`; returns (poses, disps, (dx, dz)) on the device"""
    cfg, kw, itrs, motion_only = BA_CASES[name]
    s = scene if scene is not None else synth.make_scene(cfg, **kw)
    args = [s[k].to(DEV) for k in ("intrinsics", "disps_sens", "targets", "weights", "eta", "ii", "jj")]
    P, D = s["poses"].to(DEV), s["disps"].to(DEV)
    out = be.ba(P, D, *args, s["t0"], s["t1"], itrs, s["lm"], s["ep"], motion_only)
    torch.cuda.synchronize()
    return P, D, out


# ---- generation --------------------------------------------------------------------------------------------------------------------
def main(out_path):
    sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))
    import droid_backends_ref as ref
    import droid_slam_b200
    ours = droid_slam_b200.install()
    G, report, seed = {}, {}, [0]

    def exact(key, o, r):
        assert torch.equal(o, r), key                          # the live comparison the test used to make
        seed[0] += 1
        G[key] = fingerprint(r, seed[0])
        assert mismatch(o, G[key]) is None, key

    for lvl, (vol, c) in enumerate(corr_metric_case()):
        o, = ours.corr_index_forward(vol, c, 3)
        r = torch.cat([ref.corr_index_forward(vol[a:a + CHUNK], c[a:a + CHUNK].contiguous(), 3)[0] for a in range(0, vol.shape[0], CHUNK)])
        exact("corr_metric_l%d" % lvl, o, r)
        del o, r
    torch.cuda.empty_cache()
    for lvl, (vol, c, grad) in enumerate(corr_c2_case()):
        exact("corr_c2_f32_l%d" % lvl, ours.corr_index_forward(vol, c, 3)[0], ref.corr_index_forward(vol, c, 3)[0])
        if grad is not None:
            exact("corr_c2_f32_bwd_l%d" % lvl, ours.corr_index_backward(vol, c, grad, 3)[0], ref.corr_index_backward(vol, c, grad, 3)[0])
    for lvl, a in enumerate(altcorr_case()):
        exact("altcorr_l%d" % lvl, ours.altcorr_forward(*a)[0].contiguous(), ref.altcorr_forward(*a)[0].contiguous())
    (P, D, K, ii, jj), (ix, th), (a, b) = geometry_case()
    (c, v), (cr, vr) = ours.projmap(P, D, K, ii, jj), ref.projmap(P, D, K, ii, jj)
    exact("projmap_coords", c, cr); exact("projmap_valid", v, vr)
    exact("iproj", ours.iproj(P, D, K), ref.iproj(P, D, K))
    exact("depth_filter", ours.depth_filter(P, D, K, ix, th), ref.depth_filter(P, D, K, ix, th))
    d, dr = ours.frame_distance(P, D, K, a, b, 0.3), ref.frame_distance(P, D, K, a, b, 0.3)
    assert float(((d - dr).abs() / dr.abs().clamp(min=1e-3)).max()) < 1e-5
    G["frame_distance"] = dr.cpu()                             # 5184 values, kept whole
    for name, (cfg, kw, itrs, motion_only) in BA_CASES.items():
        s = synth.make_scene(cfg, **kw)
        P, D, o = run_ba(ours, name, s)
        Pr, Dr, r = run_ba(ref, name, s)
        seed[0] += 1
        e = dict(poses=Pr.cpu(), disps_seed=seed[0], disps_sample=disp_sample(Dr, seed[0]))
        if motion_only:                                        # the reference returns no dz here
            assert pose_rel(P, Pr) < 1e-4 and torch.equal(D, Dr), name
            e["disps"] = fingerprint(Dr, seed[0])
            report[name] = dict(pose_rel=pose_rel(P, Pr))
        else:
            ok, full = ba_ok(P, D, Pr, Dr)
            ok_s, smp = ba_ok(P, disp_sample(D, seed[0]), Pr, e["disps_sample"])
            assert ok and ok_s, (name, full, smp)
            assert o[0].shape == r[0].shape and o[1].shape == r[1].shape, name
            e["dx_shape"], e["dz_shape"] = tuple(r[0].shape), tuple(r[1].shape)
            report[name] = dict(full=full, sample=smp)
        G["ba_" + name] = e
    G["_meta"] = dict(gpu=torch.cuda.get_device_name(0), torch=str(torch.__version__), cuda=torch.version.cuda, ours_vs_reference_ba=report,
                      note="reference = the unmodified reference src/*.cu + droid.cpp built for sm_100a by oracle/build_ref.sh (Eigen stand-in: dense fp64 LLT)")
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    torch.save(G, out_path)
    for k, v in report.items():
        print(k, v)
    print("saved", out_path, os.path.getsize(out_path), "bytes")


if __name__ == "__main__":
    main(sys.argv[1])
