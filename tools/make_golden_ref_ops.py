"""Store what the REFERENCE's own native code computes on the tests' inputs, so that the tests compare against it on
any machine (the reference binaries under oracle/_ref are built only where the reference sources are).

  python tools/make_golden_ref_ops.py cpu [OUT]    -> tests/golden/ref_cpu_ops.npz
      FPS (core/csrc/fps/src/farthest_point_sampling.cpp, oracle/_ref/libfps_ref.so) and the uncertainty PnP solved
      with the reference's vendored Ceres (oracle/_ref/libupnp_ceres_ref.so).
  python tools/make_golden_ref_ops.py cuda [OUT]   -> tests/golden/ref_cuda_ops.npz   (needs a GPU)
      the reference's CUDA extensions ransac_voting, torch_nndistance_aten and flow_cuda, compiled unmodified for
      sm_100a into oracle/_ref (python oracle/build_ref.py --cuda-refs).

Inputs come from the tests' own seeded recipes (imported from tests/).  Large outputs are stored as a SHA-256 plus a
seeded sample (tests/test_gpu_parity.py: golden_record).
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def make_cpu():
    import ctypes

    import test_oracle_pinning as TP

    so = os.path.join(ROOT, "oracle", "_ref", "libfps_ref.so")
    if not os.path.exists(so):
        raise SystemExit("%s not built (python oracle/build_ref.py)" % so)
    fps = ctypes.CDLL(so)

    def fps_ref(pts, sn):
        idx = np.zeros(sn, np.int32)
        fps.farthest_point_sampling_init_center(pts.ctypes.data_as(ctypes.c_void_p), idx.ctypes.data_as(ctypes.c_void_p),
                                                len(pts), sn)
        return idx

    out = {}
    for pn, sn, pts in TP.fps_ref_cases():
        out["fps/%d_%d" % (pn, sn)] = fps_ref(pts, sn)
    # test_baseline_config0_cpu_plumbing: the first draw of RandomState(0)
    out["fps/config0"] = fps_ref(np.random.RandomState(0).uniform(-0.1, 0.1, (8192, 3)).astype(np.float32), 64)

    def upnp(prefix, probs):
        out[prefix + "/n"] = np.int64(len(probs))
        for i, (K, rt, p2, p3, w, init) in enumerate(probs):
            ref = TP.upnp_ceres_ref(p2, p3, w, K, init)
            if ref is None:
                raise SystemExit("oracle/_ref/libupnp_ceres_ref.so not built (python oracle/build_ref.py)")
            for f, v in zip(TP.UPNP_REF_FIELDS, (K, rt, p2, p3, w, init, ref)):
                out["%s/%d/%s" % (prefix, i, f)] = v

    # the problem sequences the tests drew before their inputs were stored (two discarded problems first on the CPU side)
    rs = np.random.RandomState(3)
    TP._upnp_problem(rs, 8, 0.0)
    TP._upnp_problem(rs, 8, 0.0)
    upnp("upnp_cpu", [TP._upnp_problem(rs, 8 + trial, 0.0 if trial % 2 == 0 else 0.5) for trial in range(12)])
    rs = np.random.RandomState(21)
    upnp("upnp_gpu", [TP._upnp_problem(rs, 9, 0.0 if i % 2 == 0 else 0.4) for i in range(10)])
    return out


def make_cuda():
    import torch

    import test_gpu_parity as TG
    from conftest import load_ref_ext

    dev = torch.device("cuda:0")
    exts = {n: load_ref_ext(n) for n in ("ransac_voting", "torch_nndistance_aten", "flow_cuda")}
    missing = [n for n, m in exts.items() if m is None]
    if missing:
        raise SystemExit("oracle/_ref/%s not built (python oracle/build_ref.py --cuda-refs)" % missing)
    out = {"device": torch.cuda.get_device_name(dev)}
    rv = exts["ransac_voting"]
    for tn, vn, hn, seed in TG.VOTING_REF_CASES:
        direct, coords, idxs = TG._voting_inputs(tn, vn, hn, seed)
        out[TG.voting_ref_key(tn, vn, hn) + "/inputs_sha256"] = TG.sha256(direct, coords, idxs)
        D, C, I = (torch.from_numpy(a).to(dev) for a in (direct, coords, idxs))
        for vp in (False, True):
            key = TG.voting_ref_key(tn, vn, hn, vp)
            h = (rv.generate_hypothesis_vanishing_point if vp else rv.generate_hypothesis)(D, C, I)
            inl = torch.zeros((hn, vn, tn), dtype=torch.uint8, device=dev)
            (rv.voting_for_hypothesis_vanishing_point if vp else rv.voting_for_hypothesis)(D, C, h, inl, 0.99 if vp else 0.999)
            torch.cuda.synchronize()
            inl = inl.cpu().numpy()
            out[key + "/hyp"] = h.cpu().numpy()
            out[key + "/counts"] = inl.sum(2, dtype=np.int32)
            out[key + "/inliers_sha256"] = TG.sha256(inl)
    a, b = TG.nnd_ref_inputs()
    out["nnd/inputs_sha256"] = TG.sha256(a, b)
    for name, x in TG.nnd_forward(exts["torch_nndistance_aten"], torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev)).items():
        out.update(TG.golden_record("nnd/" + name, x.cpu().numpy()))
    for B, H, W in TG.FLOW_CASES:
        key = TG.flow_ref_key(B, H, W)
        ds, dt, KT, Kinv = TG._flow_inputs(B, H, W, seed=H)
        out[key + "/inputs_sha256"] = TG.sha256(ds, dt, KT, Kinv)
        fl, va = exts["flow_cuda"].forward(*(torch.from_numpy(x).to(dev) for x in (ds, dt, KT, Kinv)))
        torch.cuda.synchronize()
        out.update(TG.golden_record(key + "/flow", fl.cpu().numpy()))
        out.update(TG.golden_record(key + "/valid", va.cpu().numpy()))
    return out


if __name__ == "__main__":
    if len(sys.argv) < 2 or sys.argv[1] not in ("cpu", "cuda"):
        raise SystemExit(__doc__)
    kind = sys.argv[1]
    path = sys.argv[2] if len(sys.argv) > 2 else os.path.join(ROOT, "tests", "golden", "ref_%s_ops.npz" % kind)
    data = make_cpu() if kind == "cpu" else make_cuda()
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    np.savez_compressed(path, **data)
    print("wrote", path, os.path.getsize(path))
