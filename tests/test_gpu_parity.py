"""GPU parity tests (run on the B200 box): the CUDA path, called through the C ABI, against the oracle on the
same seeded inputs -- bit-exact for integer / index / mask work, stated tolerances for floating point.
The REFERENCE's own CUDA extensions (built for sm_100a) were run on the same inputs; their outputs are stored in
tests/golden/ref_cuda_ops.npz (tools/make_golden_ref_ops.py) and compared against here."""
import ctypes
import hashlib
import os

import numpy as np
import pytest
import torch

from conftest import ROOT, load_ref_ext
from oracle import gdrn_model_oracle as O
from oracle import ops_oracle as OO

pytestmark = pytest.mark.gpu

GOLD_CUDA = os.path.join(ROOT, "tests", "golden", "ref_cuda_ops.npz")


def _lib():
    from gdrnpp_bop2022_b200 import _lib

    return _lib


# ------------------------------------------------------------------------ stored outputs of the reference's kernels
# Outputs too large to store whole (inlier masks, flow fields) are kept as the SHA-256 of their bytes plus a seeded
# sample of elements; the inputs' SHA-256 is stored too, so that a changed input recipe is reported as such.
def sha256(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def _sample_idx(n, k=512):
    return np.random.RandomState(0).randint(0, n, min(n, k))


def golden_record(key, a):
    """{key/sha256, key/sample} for array ``a`` (what tools/make_golden_ref_ops.py stores)."""
    a = np.ascontiguousarray(a)
    return {key + "/sha256": sha256(a), key + "/sample": a.reshape(-1)[_sample_idx(a.size)]}


def assert_matches_golden(g, key, a):
    a = np.ascontiguousarray(a)
    ref = g[key + "/sample"]
    got = a.reshape(-1)[_sample_idx(a.size)]
    assert got.dtype == ref.dtype and np.array_equal(got.view(np.uint8), ref.view(np.uint8)), key   # bitwise
    assert sha256(a) == str(g[key + "/sha256"]), key


def assert_same_inputs(g, key, *arrays):
    assert sha256(*arrays) == str(g[key + "/inputs_sha256"]), \
        "%s: inputs differ from those the stored reference outputs were made from (tools/make_golden_ref_ops.py)" % key


# ------------------------------------------------------------------------------------------------ GEMM
@pytest.mark.parametrize("M,N,K,bn,epi,f32", [
    (128, 128, 64, 128, 0, 1), (300, 128, 64, 128, 0, 0), (128, 256, 256, 256, 0, 1), (1000, 512, 128, 256, 1, 0),
    (4096, 128, 512, 128, 2, 1), (4096, 256, 1024, 256, 2, 1), (64, 1024, 8192, 64, 1, 0), (64, 9, 256, 16, 0, 1),
    (1, 256, 64, 256, 0, 1), (129, 512, 2048, 256, 1, 0),
    # CTA-pair (cta_group::2) kernel: M >= 4096, BLOCK_N 256; ragged M (odd number of 128-row tiles + a partial tile),
    # short K with the 16-warp GELU epilogue, fp32 and bf16 plain stores
    (4296, 512, 1024, 256, 1, 0), (4224, 256, 128, 256, 1, 0), (8192, 256, 2048, 256, 0, 1), (4100, 256, 1024, 256, 0, 0),
])
def test_gemm_vs_torch(dev, lib, M, N, K, bn, epi, f32):
    """tcgen05 kernel vs a plain fp32 torch reference of the same op (bf16 operands, fp32 accumulate)."""
    L = _lib()
    g = torch.Generator().manual_seed(M * 7 + N * 3 + K)
    A = (torch.randn(M, K, generator=g) * 0.5).to(dev).bfloat16()
    W = (torch.randn(N, K, generator=g) / np.sqrt(K)).to(dev).bfloat16()
    bias, gamma, resid = torch.randn(N, generator=g).to(dev), torch.rand(N, generator=g).to(dev), torch.randn(M, N, generator=g).to(dev)
    ref = A.float() @ W.float().t() + bias
    if epi == 1:
        ref = torch.nn.functional.gelu(ref)
    if epi == 2:
        ref = resid + gamma * ref
    is_f32 = epi == 2 or (epi == 0 and f32)
    out = torch.full((M, N), float("nan"), dtype=torch.float32 if is_f32 else torch.bfloat16, device=dev)
    L.check(lib.gdrn_gemm_bf16(L.ptr(A), L.ptr(W), L.ptr(bias), L.ptr(gamma), L.ptr(resid), L.ptr(out), M, N, K, epi,
                               int(f32), bn, L.current_stream()), "gemm")
    torch.cuda.synchronize()
    err = (out.float() - ref).abs().max().item()
    # fp32 outputs: accumulation-order noise only; bf16 outputs: half an ulp of bf16 at |x| <= 8 (2^-6)
    assert err < (2e-4 if is_f32 else 0.04), err


@pytest.mark.parametrize("M,N,K,bn", [(4096, 256, 1024, 256), (4296, 256, 1024, 256), (1000, 128, 512, 128), (300, 512, 128, 256)])
def test_gemm_residual_in_place(dev, lib, M, N, K, bn):
    """EPI_RESID with out == resid (how the model calls it): the epilogue turns into a TMA reduce-add
    (x += gamma*(acc+bias) performed by the L2).  M not a multiple of 128 checks the tensor-map row clipping."""
    L = _lib()
    g = torch.Generator().manual_seed(M + N + K)
    A = (torch.randn(M, K, generator=g) * 0.5).to(dev).bfloat16()
    W = (torch.randn(N, K, generator=g) / np.sqrt(K)).to(dev).bfloat16()
    bias, gamma = torch.randn(N, generator=g).to(dev), torch.rand(N, generator=g).to(dev)
    pad = torch.full((M + 256, N), 7.0, device=dev)      # canary rows behind the matrix must stay untouched
    x = torch.randn(M, N, generator=g).to(dev)
    pad[:M] = x
    ref = x + gamma * (A.float() @ W.float().t() + bias)
    L.check(lib.gdrn_gemm_bf16(L.ptr(A), L.ptr(W), L.ptr(bias), L.ptr(gamma), L.ptr(pad), L.ptr(pad), M, N, K, 2, 1, bn,
                               L.current_stream()), "gemm")
    torch.cuda.synchronize()
    assert (pad[:M] - ref).abs().max().item() < 2e-4
    assert torch.equal(pad[M:], torch.full((256, N), 7.0, device=dev))


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_gemm_gelu_modes(dev, lib, mode, monkeypatch):
    """The three epilogue GELU evaluations (fp32 ex2/rcp, packed half2 tanh.approx, fp32 tanh.approx) vs erf-GELU."""
    L = _lib()
    monkeypatch.setenv("GDRN_GELU_MODE", str(mode))
    g = torch.Generator().manual_seed(mode)
    M, N, K = 512, 512, 256
    A = (torch.randn(M, K, generator=g)).to(dev).bfloat16()
    W = (torch.randn(N, K, generator=g) * (3.0 / np.sqrt(K))).to(dev).bfloat16()   # pre-activations up to ~ +-12
    bias = torch.randn(N, generator=g).to(dev)
    pre = A.float() @ W.float().t() + bias
    ref = torch.nn.functional.gelu(pre)
    out = torch.empty((M, N), dtype=torch.bfloat16, device=dev)
    L.check(lib.gdrn_gemm_bf16(L.ptr(A), L.ptr(W), L.ptr(bias), None, None, L.ptr(out), M, N, K, 1, 0, 256,
                               L.current_stream()), "gemm")
    torch.cuda.synchronize()
    err = (out.float() - ref).abs()
    tol = 2.0 ** -8 * ref.abs().clamp_min(1.0) + (0.0 if mode == 0 else 6e-4 * pre.abs().clamp_min(1.0))
    assert (err <= tol).all(), float((err - tol).max())


def _split_bf16(t):
    hi = t.bfloat16()
    lo = (t - hi.float()).bfloat16()
    return torch.cat([hi, lo], dim=1).contiguous()


@pytest.mark.parametrize("M,N,K,bn,epi", [
    # CTA-pair split kernel (>= 48 pair tiles): GELU -> split bf16, fp32 store, in-place residual (TMA reduce-add),
    # BLOCK_N 128, ragged M (odd tile count + partial tile: the peer CTA of the last pair has no rows)
    (8192, 512, 256, 256, 1), (8192, 1024, 128, 256, 0), (12417, 256, 512, 256, 2), (16384, 128, 512, 128, 2),
    (12300, 128, 128, 128, 1), (16384, 512, 2048, 256, 2),
    # general kernel with the 3x tap list (too few tiles for the pairs, or BLOCK_N 64)
    (300, 128, 64, 128, 0), (1000, 512, 128, 256, 1), (64, 1024, 8192, 64, 1), (4096, 256, 1024, 256, 2),
    # narrow tiles the forward picks for small batches (B = 5: stage-2 / stage-3 fc2, stage-3 fc1)
    (1280, 512, 2048, 64, 2), (320, 1024, 4096, 64, 2), (320, 4096, 1024, 128, 1), (1280, 256, 512, 64, 0),
])
def test_gemm_x3_vs_fp64(dev, lib, M, N, K, bn, epi):
    """Split-bf16 ("bf16x3") GEMM -- the tensor-core path of the fp32-parity mode -- vs an fp64 torch reference of the
    same op on the ORIGINAL fp32 operands: the dropped lo*lo term and the hi+lo representation are ~2^-17 relative."""
    L = _lib()
    g = torch.Generator().manual_seed(M * 7 + N * 3 + K + epi)
    A = (torch.randn(M, K, generator=g) * 0.5).to(dev)
    W = (torch.randn(N, K, generator=g) / np.sqrt(K)).to(dev)
    bias, gamma = torch.randn(N, generator=g).to(dev), torch.rand(N, generator=g).to(dev)
    x = torch.randn(M, N, generator=g).to(dev)
    ref = A.double() @ W.double().t() + bias.double()
    if epi == 1:
        ref = torch.nn.functional.gelu(ref)
    if epi == 2:
        ref = x.double() + gamma.double() * ref
    A2, W2 = _split_bf16(A), _split_bf16(W)
    if epi == 1:
        out = torch.full((M + 64, 2 * N), float("nan"), dtype=torch.bfloat16, device=dev)
    else:
        out = torch.full((M + 64, N), 7.0, dtype=torch.float32, device=dev)   # canary rows behind the matrix
        if epi == 2:
            out[:M] = x
    L.check(lib.gdrn_gemm_x3(L.ptr(A2), L.ptr(W2), L.ptr(bias), L.ptr(gamma), L.ptr(out), L.ptr(out), M, N, K, epi, bn,
                             L.current_stream()), "gemm_x3")
    torch.cuda.synchronize()
    if epi == 1:
        got = out[:M, :N].double() + out[:M, N:].double()
        assert torch.isnan(out[M:].float()).all()
    else:
        got = out[:M].double()
        assert torch.equal(out[M:], torch.full((64, N), 7.0, device=dev))
    err = (got - ref).abs().max().item()
    assert err < 4e-5 * max(1.0, ref.abs().max().item()), err


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,K,bn", [
    (16384, 512, 2048, 256),    # stage-2 fc2 at B = 64: 128 tiles x 32 k-iterations on 74 pairs (tiles cut in two)
    (65536, 256, 1024, 256),    # stage-1 fc2: 256 tiles x 16
    (4096, 1024, 4096, 256),    # stage-3 fc2: 64 tiles x 64 (fewer tiles than pairs: some tiles are cut in THREE)
    (20000, 256, 1024, 256),    # ragged M, odd tile count (the peer CTA of the last pair has no rows)
    (16384, 128, 512, 128),     # BLOCK_N 128
])
def test_gemm_x3_ksplit_residual(dev, lib, M, N, K, bn):
    """Balanced k-split schedule of the CTA-pair split-bf16 kernel (in-place residual GEMMs whose tile count leaves the
    last wave partly empty): same result as the fp64 reference, run-to-run bit-identical (partial tiles are reduce-added
    in a fixed order), ordering words left at zero."""
    L = _lib()
    g = torch.Generator().manual_seed(M + N + K)
    A = (torch.randn(M, K, generator=g) * 0.5).to(dev)
    W = (torch.randn(N, K, generator=g) / np.sqrt(K)).to(dev)
    bias, gamma = torch.randn(N, generator=g).to(dev), torch.rand(N, generator=g).to(dev)
    x = torch.randn(M, N, generator=g).to(dev)
    ref = x.double() + gamma.double() * (A.double() @ W.double().t() + bias.double())
    A2, W2 = _split_bf16(A), _split_bf16(W)
    flags = torch.zeros(8192, dtype=torch.int32, device=dev)
    outs = []
    for _ in range(3):
        out = torch.full((M + 64, N), 7.0, dtype=torch.float32, device=dev)
        out[:M] = x
        L.check(lib.gdrn_gemm_x3_ksplit(L.ptr(A2), L.ptr(W2), L.ptr(bias), L.ptr(gamma), L.ptr(out), M, N, K, bn,
                                        L.ptr(flags), flags.numel(), L.current_stream()), "gemm_x3_ksplit")
        torch.cuda.synchronize()
        assert int(flags.abs().max().item()) == 0
        assert torch.equal(out[M:], torch.full((64, N), 7.0, device=dev))
        outs.append(out[:M].clone())
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])
    err = (outs[0].double() - ref).abs().max().item()
    assert err < 4e-5 * max(1.0, ref.abs().max().item()), err
    # whole-tile schedule (no flags): same sums up to the fp32 rounding of the partial adds
    whole = torch.full((M + 64, N), 7.0, dtype=torch.float32, device=dev)
    whole[:M] = x
    L.check(lib.gdrn_gemm_x3(L.ptr(A2), L.ptr(W2), L.ptr(bias), L.ptr(gamma), L.ptr(whole), L.ptr(whole), M, N, K, 2, bn,
                             L.current_stream()), "gemm_x3")
    torch.cuda.synchronize()
    assert (whole[:M] - outs[0]).abs().max().item() < 2e-5 * max(1.0, ref.abs().max().item())


@pytest.mark.gpu
def test_mlp_fused_x3_vs_unfused_and_fp64(dev, lib):
    """Fused fc1 -> GELU -> fc2 -> residual of the split-bf16 mode (ConvNeXt stage 0, C = 128; the hidden activation stays on
    chip) against (a) the two-kernel path it replaces -- same products in the same accumulation order -- and (b) an fp64
    torch reference of timm's ConvNeXtBlock MLP half on the original fp32 operands."""
    L = _lib()
    C, M = 128, 128 * 148 * 2 + 128 * 5          # two full waves + a ragged third
    g = torch.Generator().manual_seed(11)
    A = (torch.randn(M, C, generator=g) * 0.7).to(dev)
    W1 = (torch.randn(4 * C, C, generator=g) / np.sqrt(C)).to(dev)
    W2 = (torch.randn(C, 4 * C, generator=g) / np.sqrt(4 * C)).to(dev)
    b1, b2, gamma = torch.randn(4 * C, generator=g).to(dev), torch.randn(C, generator=g).to(dev), torch.rand(C, generator=g).to(dev)
    x0 = torch.randn(M, C, generator=g).to(dev)
    h = torch.nn.functional.gelu(A.double() @ W1.double().t() + b1.double())
    ref = x0.double() + gamma.double() * (h @ W2.double().t() + b2.double())
    A2, W12, W22 = _split_bf16(A), _split_bf16(W1), _split_bf16(W2)
    # unfused: fc1 (epi 1 -> split hidden) then fc2 (epi 2, in place)
    Hb = torch.empty(M, 8 * C, dtype=torch.bfloat16, device=dev)
    x_un = x0.clone()
    L.check(lib.gdrn_gemm_x3(L.ptr(A2), L.ptr(W12), L.ptr(b1), None, None, L.ptr(Hb), M, 4 * C, C, 1, 256, L.current_stream()), "fc1")
    L.check(lib.gdrn_gemm_x3(L.ptr(Hb), L.ptr(W22), L.ptr(b2), L.ptr(gamma), L.ptr(x_un), L.ptr(x_un), M, C, 4 * C, 2, 128,
                             L.current_stream()), "fc2")
    x_fu = torch.cat([x0.clone(), torch.full((64, C), 7.0, device=dev)])       # canary rows behind the matrix
    L.check(lib.gdrn_mlp_fused_x3(L.ptr(A2), L.ptr(W12), L.ptr(b1), L.ptr(W22), L.ptr(b2), L.ptr(gamma), L.ptr(x_fu), M, C,
                                  L.current_stream()), "mlp_fused_x3")
    torch.cuda.synchronize()
    assert torch.equal(x_fu[M:], torch.full((64, C), 7.0, device=dev))
    err = (x_fu[:M].double() - ref).abs().max().item()
    assert err < 4e-5 * max(1.0, ref.abs().max().item()), err
    d = (x_fu[:M] - x_un).abs().max().item()
    assert d < 2e-6 * max(1.0, ref.abs().max().item()), d     # same math; fp32 reduce-add order aside, the two paths agree


# ----------------------------------------------------------------------------------------------- model
def _run_model(dev, B, seed, with_maps=True, precision="bf16"):
    from gdrnpp_bop2022_b200.gdrn_model import GDRN_DoubleMask, default_cfg
    from gdrnpp_bop2022_b200.synthetic import make_batch, make_state_dict

    sd = make_state_dict()   # the SAME weights bench.py and smoke() use (no per-test overrides)
    batch = make_batch(B=B, seed=seed)
    model = GDRN_DoubleMask(default_cfg(with_maps=with_maps), max_batch=max(B, 2), precision=precision)
    model.load_state_dict(sd)
    model.to(dev)
    gb = {k: v.to(dev) for k, v in batch.items()}
    out = model(gb["roi_img"], roi_classes=gb["roi_classes"], roi_coord_2d=gb["roi_coord_2d"], roi_cams=gb["roi_cams"],
                roi_centers=gb["roi_centers"], roi_whs=gb["roi_whs"], roi_extents=gb["roi_extents"],
                resize_ratios=gb["resize_ratios"], return_raw=True)
    torch.cuda.synchronize()
    return sd, batch, model, out


def _rot_err(Ra, Rb):
    """Rotation angle between two batches of rotation matrices: |Ra-Rb|_F = 2*sqrt(2)*sin(theta/2).
    (acos((tr-1)/2) has a ~4e-4 rad noise floor for float32 matrices; this form is exact for small angles.)"""
    d = (Ra.double() - Rb.double()).flatten(1).norm(dim=1)
    return 2 * torch.asin((d / (2 * 2 ** 0.5)).clamp(max=1.0))


@pytest.mark.parametrize("B", [1, 3, 8])
def test_forward_vs_oracle_bf16(dev, B):
    """Whole dense path (bf16 tensor-core mode) vs the fp32 oracle.  Tolerances for dtype 'bf16' (DESIGN.md
    'numerics'): conv features 2% relative L2, maps 0.15 abs, R within 0.1 rad, t within 1e-2; the 1e-4 rad /
    1e-3 bar of BASELINE.json is an fp32-class bar that bf16 operands cannot reach (SURVEY.md §7)."""
    sd, batch, model, out = _run_model(dev, B, seed=40 + B)
    with torch.no_grad():
        ref = O.gdrn_forward(sd, batch, return_maps=True, return_intermediate=True)
    feat = model.debug_read("conv_feat", B, B * 64 * 1024).reshape(B, 8, 8, 1024).permute(0, 3, 1, 2).cpu()
    rel = ((feat - ref["conv_feat"]).norm() / ref["conv_feat"].norm()).item()
    assert rel < 0.02, rel
    for k in ("mask", "full_mask", "coor_x", "coor_y", "coor_z", "region"):
        assert (out[k].cpu() - ref[k]).abs().max().item() < 0.15, k
    raw = out["raw"].cpu()
    assert (raw[:, :6] - ref["rot6d"]).abs().max().item() < 0.06
    assert (raw[:, 6:] - ref["t_"]).abs().max().item() < 0.02
    assert _rot_err(out["rot"].cpu(), ref["rot"]).max().item() < 0.1
    assert (out["trans"].cpu() - ref["trans"]).abs().max().item() < 1e-2


def _rot6d_conditioning(rot6d):
    """Gram-Schmidt amplification of rot6d -> R (core/utils/rot_reps.py:34-55): a perturbation e of the 6-D vector moves
    R by ~ e / min(|a1|, |a2 - (a2.x)x|).  A trained head emits near-orthonormal pairs (kappa ~ 1); random-init weights
    occasionally emit a short a1 and then ANY fp32 implementation (cuBLAS vs MKL included) moves R by kappa x its own
    round-off."""
    a1, a2 = rot6d[:, :3].double(), rot6d[:, 3:].double()
    n1 = a1.norm(dim=1)
    x = a1 / n1[:, None]
    a2p = a2 - (a2 * x).sum(1, keepdim=True) * x
    return 1.0 / torch.minimum(n1, a2p.norm(dim=1))


@pytest.mark.parametrize("B", [1, 5, 16])
def test_forward_vs_oracle_north_star_tolerance(dev, B):
    """BASELINE.json north_star parity bar, met by the split-bf16 ("bf16x3") precision mode with the unmodified
    make_state_dict() weights: t within 1e-3, the raw Patch-PnP output (rot6d, t_) within 1e-4 and the maps within 2e-3
    of the fp32 oracle (= the reference's fp32 forward, pinned by tests/golden/ref_heads.npz and torchvision), and R within
    1e-4 rad x max(1, kappa) where kappa is the oracle rot6d's own Gram-Schmidt conditioning (1 for the O(1)-norm vectors
    a trained head emits; the seed-76 batch holds one random-init ROI with |a1| = 0.13, kappa = 7.4).  The un-scaled
    1e-4 rad bar is asserted on the bench's own batch in test_forward_vs_oracle_b64."""
    sd, batch, model, out = _run_model(dev, B, seed=60 + B, precision="bf16x3")
    with torch.no_grad():
        ref = O.gdrn_forward(sd, batch, return_maps=True, return_intermediate=True)
    x3 = model.debug_read("stage3_x", B, B * 64 * 1024).reshape(B, 8, 8, 1024).permute(0, 3, 1, 2).cpu()
    rel = ((x3 - ref["conv_feat"]).norm() / ref["conv_feat"].norm()).item()
    assert rel < 1e-4, rel
    for k in ("mask", "full_mask", "coor_x", "coor_y", "coor_z", "region"):
        assert (out[k].cpu() - ref[k]).abs().max().item() < 2e-3, k
    raw = out["raw"].cpu()
    assert (raw[:, :6] - ref["rot6d"]).abs().max().item() < 1e-4
    assert (raw[:, 6:] - ref["t_"]).abs().max().item() < 1e-4
    rerr = _rot_err(out["rot"].cpu(), ref["rot"])
    kappa = _rot6d_conditioning(ref["rot6d"]).clamp_min(1.0)
    terr = (out["trans"].cpu() - ref["trans"]).abs().max().item()
    assert (rerr < 1e-4 * kappa).all(), (rerr, kappa)   # north_star: R within 1e-4 rad (at unit conditioning)
    assert terr < 1e-3, terr                           # north_star: t within 1e-3


@pytest.mark.parametrize("arch,B", [("convnext_tiny", 4), ("convnext_small", 2)])
def test_forward_vs_oracle_convnext_tiny_small(dev, arch, B):
    """The other ConvNeXt widths the reference's backbone factory accepts (models/net_factory.py:73-74; BASELINE configs[0]
    names convnext_tiny): dims 96/192/384/768.  The 96-channel first stage is stored 128 wide with zero pad channels and the
    LayerNorms take their statistics over the 96 real channels; both precision modes against the fp32 oracle (whose backbone
    is pinned to torchvision's convnext_tiny / convnext_small in test_oracle_pinning.py)."""
    from gdrnpp_bop2022_b200.gdrn_model import GDRN_DoubleMask, default_cfg
    from gdrnpp_bop2022_b200.synthetic import make_batch, make_state_dict

    sd = make_state_dict(arch=arch)
    batch = make_batch(B=B, seed=90 + B)
    with torch.no_grad():
        ref = O.gdrn_forward(sd, batch, arch=arch, return_maps=True, return_intermediate=True)
    gb = {k: v.to(dev) for k, v in batch.items()}
    for precision in ("bf16x3", "bf16"):
        model = GDRN_DoubleMask(default_cfg(arch=arch, with_maps=True), arch=arch, max_batch=max(B, 2), precision=precision)
        model.load_state_dict(sd)
        model.to(dev)
        out = model(gb["roi_img"], roi_classes=gb["roi_classes"], roi_coord_2d=gb["roi_coord_2d"], roi_cams=gb["roi_cams"],
                    roi_centers=gb["roi_centers"], roi_whs=gb["roi_whs"], roi_extents=gb["roi_extents"],
                    resize_ratios=gb["resize_ratios"], return_raw=True)
        torch.cuda.synchronize()
        x3 = model.debug_read("stage3_x", B, B * 64 * 768).reshape(B, 8, 8, 768).permute(0, 3, 1, 2).cpu()
        rel = ((x3 - ref["conv_feat"]).norm() / ref["conv_feat"].norm()).item()
        raw = out["raw"].cpu()
        rerr = _rot_err(out["rot"].cpu(), ref["rot"])
        terr = (out["trans"].cpu() - ref["trans"]).abs().max().item()
        if precision == "bf16x3":
            assert rel < 1e-4, rel
            for k in ("mask", "full_mask", "coor_x", "coor_y", "coor_z", "region"):
                assert (out[k].cpu() - ref[k]).abs().max().item() < 2e-3, k
            assert (raw[:, :6] - ref["rot6d"]).abs().max().item() < 1e-4
            assert (raw[:, 6:] - ref["t_"]).abs().max().item() < 1e-4
            kappa = _rot6d_conditioning(ref["rot6d"]).clamp_min(1.0)
            assert (rerr < 1e-4 * kappa).all(), (rerr, kappa)
            assert terr < 1e-3, terr
        else:
            assert rel < 0.02, rel
            assert rerr.max().item() < 0.1 and terr < 1e-2, (rerr, terr)


@pytest.mark.parametrize("precision", ["bf16x3", "bf16"])
def test_forward_vs_oracle_b64(dev, precision):
    """BASELINE.json configs[1] at its full size: the bench's own first batch (B = 64, seed 0, unmodified
    make_state_dict() weights) against the fp32 oracle.  At B = 64 every GEMM takes the kernel the bench times (CTA-pair
    kernels from M >= 4096 rows, the fused stage-0 MLP in bf16 mode) -- paths the small-batch tests do not reach.
    bf16x3 (the mode of record): north-star bar R < 1e-4 rad, t < 1e-3.  bf16 (secondary throughput mode): its own
    documented tolerances."""
    sd, batch, model, out = _run_model(dev, 64, seed=0, precision=precision)
    with torch.no_grad():
        ref = O.gdrn_forward(sd, batch, return_maps=True, return_intermediate=True)
    rerr = _rot_err(out["rot"].cpu(), ref["rot"]).max().item()
    terr = (out["trans"].cpu() - ref["trans"]).abs().max().item()
    raw = out["raw"].cpu()
    if precision == "bf16x3":
        x3 = model.debug_read("stage3_x", 64, 64 * 64 * 1024).reshape(64, 8, 8, 1024).permute(0, 3, 1, 2).cpu()
        assert ((x3 - ref["conv_feat"]).norm() / ref["conv_feat"].norm()).item() < 1e-4
        for k in ("mask", "full_mask", "coor_x", "coor_y", "coor_z", "region"):
            assert (out[k].cpu() - ref[k]).abs().max().item() < 2e-3, k
        assert (raw[:, :6] - ref["rot6d"]).abs().max().item() < 1e-4
        assert rerr < 1e-4, rerr
        assert terr < 1e-3, terr
        # run-to-run determinism at the bench's batch size (the k-split fc2 GEMMs add partial tiles in a fixed order; the
        # GroupNorm sums are double atomics whose order noise disappears in the float rounding of mean / rstd)
        gb = {k: v.to(dev) for k, v in batch.items()}
        out2 = model(gb["roi_img"], roi_classes=gb["roi_classes"], roi_coord_2d=gb["roi_coord_2d"], roi_cams=gb["roi_cams"],
                     roi_centers=gb["roi_centers"], roi_whs=gb["roi_whs"], roi_extents=gb["roi_extents"],
                     resize_ratios=gb["resize_ratios"], return_raw=True)
        torch.cuda.synchronize()
        x3b = model.debug_read("stage3_x", 64, 64 * 64 * 1024).reshape(64, 8, 8, 1024).permute(0, 3, 1, 2).cpu()
        assert torch.equal(x3, x3b)
        assert (out2["rot"] - out["rot"]).abs().max().item() < 1e-6
    else:
        for k in ("mask", "full_mask", "coor_x", "coor_y", "coor_z", "region"):
            assert (out[k].cpu() - ref[k]).abs().max().item() < 0.15, k
        assert rerr < 0.1 and terr < 1e-2, (rerr, terr)


def test_sharded_4096_rois_vs_oracle_sample(dev):
    """BASELINE.json configs[3]: 4096 ROIs in contiguous shards of 512 (dist.shard_range, 8 ranks), 64 ROIs per step
    through one captured CUDA graph, poses packed / gathered in rank order like dist.all_gather_poses.  Here the 8
    shards run back to back on one GPU (the NCCL gather itself is covered by the gloo world-2 test and by
    bench.py --gpus N); three ROIs of every shard are checked against the fp32 oracle at the north-star bar."""
    from gdrnpp_bop2022_b200.dist import pack_poses, shard_range, unpack_poses
    from gdrnpp_bop2022_b200.gdrn_model import GDRN_DoubleMask, default_cfg
    from gdrnpp_bop2022_b200.synthetic import make_batch, make_state_dict

    total, world, step = 4096, 8, 64
    sd = make_state_dict()
    model = GDRN_DoubleMask(default_cfg(), max_batch=step, precision="bf16x3")
    model.load_state_dict(sd)
    model.to(dev)
    keys = ("roi_img", "roi_classes", "roi_coord_2d", "roi_cams", "roi_centers", "roi_whs", "resize_ratios", "roi_extents")
    static = {k: v.to(dev) for k, v in make_batch(B=step, seed=1).items() if k in keys}
    replay, out = model.capture_graph(static)
    gathered, sample_in, sample_idx = [], {k: [] for k in keys}, []
    rs = np.random.RandomState(4)
    for rank in range(world):
        b, e = shard_range(total, rank, world)
        assert (e - b) == 512 and b % step == 0
        local = []
        picks = set((b + rs.choice(e - b, 3, replace=False)).tolist())
        for s0 in range(b, e, step):
            hb = make_batch(B=step, seed=1 + s0 // step)     # ROI i lives in step i // 64 (seed 1 + step), slot i % 64
            for k in keys:
                static[k].copy_(hb[k])
            replay()
            local.append(pack_poses(out["rot"], out["trans"]).clone())
            for i in range(s0, s0 + step):
                if i in picks:
                    sample_idx.append(i)
                    for k in keys:
                        sample_in[k].append(hb[k][i - s0])
        gathered.append(torch.cat(local))
    rot, trans = unpack_poses(torch.cat(gathered))
    torch.cuda.synchronize()
    assert rot.shape == (total, 3, 3) and trans.shape == (total, 3)
    assert torch.isfinite(rot).all() and torch.isfinite(trans).all()
    # rotations are orthonormal over the whole job (size-independent property)
    eye = torch.eye(3, device=dev)
    assert ((rot @ rot.transpose(1, 2)) - eye).abs().max().item() < 1e-5
    sb = {k: torch.stack(v) for k, v in sample_in.items()}
    with torch.no_grad():
        ref = O.gdrn_forward(sd, sb, return_intermediate=True)
    idx = torch.tensor(sample_idx)
    kappa = _rot6d_conditioning(ref["rot6d"]).clamp_min(1.0)   # see test_forward_vs_oracle_north_star_tolerance
    assert (_rot_err(rot[idx].cpu(), ref["rot"]) < 1e-4 * kappa).all()
    assert (trans[idx].cpu() - ref["trans"]).abs().max().item() < 1e-3


def test_precisions_agree_and_report(dev):
    """The throughput mode (bf16) stays within its documented distance of the precise mode on the same inputs."""
    _, _, m1, o1 = _run_model(dev, 4, seed=9, precision="bf16")
    _, _, m2, o2 = _run_model(dev, 4, seed=9, precision="bf16x3")
    assert m1.precision == "bf16" and m2.precision == "bf16x3"
    assert _rot_err(o1["rot"].cpu(), o2["rot"].cpu()).max().item() < 0.1
    assert (o1["trans"] - o2["trans"]).abs().max().item() < 1e-2


def test_pose_lift_exact_given_head_output(dev):
    """rot6d -> R, centroid/z -> t, allo -> ego on the device vs the oracle's numpy/float64 path fed with the SAME
    Patch-PnP output: R within 1e-4 rad (measured ~1e-7), t within 1e-6 relative."""
    sd, batch, model, out = _run_model(dev, 8, seed=77, precision="bf16")
    raw = out["raw"].cpu()
    Rm = O.rot6d_to_mat_batch(raw[:, :6])
    ego, trans = O.pose_from_predictions_test(Rm, raw[:, 6:8], raw[:, 8:9], batch["roi_cams"], batch["roi_centers"],
                                              batch["resize_ratios"], batch["roi_whs"])
    # The reference's allo->ego step takes acos() of a float32 cosine (core/utils/utils.py:49-50): for a ROI at angle
    # a from the optical axis, one float32 ulp in |t| moves the result by ~6e-8/sin(a) rad, and numpy's float32 norm
    # (BLAS sdot) is itself platform dependent at that level -> tolerance 1e-4 + 4 ulp / sin(a).
    t = trans.double()
    sin_a = (t[:, :2].norm(dim=1) / t.norm(dim=1)).clamp_min(1e-6)
    tol = 1e-4 + 4 * 6e-8 / sin_a
    assert (_rot_err(out["rot"].cpu(), ego) < tol).all(), (_rot_err(out["rot"].cpu(), ego), tol)
    assert (out["trans"].cpu() - trans).abs().max().item() < 1e-6


def test_forward_is_deterministic_and_batch_invariant(dev):
    """Size-independent property: a ROI's pose does not depend on its batch neighbours (ROIs shard freely)."""
    from gdrnpp_bop2022_b200.gdrn_model import GDRN_DoubleMask, default_cfg
    from gdrnpp_bop2022_b200.synthetic import make_batch, make_state_dict

    sd = make_state_dict()
    model = GDRN_DoubleMask(default_cfg(), max_batch=8)   # default precision = bf16x3, the mode of record
    assert model.precision == "bf16x3"
    model.load_state_dict(sd)
    model.to(dev)
    b8 = {k: v.to(dev) for k, v in make_batch(B=8, seed=5).items()}
    kw = lambda b: dict(roi_classes=b["roi_classes"], roi_coord_2d=b["roi_coord_2d"], roi_cams=b["roi_cams"],
                        roi_centers=b["roi_centers"], roi_whs=b["roi_whs"], roi_extents=b["roi_extents"],
                        resize_ratios=b["resize_ratios"])
    o8 = model(b8["roi_img"], **kw(b8))
    o8b = model(b8["roi_img"], **kw(b8))
    b3 = {k: v[2:5].contiguous() for k, v in b8.items()}
    o3 = model(b3["roi_img"], **kw(b3))
    torch.cuda.synchronize()
    assert torch.equal(o8["rot"], o8b["rot"]) and torch.equal(o8["trans"], o8b["trans"])
    # GroupNorm statistics are accumulated with double atomics -> order noise ~1e-16 relative only
    assert (o8["rot"][2:5] - o3["rot"]).abs().max().item() < 1e-3
    assert (o8["trans"][2:5] - o3["trans"]).abs().max().item() < 1e-4


def test_fused_mlp_matches_unfused(dev, monkeypatch):
    """Stage-0 blocks run fc1 -> GELU -> fc2 -> residual in one kernel when the batch is large enough (B >= 5); the
    two-kernel path must give the same poses (same operands, same accumulation order; only scheduling differs)."""
    outs = []
    for fused in ("0", "1"):
        monkeypatch.setenv("GDRN_MLP_FUSED", fused)
        _, _, _, out = _run_model(dev, 8, seed=21, precision="bf16")   # the fused kernel is a bf16-mode kernel
        outs.append(out)
    assert _rot_err(outs[0]["rot"].cpu(), outs[1]["rot"].cpu()).max().item() < 1e-3
    assert (outs[0]["trans"] - outs[1]["trans"]).abs().max().item() < 1e-4
    for k in ("mask", "coor_x", "region"):
        assert (outs[0][k] - outs[1][k]).abs().max().item() < 2e-2, k


def test_forward_error_paths(dev, lib):
    from gdrnpp_bop2022_b200 import _lib as L
    from gdrnpp_bop2022_b200.gdrn_model import GDRN_DoubleMask, default_cfg

    m = GDRN_DoubleMask(default_cfg())
    x = torch.zeros(1, 3, 256, 256)
    with pytest.raises(L.GdrnError):
        m(x, roi_classes=torch.zeros(1, dtype=torch.long), roi_coord_2d=torch.zeros(1, 2, 64, 64), roi_cams=torch.eye(3)[None],
          roi_centers=torch.zeros(1, 2), roi_whs=torch.ones(1, 2), roi_extents=torch.ones(1, 3), resize_ratios=torch.ones(1))
    h = ctypes.c_void_p()
    assert lib.gdrn_model_create(ctypes.byref(h), b"resnet34", 21, 4) != 0
    assert b"unknown arch" in lib.gdrn_last_error()
    assert lib.gdrn_model_create(ctypes.byref(h), b"convnext_base", 21, 4) == 0
    t = torch.zeros(10, device=dev)
    assert lib.gdrn_model_load_tensor(h, b"backbone.no_such.weight", L.ptr(t), 10, None) != 0
    assert lib.gdrn_model_load_tensor(h, b"backbone.stem_0.bias", L.ptr(t), 10, None) != 0  # wrong size
    assert lib.gdrn_model_missing(h) > 0
    lib.gdrn_model_destroy(h)


# ------------------------------------------------------------------------------------------------- FPS
@pytest.mark.parametrize("pn,sn", [(1, 1), (7, 7), (100, 16), (4096, 64), (8192, 64), (14000, 32), (30000, 64)])
def test_fps_bit_exact(dev, pn, sn):
    from gdrnpp_bop2022_b200 import native_ops

    rs = np.random.RandomState(pn)
    pts = ((rs.rand(2, pn, 3) - 0.5) * 0.2).astype(np.float32)
    if pn == 100:
        pts[0, 10:30] = pts[0, 3]
    idx = native_ops.farthest_point_sampling_idx(torch.from_numpy(pts).to(dev), sn).cpu().numpy()
    for b in range(2):
        assert (idx[b] == OO.fps(pts[b], sn)).all(), (pn, sn, b)
    start = torch.tensor([0, pn - 1], dtype=torch.int32)
    idx2 = native_ops.farthest_point_sampling_idx(torch.from_numpy(pts).to(dev), sn, start_idx=start).cpu().numpy()
    for b in range(2):
        assert (idx2[b] == OO.fps(pts[b], sn, start=int(start[b]))).all()


@pytest.mark.parametrize("pn,sn", [(60000, 24), (150001, 16), (300000, 12), (20000, 40), (50000, 32)])
def test_fps_large_clouds_cluster_bit_exact(dev, pn, sn):
    """pn > 56 000 (meshes reach 10^5 vertices): a cluster of 2 / 4 / 8 CTAs shares one cloud; same indices as the
    reference algorithm (core/csrc/fps/src/farthest_point_sampling.cpp:118-160 handles any pn).  The last two cases are
    few mid-size clouds (16 384 <= pn <= 56 000), which also run on a cluster so that the SMs are not left idle."""
    from gdrnpp_bop2022_b200 import native_ops

    rs = np.random.RandomState(pn % 1000)
    pts = ((rs.rand(2, pn, 3) - 0.5) * np.array([0.3, 0.2, 0.1])).astype(np.float32)
    pts[1, 1000:1100] = pts[1, 7]            # duplicates: ties resolved by the lowest index across CTA boundaries too
    idx = native_ops.farthest_point_sampling_idx(torch.from_numpy(pts).to(dev), sn).cpu().numpy()
    for b in range(2):
        assert (idx[b] == OO.fps(pts[b], sn)).all(), (pn, b)
    start = torch.tensor([pn - 1, pn // 2], dtype=torch.int32)
    idx2 = native_ops.farthest_point_sampling_idx(torch.from_numpy(pts).to(dev), sn, start_idx=start).cpu().numpy()
    for b in range(2):
        assert (idx2[b] == OO.fps(pts[b], sn, start=int(start[b]))).all()


def test_fps_golden_and_host_entry(dev):
    from gdrnpp_bop2022_b200 import native_ops

    g = np.load(os.path.join(ROOT, "tests", "golden", "fps_golden.npz"))
    for i in range(int(g["n_cases"])):
        pts, idx = g[f"pts_{i}"], g[f"idx_{i}"]
        got = native_ops.farthest_point_sampling(pts, len(idx), init_center=True)  # reference-style numpy API
        assert np.array_equal(got, pts[idx]), i
    sel = native_ops.farthest_point_sampling(g["pts_2"], 16, init_center=False)  # random start: valid distinct points
    assert sel.shape == (16, 3) and len({tuple(r) for r in sel}) == 16


# ---------------------------------------------------------------------------------------------- voting
def _voting_inputs(tn, vn, hn, seed, noise=0.05):
    rs = np.random.RandomState(seed)
    coords = (rs.rand(tn, 2) * 200).astype(np.float32)
    kp = (rs.rand(vn, 2) * 200).astype(np.float32)
    d = kp[None] - coords[:, None] + rs.randn(tn, vn, 2) * noise * 200
    direct = (d / np.linalg.norm(d, axis=2, keepdims=True)).astype(np.float32)
    direct[::97] = 0  # zero-norm directions (norm1 < 1e-6 branch)
    idxs = rs.randint(0, tn, (hn, vn, 2)).astype(np.int32)
    idxs[0, :, 1] = idxs[0, :, 0]  # degenerate pairs (|det| < 1e-6 branch)
    return direct, coords, idxs


@pytest.mark.parametrize("tn,vn,hn", [(5, 1, 1), (2048, 9, 128), (3001, 8, 33)])
@pytest.mark.parametrize("vp", [False, True])
def test_voting_bit_exact(dev, tn, vn, hn, vp):
    from gdrnpp_bop2022_b200.native_ops import ransac_voting as rv

    direct, coords, idxs = _voting_inputs(tn, vn, hn, seed=tn + vn)
    D, C, I = (torch.from_numpy(a).to(dev) for a in (direct, coords, idxs))
    hyp = (rv.generate_hypothesis_vanishing_point if vp else rv.generate_hypothesis)(D, C, I)
    hyp_o = OO.generate_hypothesis(direct, coords, idxs, vanishing_point=vp)
    assert np.array_equal(hyp.cpu().numpy().view(np.uint32), hyp_o.view(np.uint32))
    inl = torch.zeros((hn, vn, tn), dtype=torch.uint8, device=dev)
    thr = 0.99 if vp else 0.999
    (rv.voting_for_hypothesis_vanishing_point if vp else rv.voting_for_hypothesis)(D, C, hyp, inl, thr)
    inl_o, cnt_o = OO.voting(direct, coords, hyp_o, thr, vanishing_point=vp)
    assert np.array_equal(inl.cpu().numpy(), inl_o)                      # bit-exact inlier sets
    cnt = rv.vote_count(D, C, hyp, thr, vanishing_point=vp).cpu().numpy()
    assert np.array_equal(cnt, cnt_o)                                    # fused count == sum of the mask
    # in/out semantics: existing ones survive
    inl2 = torch.ones((hn, vn, tn), dtype=torch.uint8, device=dev)
    (rv.voting_for_hypothesis_vanishing_point if vp else rv.voting_for_hypothesis)(D, C, hyp, inl2, thr)
    assert int(inl2.min()) == 1


VOTING_REF_CASES = ((2048, 9, 128, 1), (30000, 9, 128, 2), (777, 3, 64, 3))


def voting_ref_key(tn, vn, hn, vp=None):
    return "voting/%d_%d_%d" % (tn, vn, hn) + ("" if vp is None else "/vp" if vp else "/plain")


def test_voting_vs_reference_cuda_build(dev):
    """Against the REFERENCE's own kernels (ransac_voting_kernel.cu compiled unmodified for sm_100a), whose outputs on
    these inputs are stored in tests/golden/ref_cuda_ops.npz: bit-identical hypotheses, identical inlier masks."""
    from gdrnpp_bop2022_b200.native_ops import ransac_voting as rv

    g = np.load(GOLD_CUDA)
    for tn, vn, hn, seed in VOTING_REF_CASES:
        direct, coords, idxs = _voting_inputs(tn, vn, hn, seed)
        assert_same_inputs(g, voting_ref_key(tn, vn, hn), direct, coords, idxs)
        D, C, I = (torch.from_numpy(a).to(dev) for a in (direct, coords, idxs))
        for vp in (False, True):
            key = voting_ref_key(tn, vn, hn, vp)
            gen_m = rv.generate_hypothesis_vanishing_point if vp else rv.generate_hypothesis
            vote_m = rv.voting_for_hypothesis_vanishing_point if vp else rv.voting_for_hypothesis
            h_m = gen_m(D, C, I)
            i_m = torch.zeros((hn, vn, tn), dtype=torch.uint8, device=dev)
            vote_m(D, C, h_m, i_m, 0.99 if vp else 0.999)
            torch.cuda.synchronize()
            assert np.array_equal(h_m.cpu().numpy().view(np.int32), g[key + "/hyp"].view(np.int32)), (tn, vp)
            inl = i_m.cpu().numpy()
            assert np.array_equal(inl.sum(2, dtype=np.int32), g[key + "/counts"]), (tn, vp)
            assert sha256(inl) == str(g[key + "/inliers_sha256"]), (tn, vp)


def _voting_field(h, w, kp, noise, rs):
    yy, xx = np.meshgrid(np.arange(h), np.arange(w), indexing="ij")
    pix = np.stack([xx, yy], -1).astype(np.float32)
    d = kp[None, None] - pix[:, :, None] + rs.randn(h, w, kp.shape[0], 2).astype(np.float32) * noise
    return (d / (np.linalg.norm(d, axis=-1, keepdims=True) + 1e-9)).astype(np.float32)


def test_ransac_voting_layer_device_side_vs_reference_driver(dev):
    """ransac_voting_layer / _v3 (ONE device call: compaction, hypotheses, fused vote + count, winner, refit) against the
    reference's driver loop (ransac_voting_gpu.py:24-104) restated in the test on top of the op-level entry points --
    the reference's own CUDA extension when oracle/_ref holds it, else ours (bit-identical to it, see
    test_voting_vs_reference_cuda_build) -- fed with the SAME pixel pairs: identical winners, bit-identical inlier
    sets, final keypoints equal to fp32 rounding.  Also: keypoint recovery, empty / tiny masks, batch invariance."""
    from gdrnpp_bop2022_b200.native_ops import ransac_voting as rv_mine
    from gdrnpp_bop2022_b200.native_ops import ransac_voting_layer, ransac_voting_layer_v3

    ops = load_ref_ext("ransac_voting") or rv_mine
    rs = np.random.RandomState(0)
    h = w = 64
    kp = np.array([[20.3, 30.1], [50.2, 10.4], [5.5, 60.0], [40.0, 40.0]], np.float32)
    vn, hn = kp.shape[0], 64
    yy, xx = np.meshgrid(np.arange(h), np.arange(w), indexing="ij")
    masks = np.stack([((yy - 32) ** 2 + (xx - 32) ** 2 < 25 ** 2), ((yy - 20) ** 2 + (xx - 40) ** 2 < 12 ** 2),
                      np.zeros((h, w), bool), (yy == 3) & (xx < 4)]).astype(np.float32)      # disc, small disc, empty, 4 pixels (< min_num)
    vertex = np.stack([_voting_field(h, w, kp, 0.02, rs) for _ in range(4)])
    M, V = torch.from_numpy(masks).to(dev), torch.from_numpy(vertex).to(dev)
    idxs = torch.from_numpy(rs.randint(0, 1 << 30, (4, hn, vn, 2)).astype(np.int32)).to(dev)
    win, inl, tn = ransac_voting_layer(M, V, hn, inlier_thresh=0.999, idxs=idxs, return_inliers=True)
    win3 = ransac_voting_layer_v3(M, V, hn, inlier_thresh=0.999, idxs=idxs)
    torch.cuda.synchronize()
    assert torch.equal(win, win3)
    assert tn.cpu().tolist() == [int(masks[0].sum()), int(masks[1].sum()), 0, 0]
    assert torch.equal(win[2:], torch.zeros(2, vn, 2, device=dev))                          # empty / too-few-pixel images
    assert (win[0].cpu().numpy() - kp).__abs__().max() < 0.5 and np.abs(win[1].cpu().numpy() - kp).max() < 1.5
    # ---- the reference driver on image 0 and 1 with the same pixel pairs ----
    for bi in (0, 1):
        cur_mask = M[bi].to(torch.bool)
        coords = torch.nonzero(cur_mask).float()[:, [1, 0]].contiguous()
        direct = V[bi].masked_select(cur_mask[:, :, None, None]).view([coords.shape[0], vn, 2]).contiguous()
        t = coords.shape[0]
        ix = (idxs[bi].to(torch.int64) % t).to(torch.int32).contiguous()
        hyp = ops.generate_hypothesis(direct, coords, ix)
        cur_inlier = torch.zeros([hn, vn, t], dtype=torch.uint8, device=dev)
        ops.voting_for_hypothesis(direct, coords, hyp, cur_inlier, 0.999)
        counts = torch.sum(cur_inlier, 2)
        win_counts, win_idx = torch.max(counts, 0)
        win_pts = hyp[win_idx, torch.arange(vn, device=dev)]
        # any hypothesis with the maximal count is a legitimate torch.max winner: compare by count, then use ours
        all_inlier = torch.zeros([1, vn, t], dtype=torch.uint8, device=dev)
        ops.voting_for_hypothesis(direct, coords, win_pts[None].contiguous(), all_inlier, 0.999)
        ours_inl = inl[bi, :, :t]
        same_winner = (all_inlier[0] == ours_inl).all(dim=1)
        for v in range(vn):
            if not bool(same_winner[v]):      # a tie in the counts resolved to another hypothesis: it must be as good
                assert int(ours_inl[v].sum()) >= int(all_inlier[0, v].sum()) - 0
        assert int(same_winner.sum()) >= vn - 1
        normal = torch.zeros_like(direct)
        normal[:, :, 0], normal[:, :, 1] = direct[:, :, 1], -direct[:, :, 0]
        nrm = normal.permute(1, 0, 2) * ours_inl.float().unsqueeze(2)
        bvec = torch.sum(nrm * coords.unsqueeze(0), 2)
        ATA = torch.matmul(nrm.permute(0, 2, 1), nrm)
        ATb = torch.sum(nrm * bvec.unsqueeze(2), 1)
        ref_pts = torch.linalg.solve(ATA.double(), ATb.double().unsqueeze(2))[:, :, 0].float()
        assert (win[bi] - ref_pts).abs().max().item() < 2e-3
    # batch invariance: an image gives the same result alone as inside a batch
    alone = ransac_voting_layer(M[1:2], V[1:2], hn, inlier_thresh=0.999, idxs=idxs[1:2])
    assert torch.equal(alone[0], win[1])
    # RNG path: reproducible under torch.manual_seed, recovers the keypoints
    torch.manual_seed(0)
    a = ransac_voting_layer(M[:1], V[:1], 128)
    torch.manual_seed(0)
    b2 = ransac_voting_layer(M[:1], V[:1], 128)
    assert torch.equal(a, b2) and np.abs(a[0].cpu().numpy() - kp).max() < 0.5


def test_estimate_voting_distribution_with_mean(dev):
    """ransac_voting_gpu.py:221-330 on the device-side hypothesis generator: covariance of the inlier-weighted hypothesis
    cloud around the given mean: symmetric, positive semi-definite, and growing with the noise of the vector field."""
    from gdrnpp_bop2022_b200.native_ops import estimate_voting_distribution_with_mean, ransac_voting_layer

    rs = np.random.RandomState(1)
    h = w = 64
    kp = np.array([[20.3, 30.1], [50.2, 10.4], [40.0, 40.0]], np.float32)
    yy, xx = np.meshgrid(np.arange(h), np.arange(w), indexing="ij")
    mask = ((yy - 32) ** 2 + (xx - 32) ** 2 < 25 ** 2).astype(np.float32)[None]
    covs = []
    for noise in (0.005, 0.05):
        V = torch.from_numpy(_voting_field(h, w, kp, noise, rs)[None]).to(dev)
        M = torch.from_numpy(mask).to(dev)
        mean = ransac_voting_layer(M, V, 128, inlier_thresh=0.99, seed=5)
        m2, cov = estimate_voting_distribution_with_mean(M, V, mean, round_hyp_num=256, min_hyp_num=1024, inlier_thresh=0.99, seed=7)
        assert torch.equal(m2, mean) and cov.shape == (1, 3, 2, 2)
        c = cov[0].cpu().double()
        assert (c - c.transpose(1, 2)).abs().max() < 1e-4 * c.abs().max().clamp_min(1e-6)
        assert (torch.linalg.eigvalsh((c + c.transpose(1, 2)) / 2) > -1e-6).all()
        covs.append(c.diagonal(dim1=1, dim2=2).sum(1))
    assert (covs[1] > covs[0]).all()


# ------------------------------------------------------------------------------------------ nnd / flow
@pytest.mark.parametrize("b,n,m", [(1, 1, 1), (2, 3, 2050), (10, 1000, 1500), (3, 2048, 2048)])
def test_nnd_bit_exact(dev, b, n, m):
    from gdrnpp_bop2022_b200.native_ops import nnd, torch_nndistance_aten

    rs = np.random.RandomState(b * 100 + n)
    a, bb = rs.rand(b, n, 3).astype(np.float32), rs.rand(b, m, 3).astype(np.float32)
    if n > 10:
        bb[:, 5] = bb[:, 4]  # exact ties -> lowest index must win
    A, Bt = torch.from_numpy(a).to(dev), torch.from_numpy(bb).to(dev)
    d1 = torch.zeros(b, n, device=dev); d2 = torch.zeros(b, m, device=dev)
    i1 = torch.zeros(b, n, dtype=torch.int32, device=dev); i2 = torch.zeros(b, m, dtype=torch.int32, device=dev)
    assert torch_nndistance_aten.nnd_forward_cuda(A, Bt, d1, d2, i1, i2) == 1
    od1, od2, oi1, oi2 = OO.nnd_forward(a, bb)
    assert np.array_equal(d1.cpu().numpy().view(np.uint32), od1.view(np.uint32))
    assert np.array_equal(d2.cpu().numpy().view(np.uint32), od2.view(np.uint32))
    assert np.array_equal(i1.cpu().numpy(), oi1) and np.array_equal(i2.cpu().numpy(), oi2)
    # backward through the autograd Function vs the oracle (atomics: tolerance)
    A.requires_grad_(True); Bt.requires_grad_(True)
    e1, e2 = nnd(A, Bt)
    g1 = torch.from_numpy(rs.rand(b, n).astype(np.float32)).to(dev); g2 = torch.from_numpy(rs.rand(b, m).astype(np.float32)).to(dev)
    (e1 * g1).sum().backward(retain_graph=True)
    ga_only1 = A.grad.clone()
    A.grad = None; Bt.grad = None
    ((e1 * g1).sum() + (e2 * g2).sum()).backward()
    oga, ogb = OO.nnd_backward(a, bb, g1.cpu().numpy(), g2.cpu().numpy(), oi1, oi2)
    assert np.abs(A.grad.cpu().numpy() - oga).max() < 1e-4 * max(1.0, np.abs(oga).max())
    assert np.abs(Bt.grad.cpu().numpy() - ogb).max() < 1e-4 * max(1.0, np.abs(ogb).max())
    assert ga_only1.shape == A.shape


def nnd_ref_inputs():
    # the reference's test.py shapes and distribution (U[0, 1)^3 clouds), drawn with numpy's stable legacy generator
    rs = np.random.RandomState(0)
    return rs.rand(10, 1000, 3).astype(np.float32), rs.rand(10, 1500, 3).astype(np.float32)


def nnd_forward(mod, a, b):
    d1 = torch.zeros(a.shape[:2], device=a.device); d2 = torch.zeros(b.shape[:2], device=a.device)
    i1 = torch.zeros(a.shape[:2], dtype=torch.int32, device=a.device); i2 = torch.zeros(b.shape[:2], dtype=torch.int32, device=a.device)
    assert mod.nnd_forward_cuda(a, b, d1, d2, i1, i2) == 1
    torch.cuda.synchronize()
    return {"d1": d1, "d2": d2, "i1": i1, "i2": i2}


def test_nnd_vs_reference_cuda_build(dev):
    """Against the REFERENCE's own kernel (nnd_cuda_kernel.cu compiled for sm_100a), whose outputs on these inputs are
    stored in tests/golden/ref_cuda_ops.npz: bit-identical distances and indices."""
    from gdrnpp_bop2022_b200.native_ops import torch_nndistance_aten as mine

    g = np.load(GOLD_CUDA)
    a, b = nnd_ref_inputs()
    assert_same_inputs(g, "nnd", a, b)
    for name, x in nnd_forward(mine, torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev)).items():
        assert_matches_golden(g, "nnd/" + name, x.cpu().numpy())


def _flow_inputs(B, H, W, seed):
    rs = np.random.RandomState(seed)
    K = np.array([[572.4, 0, W / 2 - 3.5], [0, 573.6, H / 2 + 2.1], [0, 0, 1]], np.float32)
    yy, xx = np.meshgrid(np.arange(H, dtype=np.float32), np.arange(W, dtype=np.float32), indexing="ij")
    smooth = (0.7 + 0.02 * np.sin(xx / 40.0) + 0.02 * np.cos(yy / 30.0)).astype(np.float32)
    depth_src = np.tile(smooth[None, None], (B, 1, 1, 1)).copy()
    depth_src[:, :, : max(1, H // 8)] = 0  # invalid depth rows
    T = np.tile(np.eye(4, dtype=np.float32)[:3][None], (B, 1, 1))
    T[:, :, 3] = rs.randn(B, 3) * 0.0007  # sub-pixel .. ~1 px of image motion
    # float64 products of float32 values are exact, and K's zeros fix the sums: KT and Kinv come out bit-identical
    # whichever BLAS / LAPACK kernel the host picks (the stored reference outputs depend on them)
    KT = (K[None].astype(np.float64) @ T.astype(np.float64)).astype(np.float32)
    K64 = K.astype(np.float64)
    Kinv1 = np.array([[1 / K64[0, 0], 0, -K64[0, 2] / K64[0, 0]], [0, 1 / K64[1, 1], -K64[1, 2] / K64[1, 1]], [0, 0, 1]])
    Kinv = np.tile(Kinv1[None], (B, 1, 1)).astype(np.float32)
    depth_tgt = (np.tile(smooth[None, None], (B, 1, 1, 1)) + T[:, 2, 3][:, None, None, None]
                 + (rs.rand(B, 1, H, W) < 0.3) * 0.01).astype(np.float32)  # 30 % of the target pixels are occluders
    return depth_src, depth_tgt, KT, Kinv


FLOW_CASES = [(1, 8, 8), (2, 120, 160), (8, 480, 640)]


def flow_ref_key(B, H, W):
    return "flow/%d_%d_%d" % (B, H, W)


@pytest.mark.parametrize("B,H,W", FLOW_CASES)
def test_flow_bit_exact(dev, B, H, W):
    from gdrnpp_bop2022_b200.native_ops import flow_cuda

    ds, dt, KT, Kinv = _flow_inputs(B, H, W, seed=H)
    fl, va = flow_cuda.forward(*(torch.from_numpy(x).to(dev) for x in (ds, dt, KT, Kinv)))
    ofl, ova = OO.flow(ds, dt, KT, Kinv)
    assert np.array_equal(va.cpu().numpy(), ova)
    assert np.array_equal(fl.cpu().numpy().view(np.uint32), ofl.view(np.uint32))
    assert 0.2 < ova.mean() < 0.9  # the case exercises both branches
    # the REFERENCE's own kernel (flow_cuda_kernel.cu compiled for sm_100a): outputs stored in tests/golden/ref_cuda_ops.npz
    g = np.load(GOLD_CUDA)
    key = flow_ref_key(B, H, W)
    assert_same_inputs(g, key, ds, dt, KT, Kinv)
    assert_matches_golden(g, key + "/flow", fl.cpu().numpy())
    assert_matches_golden(g, key + "/valid", va.cpu().numpy())


# --------------------------------------------------------------------------------- uncertainty PnP
def test_upnp_known_answer_and_vs_oracle(dev):
    from gdrnpp_bop2022_b200 import native_ops

    rs = np.random.RandomState(3)
    K = np.array([[400.0, 0, 128], [0, 400, 128], [0, 0, 1]])
    n_prob, pn = 6, 8
    P2, P3, Wt, init, truth = [], [], [], [], []
    for _ in range(n_prob):
        rt = rs.rand(6)
        p3 = rs.rand(pn, 3)
        p2 = np.zeros((pn, 2))
        for i in range(pn):
            q = OO._rodrigues_point(rt[:3], p3[i]) + rt[3:]
            p2[i] = [K[0, 0] * q[0] / q[2] + K[0, 2], K[1, 1] * q[1] / q[2] + K[1, 2]]
        w = np.stack([1 + rs.rand(pn), 0.1 * rs.randn(pn), 1 + rs.rand(pn)], 1)
        P2.append(p2); P3.append(p3); Wt.append(w); truth.append(rt); init.append(rt + rs.rand(6) * 0.1)
    # reference-signature host entry (blocking) : recovers the ground truth (uncertainty_pnp.cpp:98-156 recipe)
    for i in range(n_prob):
        sol = native_ops.uncertainty_pnp_refine(P2[i], Wt[i], P3[i], K, init[i])
        assert np.abs(sol - truth[i]).max() < 1e-6
        assert np.abs(sol - OO.uncertainty_pnp(P2[i], P3[i], Wt[i], K, init[i])).max() < 1e-5
    # batched device entry
    t = lambda a: torch.from_numpy(np.stack(a)).to(dev)
    res = native_ops.uncertainty_pnp_batched(t(P2), t(P3), t(Wt), torch.from_numpy(np.tile(K[None], (n_prob, 1, 1))).to(dev), t(init))
    assert np.abs(res.cpu().numpy() - np.stack(truth)).max() < 1e-6
    # noisy observations: agrees with the oracle's LM to tolerance
    p2n = P2[0] + rs.randn(pn, 2) * 0.5
    a = native_ops.uncertainty_pnp_refine(p2n, Wt[0], P3[0], K, init[0])
    b = OO.uncertainty_pnp(p2n, P3[0], Wt[0], K, init[0])
    assert np.abs(a - b).max() < 1e-4


# ------------------------------------------------------------------------- rasteriser / depth refine
def _mesh_and_poses(n, seed):
    from gdrnpp_bop2022_b200.synthetic import make_icosphere_mesh

    rs = np.random.RandomState(seed)
    v, f = make_icosphere_mesh(3, (0.12, 0.08, 0.1))
    poses, Ks = [], []
    for i in range(n):
        ax = rs.randn(3); ax /= np.linalg.norm(ax)
        R = O.axangle2mat(ax, rs.rand() * 3)
        t = np.array([rs.randn() * 0.02, rs.randn() * 0.02, 0.5 + rs.rand() * 0.3])
        poses.append(np.hstack([R, t[:, None]]))
        Ks.append(np.array([[110.0 + 10 * rs.rand(), 0, 32 + rs.randn()], [0, 112.0, 31 + rs.randn()], [0, 0, 1]]))
    return v, f, np.stack(poses).astype(np.float32), np.stack(Ks).astype(np.float32)


def test_rasteriser_vs_numpy_oracle(dev):
    from gdrnpp_bop2022_b200.renderer import render_depth

    v, f, poses, Ks = _mesh_and_poses(4, seed=1)
    d = render_depth(torch.from_numpy(v).to(dev), torch.from_numpy(f).to(dev), torch.from_numpy(poses).to(dev),
                     torch.from_numpy(Ks).to(dev), 64, 64).cpu().numpy()
    for i in range(4):
        ref = OO.render_depth(v, f, poses[i], Ks[i], 64, 64)
        both = (d[i] > 0) & (ref > 0)
        # coverage may differ only on silhouette pixels whose centre lies (to fp32 rounding) on an edge
        assert ((d[i] > 0) != (ref > 0)).sum() <= 6, i
        assert both.sum() > 150
        assert np.abs(d[i][both] - ref[both]).max() < 1e-3  # the tolerance fast depth refine needs (metres)
        assert np.median(np.abs(d[i][both] - ref[both])) < 2e-6


def test_depth_refine_vs_oracle(dev):
    from gdrnpp_bop2022_b200.renderer import depth_refine, render_depth

    n = 5
    v, f, poses, Ks = _mesh_and_poses(n, seed=2)
    rs = np.random.RandomState(9)
    V, F = torch.from_numpy(v).to(dev), torch.from_numpy(f).to(dev)
    true_poses = poses.copy()
    true_poses[:, :, 3] *= (1 + rs.uniform(-0.04, 0.04, (n, 1)))   # sensor sees the object a bit nearer / farther
    sensor = render_depth(V, F, torch.from_numpy(true_poses).to(dev), torch.from_numpy(Ks).to(dev), 64, 64)
    sensor[4] = 0  # one ROI without valid depth -> pose must stay unchanged
    xyz = torch.rand(n, 3, 64, 64, generator=torch.Generator().manual_seed(0)).to(dev) - 0.5
    mask = torch.rand(n, 1, 64, 64, generator=torch.Generator().manual_seed(1)).to(dev)
    rot = torch.from_numpy(poses[:, :, :3]).to(dev).contiguous()
    trans = torch.from_numpy(poses[:, :, 3]).to(dev).contiguous()
    new_t = depth_refine(V, F, rot, trans, torch.from_numpy(Ks).to(dev), xyz, mask, sensor, iters=2, thresh=0.8)
    torch.cuda.synchronize()
    # oracle: same loop with the numpy renderer + the reference's refine arithmetic
    mx = mask.view(n, -1).max(1)[0].view(n, 1, 1, 1); mn = mask.view(n, -1).min(1)[0].view(n, 1, 1, 1)
    mnorm = ((mask - mn) / (mx - mn)).cpu().numpy()
    for i in range(n):
        t = poses[i, :, 3].astype(np.float64).copy()
        for _ in range(2):
            pose = np.hstack([poses[i, :, :3], t[:, None]]).astype(np.float32)
            ren = OO.render_depth(v, f, pose, Ks[i], 64, 64)
            t = OO.depth_refine_step(xyz[i].permute(1, 2, 0).cpu().numpy(), mnorm[i, 0], sensor[i].cpu().numpy(), ren, Ks[i], t)
        assert np.abs(new_t[i].cpu().numpy() - t).max() < 1e-3, i       # north_star: t within 1e-3
    assert torch.equal(new_t[4].cpu(), torch.from_numpy(poses[4, :, 3]))
    # and the refinement actually moves towards the truth
    err0 = np.abs(poses[:4, 2, 3] - true_poses[:4, 2, 3]); err1 = np.abs(new_t[:4, 2].cpu().numpy() - true_poses[:4, 2, 3])
    assert (err1 < err0).all()


# ----------------------------------------------------------------------------------------------- ROI crop + resize
def _crop_Ms(rng, n, out, W=640, H=480):
    Ms = []
    for i in range(n):
        cx, cy, scale = rng.uniform(-40, W + 40), rng.uniform(-40, H + 40), float(rng.uniform(24, 720))
        s = out / scale
        M = np.array([[s, 0, out * 0.5 - cx * s], [0, s, out * 0.5 - cy * s]], np.float64)
        if i % 4 == 3:
            a = rng.uniform(-0.6, 0.6)
            M[:, :2] = np.array([[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]]) * s
        Ms.append(M)
    return np.stack(Ms)


def test_crop_resize_bit_exact(dev):
    """ROI crops on the GPU == the oracle restatement of cv2.warpAffine (pinned bit-exactly against cv2 on the CPU):
    uint8 bilinear + normalize_image, float bilinear (coordinate grid), float nearest (depth)."""
    from gdrnpp_bop2022_b200 import native_ops as NO

    rng = np.random.RandomState(5)
    img = rng.randint(0, 256, (480, 640, 3)).astype(np.uint8)
    coord = rng.rand(480, 640, 2).astype(np.float32)
    depth = (rng.rand(480, 640) * 2).astype(np.float32)
    M256, M64 = _crop_Ms(rng, 9, 256), _crop_Ms(rng, 9, 64)
    got = NO.crop_resize_image(torch.from_numpy(img).to(dev), M256, 256).cpu().numpy()
    for i in range(9):
        assert np.array_equal(got[i], OO.crop_resize_roi(img, M256[i], 256)), i
    got = NO.crop_resize_float(torch.from_numpy(coord).to(dev), M64, 64).cpu().numpy()
    for i in range(9):
        assert np.array_equal(got[i], OO.warp_affine_f32(coord, M64[i], (64, 64)).transpose(2, 0, 1)), i
    got = NO.crop_resize_float(torch.from_numpy(depth).to(dev), M256, 256, nearest=True).cpu().numpy()
    for i in range(9):
        assert np.array_equal(got[i, 0], OO.warp_affine_f32(depth, M256[i], (256, 256), nearest=True)[:, :, 0]), i
    # empty batch and the committed cv2 golden crop
    assert NO.crop_resize_image(torch.from_numpy(img).to(dev), np.zeros((0, 2, 3)), 256).shape == (0, 3, 256, 256)
    g = np.load(os.path.join(ROOT, "tests", "golden", "crop_golden.npz"))
    gi = torch.from_numpy(g["img"]).to(dev)
    for i in range(g["M"].shape[0]):
        out = int(g["out"][i])
        crop = NO.crop_resize_image(gi, g["M"][i][None], out, pixel_std=(1.0, 1.0, 1.0))[0].cpu().numpy()
        assert np.array_equal(crop.transpose(1, 2, 0).astype(np.uint8), g["crop_%d" % i]), i


def test_predictor_preprocessing_matches_reference_recipe(dev):
    """GdrnPredictor.preprocessing (GPU crops) vs the per-ROI host recipe of predictor_gdrn.py:396-438 restated with the
    oracle warp: roi_img, roi_coord_2d, roi_depth, scale / resize_ratio / roi_wh bookkeeping."""
    from gdrnpp_bop2022_b200.native_ops import get_affine_transform
    from gdrnpp_bop2022_b200.predictor import GdrnPredictor
    from gdrnpp_bop2022_b200.synthetic import make_state_dict

    rng = np.random.RandomState(11)
    H, W = 480, 640
    image = rng.randint(0, 256, (H, W, 3)).astype(np.uint8)
    depth = (rng.rand(H, W) * 1.5).astype(np.float32)
    K = np.array([[1066.778, 0, 312.9869], [0, 1067.487, 241.3109], [0, 0, 1]], np.float32)
    objs = {i + 1: "obj_%d" % (i + 1) for i in range(21)}
    extents = {i + 1: np.array([0.1, 0.12, 0.08], np.float32) for i in range(21)}
    pred = GdrnPredictor(cam=K, objs=objs, extents=extents, state_dict=make_state_dict(), device=dev, use_pnp=False)
    dets = np.array([[100, 80, 220, 260, 0.9, 0.8, 3], [400, 200, 460, 250, 0.7, 0.9, 10], [-20, 300, 90, 470, 0.5, 0.5, 0]],
                    np.float32)
    data = pred.preprocessing(dets, image, depth)
    xx, yy = np.meshgrid(np.linspace(0, 1, W, endpoint=False, dtype=np.float32), np.linspace(0, 1, H, endpoint=False, dtype=np.float32))
    coord_2d = np.stack([xx, yy], axis=2)
    for i, d in enumerate(dets):
        x1, y1, x2, y2 = d[:4]
        c = np.array([0.5 * (x1 + x2), 0.5 * (y1 + y2)])
        bw, bh = max(x2 - x1, 1), max(y2 - y1, 1)
        scale = min(max(bh, bw) * 1.5, max(H, W)) * 1.0
        M256, M64 = get_affine_transform(c, scale, 0, 256), get_affine_transform(c, scale, 0, 64)
        assert np.array_equal(data["roi_img"][i].cpu().numpy(), OO.crop_resize_roi(image, M256, 256))
        assert np.array_equal(data["roi_coord_2d"][i].cpu().numpy(), OO.warp_affine_f32(coord_2d, M64, (64, 64)).transpose(2, 0, 1))
        assert np.array_equal(data["roi_depth"][i, 0].cpu().numpy(), OO.warp_affine_f32(depth, M256, (256, 256), nearest=True)[:, :, 0])
        assert abs(float(data["scale"][i]) - scale) < 1e-4 and abs(float(data["resize_ratio"][i]) - 64 / scale) < 1e-7
        assert np.allclose(data["roi_wh"][i].cpu().numpy(), [bw, bh])
    out = pred.inference(data)
    assert out["rot"].shape == (3, 3, 3) and torch.isfinite(out["trans"]).all()


# ------------------------------------------------------------------------- RANSAC-PnP post-process (SURVEY 8f-2)
def _rand_pose(rs):
    ax = rs.randn(3)
    ax /= np.linalg.norm(ax)
    R = O.axangle2mat(ax, rs.rand() * 3)
    t = np.array([rs.randn() * 0.05, rs.randn() * 0.05, 0.7 + rs.rand() * 0.5])
    return R, t


def _rot_angle(Ra, Rb):
    return float(np.arccos(np.clip((np.trace(Ra.T @ Rb) - 1) / 2, -1, 1)))


def test_pnp_ransac_points_vs_cv2(dev):
    """Batched GPU RANSAC-PnP on explicit correspondences vs cv2.solvePnPRansac (the call misc.pnp_v2 makes,
    lib/pysixd/misc.py:187-196: EPnP, reprojectionError 3, 100 iterations) on synthetic 2D-3D pairs with pixel noise and
    30 % gross outliers: both recover the ground truth, agree with each other to the noise level, and flag the same
    correspondences as inliers; noise-free data is recovered exactly; < 4 points -> the reference's -100 sentinel."""
    import cv2

    from gdrnpp_bop2022_b200.pnp_ransac import solve_pnp_ransac

    rs = np.random.RandomState(7)
    K = np.array([[1066.778, 0, 312.9869], [0, 1067.487, 241.3109], [0, 0, 1]])
    n, npts = 6, 600
    P3, P2, GT, OUT = [], [], [], []
    for i in range(n):
        R, t = _rand_pose(rs)
        X = (rs.rand(npts, 3) - 0.5) * np.array([0.12, 0.2, 0.09])
        xc = X @ R.T + t
        uv = np.stack([K[0, 0] * xc[:, 0] / xc[:, 2] + K[0, 2], K[1, 1] * xc[:, 1] / xc[:, 2] + K[1, 2]], 1)
        outl = np.zeros(npts, bool)
        if i > 0:                      # problem 0 is noise-free
            uv += rs.randn(npts, 2) * 0.5
            outl = rs.rand(npts) < 0.3
            uv[outl] += rs.randn(int(outl.sum()), 2) * 40 + 25
        P3.append(X); P2.append(uv); GT.append((R, t)); OUT.append(outl)
    t_ = lambda a: torch.from_numpy(np.stack(a).astype(np.float32)).to(dev)
    poses, ninl, imask = solve_pnp_ransac(t_(P3), t_(P2), torch.from_numpy(K.astype(np.float32))[None].to(dev), reproj_err=3.0,
                                          iters=100, seed=3, return_inliers=True)
    poses, ninl, imask = poses.cpu().numpy().astype(np.float64), ninl.cpu().numpy(), imask.cpu().numpy().astype(bool)
    for i in range(n):
        R, t = GT[i]
        ok, rvec, tvec, inl = cv2.solvePnPRansac(P3[i][None].astype(np.float64), P2[i][None].astype(np.float64), K, np.zeros((8, 1)),
                                                 flags=cv2.SOLVEPNP_EPNP, reprojectionError=3.0, iterationsCount=100)
        assert ok
        Rc = cv2.Rodrigues(rvec)[0]
        Rm, tm = poses[i, :, :3], poses[i, :, 3]
        assert abs(np.linalg.det(Rm) - 1) < 1e-5 and np.abs(Rm @ Rm.T - np.eye(3)).max() < 1e-5
        tol_r, tol_t = (1e-4, 1e-5) if i == 0 else (4e-3, 2e-3)
        assert _rot_angle(Rm, R) < tol_r and np.abs(tm - t).max() < tol_t, (i, _rot_angle(Rm, R), np.abs(tm - t).max())
        assert _rot_angle(Rm, Rc) < 2 * tol_r + 1e-3 and np.abs(tm - tvec[:, 0]).max() < 2 * tol_t + 1e-3
        cv_in = np.zeros(npts, bool)
        cv_in[inl[:, 0]] = True
        assert (imask[i] != cv_in).mean() < 0.03            # same inlier set up to points at the 3 px boundary
        assert (imask[i] & OUT[i]).sum() <= 2 and ninl[i] == imask[i].sum()
    few = solve_pnp_ransac(t_([P3[0][:3]]), t_([P2[0][:3]]), torch.from_numpy(K.astype(np.float32))[None].to(dev)).cpu().numpy()
    assert (few == -100).all()
    # caller-supplied samples: deterministic and independent of the seed
    idxs = torch.from_numpy(rs.randint(0, npts, (n, 64, 4)).astype(np.int32))
    a = solve_pnp_ransac(t_(P3), t_(P2), torch.from_numpy(K.astype(np.float32))[None].to(dev), idxs=idxs, seed=1)
    b = solve_pnp_ransac(t_(P3), t_(P2), torch.from_numpy(K.astype(np.float32))[None].to(dev), idxs=idxs, seed=2)
    assert torch.equal(a, b)


def test_pnp_ransac_from_maps_vs_reference_recipe(dev):
    """The map entry (get_pnp_ransac_pose, gdrn_evaluator.py:1122-1221) vs the reference recipe restated on the host with
    numpy + cv2.solvePnPRansac: L1 mask min-max normalisation, xyz denormalisation by the extent, selection mask > 0.5 &
    |xyz| > 1e-4 extent, image points = roi_coord_2d * (im_W, im_H).  Maps are synthesised from a known pose (object
    points on a sphere seen through the ROI grid) with noise; one ROI has an empty mask."""
    import cv2

    from gdrnpp_bop2022_b200.pnp_ransac import pnp_ransac_from_maps

    rs = np.random.RandomState(11)
    K = np.array([[1066.778, 0, 312.9869], [0, 1067.487, 241.3109], [0, 0, 1]])
    n, hw, imH, imW = 5, 64, 480, 640
    cx_, cy_, cz_, mk, c2d, ext, GT = [], [], [], [], [], [], []
    for i in range(n):
        R, t = _rand_pose(rs)
        r_obj = 0.05
        e = np.array([0.12, 0.13, 0.11])
        # ROI grid around the projected centre
        pc = K @ t
        pc = pc[:2] / pc[2]
        scale = 2.6 * r_obj * K[0, 0] / t[2]
        u = pc[0] + (np.arange(hw) - hw / 2) * scale / hw
        v = pc[1] + (np.arange(hw) - hw / 2) * scale / hw
        U, V = np.meshgrid(u, v)
        rays = np.stack([(U - K[0, 2]) / K[0, 0], (V - K[1, 2]) / K[1, 1], np.ones_like(U)], -1)
        rays /= np.linalg.norm(rays, axis=-1, keepdims=True)
        b_ = (rays * t).sum(-1)
        disc = b_ ** 2 - (t @ t - r_obj ** 2)
        hit = disc > 0
        depth = b_ - np.sqrt(np.where(hit, disc, 0))
        Xc = rays * depth[..., None]
        Xo = (Xc - t) @ R                     # R^T (Xc - t)
        coor = Xo / e + 0.5 + rs.randn(hw, hw, 3) * 0.002
        coor[~hit] = 0.5                      # background: exactly the centre -> rejected by the |xyz| > 1e-4 extent rule
        m = np.where(hit, 0.9, 0.05) + rs.randn(hw, hw) * 0.02
        if i == 3:
            m[:] = 0.1; m[0, 0] = 0.2; coor[:] = 0.5      # nothing selectable
        cx_.append(coor[..., 0]); cy_.append(coor[..., 1]); cz_.append(coor[..., 2]); mk.append(m)
        c2d.append(np.stack([U / imW, V / imH])); ext.append(e); GT.append((R, t))
    f = lambda a: torch.from_numpy(np.stack(a).astype(np.float32)).to(dev)
    CX, CY, CZ, M = f(cx_)[:, None], f(cy_)[:, None], f(cz_)[:, None], f(mk)[:, None]
    poses, ninl, imask = pnp_ransac_from_maps(CX, CY, CZ, M, f(c2d), torch.full((n,), imH), torch.full((n,), imW), f(ext),
                                              torch.from_numpy(K.astype(np.float32))[None].repeat(n, 1, 1).to(dev), return_inliers=True)
    poses = poses.cpu().numpy().astype(np.float64)
    for i in range(n):
        # host restatement of the reference recipe on the same float32 maps
        m32 = np.stack(mk).astype(np.float32)[i]
        mn = (m32 - m32.min()) / (m32.max() - m32.min())
        e32 = ext[i].astype(np.float32)
        xyz = np.stack([(np.float32(cx_[i]) - np.float32(0.5)) * e32[0], (np.float32(cy_[i]) - np.float32(0.5)) * e32[1],
                        (np.float32(cz_[i]) - np.float32(0.5)) * e32[2]], -1).astype(np.float32)
        sel = (mn > 0.5) & (np.abs(xyz[..., 0]) > 1e-4 * e32[0]) & (np.abs(xyz[..., 1]) > 1e-4 * e32[1]) & (np.abs(xyz[..., 2]) > 1e-4 * e32[2])
        img = np.stack([np.float32(c2d[i][0]) * imW, np.float32(c2d[i][1]) * imH], -1)
        if sel.sum() < 4:
            assert (poses[i] == -100).all() and int(ninl[i]) == 0
            continue
        assert int(imask[i].sum()) <= int(sel.sum()) and not bool((imask[i].cpu().numpy().astype(bool) & ~sel).any())
        ok, rvec, tvec, _ = cv2.solvePnPRansac(xyz[sel][None].astype(np.float64), img[sel][None].astype(np.float64), K, np.zeros((8, 1)),
                                               flags=cv2.SOLVEPNP_EPNP, reprojectionError=3.0, iterationsCount=100)
        Rc = cv2.Rodrigues(rvec)[0]
        R, t = GT[i]
        assert _rot_angle(poses[i, :, :3], R) < 0.02 and np.abs(poses[i, :, 3] - t).max() < 5e-3
        assert _rot_angle(poses[i, :, :3], Rc) < 0.02 and np.abs(poses[i, :, 3] - tvec[:, 0]).max() < 5e-3


def test_predictor_reference_constructor_and_use_pnp(dev, tmp_path):
    """GdrnPredictor(config_file_path, ckpt_file_path, camera_json_path, path_to_obj_models) -- the reference's
    constructor (predictor_gdrn.py:45-120): python config with _base_, checkpoint {"model": ...} with "_module."
    prefixes, BOP camera.json, a directory of obj_{id:06d}.ply in millimetres; TEST.USE_PNP defaults to True like the
    reference predictor and postprocessing returns {name: 4x4}."""
    import json

    from gdrnpp_bop2022_b200.ply import save_ply
    from gdrnpp_bop2022_b200.predictor import GdrnPredictor
    from gdrnpp_bop2022_b200.synthetic import make_icosphere_mesh, make_state_dict

    nc = 3
    (tmp_path / "cfg.py").write_text(
        "MODEL = dict(PIXEL_MEAN=[0.0, 0.0, 0.0], PIXEL_STD=[255.0, 255.0, 255.0], POSE_NET=dict(NAME='GDRN_double_mask', NUM_CLASSES=%d,\n"
        "    OUTPUT_RES=64, BACKBONE=dict(INIT_CFG=dict(type='timm/convnext_base')),\n"
        "    GEO_HEAD=dict(NUM_REGIONS=64, XYZ_CLASS_AWARE=True, MASK_CLASS_AWARE=True, REGION_CLASS_AWARE=True, MASK_THR_TEST=0.5),\n"
        "    PNP_NET=dict(ROT_TYPE='allo_rot6d', TRANS_TYPE='centroid_z', Z_TYPE='REL')))\n"
        "TEST = dict(USE_PNP=False, USE_DEPTH_REFINE=False, DEPTH_REFINE_ITER=2, DEPTH_REFINE_THRESHOLD=0.8)\n"
        "INPUT = dict(DZI_PAD_SCALE=1.5, WITH_DEPTH=False)\n" % nc)
    sd = make_state_dict(num_classes=nc)
    torch.save({"model": {"_module." + k: v for k, v in sd.items()}}, str(tmp_path / "model_final.pth"))
    (tmp_path / "camera.json").write_text(json.dumps({"fx": 1066.778, "fy": 1067.487, "cx": 312.9869, "cy": 241.3109, "depth_scale": 0.1}))
    mdir = tmp_path / "models"
    mdir.mkdir()
    for i, e in zip((1, 2, 5), ((120.0, 80.0, 100.0), (60.0, 60.0, 150.0), (90.0, 140.0, 70.0))):
        v, f_ = make_icosphere_mesh(2, e)
        save_ply(str(mdir / ("obj_%06d.ply" % i)), v, f_, binary=(i != 2))
    pred = GdrnPredictor(str(tmp_path / "cfg.py"), str(tmp_path / "model_final.pth"), str(tmp_path / "camera.json"), str(mdir), device=dev)
    assert pred.obj_ids == [1, 2, 5] and pred.cfg.TEST.USE_PNP is True and abs(pred.depth_scale - 0.1) < 1e-12
    assert np.allclose(pred.extents[2], [0.06, 0.06, 0.15], atol=2e-3) and pred.ren_models is not None
    assert abs(float(pred.cam[0, 0]) - 1066.778) < 1e-3
    rng = np.random.RandomState(2)
    image = rng.randint(0, 256, (480, 640, 3)).astype(np.uint8)
    dets = np.array([[100, 80, 220, 260, 0.9, 0.8, 0], [400, 200, 460, 250, 0.7, 0.9, 2]], np.float32)
    data = pred.preprocessing(dets, image)
    out = pred.inference(data)
    poses = pred.postprocessing(data, out)
    assert set(poses.keys()) == {"obj_000001", "obj_000005"} and all(p.shape == (4, 4) for p in poses.values())
    for r in data["cur_res"]:     # random-init maps carry no geometry: either a RANSAC pose or the -100 sentinel, never NaN
        assert np.isfinite(r["R"]).all() and np.isfinite(r["t"]).all()
    assert pred.postprocessing(pred.preprocessing(np.zeros((0, 7), np.float32), image), pred.inference(pred.preprocessing(np.zeros((0, 7), np.float32), image))) == {}


# ------------------------------------------------------------- renderer class surfaces / z-buffer decode (a11, a12)
def _plane_quad(K, n_pl, d_pl, half=0.6):
    corners = []
    for sx, sy in ((-1, -1), (1, -1), (1, 1), (-1, 1)):
        ray = np.array([sx * half, sy * half, 1.0])
        corners.append(ray * (d_pl / (n_pl @ ray)))
    return np.array(corners, np.float32), np.array([[0, 1, 2], [0, 2, 3]], np.int32)


def test_renderer_surfaces_plane_analytic_and_quantised_decode(dev, tmp_path):
    """lib/render_vispy Renderer (set_cam / draw_model / finish) and lib/egl_renderer EGLRenderer.render(pc_cam_tensor=)
    surfaces on an analytic case: a tilted plane covering the window renders to the ray/plane intersection depth at the
    pixel centres (float path, EGL) and to the 24- / 16-bit fixed-point z-buffer decode of renderer.py:176-182 (vispy);
    model paths are PLY files like the reference; two draws share one z-buffer (nearest wins)."""
    from gdrnpp_bop2022_b200.ply import save_ply
    from gdrnpp_bop2022_b200.renderer import EGLRenderer, Renderer, render_depth

    K = np.array([[110.0, 0, 31.5], [0, 112.0, 30.25], [0, 0, 1]], np.float32)
    n_pl, d_pl = np.array([0.2, -0.1, 1.0]), 0.8
    v, f = _plane_quad(K, n_pl, d_pl)
    cc, rr = np.meshgrid(np.arange(64) + 0.5, np.arange(64) + 0.5)
    rays = np.stack([(cc - K[0, 2]) / K[0, 0], (rr - K[1, 2]) / K[1, 1], np.ones_like(cc)], -1)
    z_true = d_pl / (rays @ n_pl)
    pose = np.hstack([np.eye(3), np.zeros((3, 1))]).astype(np.float32)
    V, F = torch.from_numpy(v).to(dev), torch.from_numpy(f).to(dev)
    P, Kt = torch.from_numpy(pose)[None].to(dev), torch.from_numpy(K)[None].to(dev)
    d0 = render_depth(V, F, P, Kt, 64, 64).cpu().numpy()[0]
    assert (d0 > 0).all() and np.abs(d0 - z_true).max() < 1e-5
    nc, fc = 0.1, 100.0
    mult, addi = np.float32((nc * fc) / (nc - fc)), np.float32(fc / (nc - fc))
    for bits in (24, 16):
        dq = render_depth(V, F, P, Kt, 64, 64, nc, fc, quantize_bits=bits).cpu().numpy()[0]
        win = (1.0 / d0.astype(np.float64) - 1.0 / nc) / (1.0 / fc - 1.0 / nc)     # window depth of the float z
        q = float((1 << bits) - 1)
        expect = mult / (np.float32(np.floor(win * q + 0.5) / q) + addi)            # fixed point -> GL_FLOAT read-back -> decode
        assert np.abs(dq - expect).max() < 1e-6 * max(1.0, float(expect.max()))
        assert np.abs(dq - z_true).max() < (2e-6 if bits == 24 else 4e-4)           # SURVEY App. B: 6e-7 m @ 1 m / 1.5e-4 m
    # vispy-style class with PLY model paths (millimetres -> metres)
    save_ply(str(tmp_path / "obj_000001.ply"), v * 1000.0, f, binary=True)
    v2, f2 = _plane_quad(K, np.array([0.0, 0.0, 1.0]), 0.75, half=0.1)              # a small nearer patch in the middle
    save_ply(str(tmp_path / "obj_000002.ply"), v2 * 1000.0, f2, binary=False)
    ren = Renderer((64, 64), K, model_paths=[str(tmp_path / "obj_000001.ply"), str(tmp_path / "obj_000002.ply")], scale_to_meter=0.001,
                   device=dev)
    ren.clear()
    ren.set_cam(K)
    ren.draw_model(ren.models[0], np.vstack([pose, [0, 0, 0, 1]]))
    ren.draw_model(ren.models[1], np.vstack([pose, [0, 0, 0, 1]]))
    rgb, dep = ren.finish()
    assert rgb.shape == (64, 64, 3) and dep.shape == (64, 64)
    near = np.abs(rays[..., 0]) < 0.09
    near &= np.abs(rays[..., 1]) < 0.09
    assert np.abs(dep[near] - 0.75).max() < 1e-5 and np.abs(dep[~near & (np.abs(rays[..., 0]) > 0.11)] - z_true[~near & (np.abs(rays[..., 0]) > 0.11)]).max() < 1e-5
    # EGL-style class: camera-space xyz written in place, depth = pc_cam[..., 2]
    egl = EGLRenderer([str(tmp_path / "obj_000001.ply")], K=K, width=64, height=64, vertex_scale=0.001, znear=0.25, zfar=6.0, device=dev)
    pc = torch.zeros((64, 64, 4), device=dev)
    seg = torch.zeros((64, 64, 4), device=dev)
    depth = egl.render([0], [pose], pc_cam_tensor=pc, seg_tensor=seg)
    assert torch.equal(depth, pc[..., 2]) and float(pc[..., 3].min()) == 1.0 and float(seg[..., 0].max()) == 1.0
    xyz = pc[..., :3].cpu().numpy()
    assert np.abs(xyz[..., 2] - z_true).max() < 1e-5
    assert np.abs(xyz[..., 0] - rays[..., 0] * z_true).max() < 1e-5 and np.abs(xyz[..., 1] - rays[..., 1] * z_true).max() < 1e-5


def test_multi_mesh_refine_matches_per_mesh_path(dev):
    """depth_refine with several meshes: every ROI picks its mesh from the library's registry inside ONE render launch
    (rast_upload_mesh / rast_render_meshes); result == rendering each mesh's ROIs separately; get_out_mask folded into
    the refine kernel == the torch min-max normalisation + the pre-normalised entry."""
    from gdrnpp_bop2022_b200 import _lib as L
    from gdrnpp_bop2022_b200.renderer import depth_refine, get_out_mask, render_depth, render_meshes, upload_mesh
    from gdrnpp_bop2022_b200.synthetic import make_icosphere_mesh

    n = 6
    _, _, poses, Ks = _mesh_and_poses(n, seed=4)
    meshes = [make_icosphere_mesh(2, e) for e in ((0.12, 0.08, 0.1), (0.06, 0.1, 0.07), (0.09, 0.09, 0.09))]
    Vs = [torch.from_numpy(v).to(dev) for v, _ in meshes]
    Fs = [torch.from_numpy(f).to(dev) for _, f in meshes]
    ids = torch.tensor([0, 2, 1, 1, 0, 2])
    P, Kt = torch.from_numpy(poses).to(dev), torch.from_numpy(Ks).to(dev)
    reg = torch.tensor([upload_mesh(v, f) for v, f in zip(Vs, Fs)], dtype=torch.int32, device=dev)
    multi = render_meshes(reg[ids.to(dev)], P, Kt, 64, 64)
    for i in range(n):
        single = render_depth(Vs[ids[i]], Fs[ids[i]], P[i:i + 1], Kt[i:i + 1], 64, 64)[0]
        assert torch.equal(multi[i], single), i
    g = torch.Generator().manual_seed(0)
    xyz = (torch.rand(n, 3, 64, 64, generator=g) - 0.5).to(dev)
    mask = torch.rand(n, 1, 64, 64, generator=g).to(dev)
    sensor = multi * 1.03
    rot, trans = P[:, :, :3].contiguous(), P[:, :, 3].contiguous()
    t_new = depth_refine(Vs, Fs, rot, trans, Kt, xyz, mask, sensor, iters=2, thresh=0.8, mesh_ids=ids)
    # reference path: per-mesh renders + torch get_out_mask + the pre-normalised kernel entry
    t_ref = trans.clone()
    mnorm = get_out_mask(mask).reshape(n, 64, 64).contiguous()
    lib = L.lib()
    for _ in range(2):
        pp = torch.cat([rot, t_ref[:, :, None]], dim=2).contiguous()
        ren = torch.stack([render_depth(Vs[ids[i]], Fs[ids[i]], pp[i:i + 1], Kt[i:i + 1], 64, 64)[0] for i in range(n)]).contiguous()
        L.check(lib.gdrn_depth_refine_step(L.ptr(xyz), L.ptr(mnorm), L.ptr(sensor.contiguous()), L.ptr(ren), L.ptr(Kt), L.ptr(t_ref), n, 64,
                                           0.8, L.current_stream()), "refine")
    torch.cuda.synchronize()
    assert (t_new - t_ref).abs().max().item() < 1e-6
    assert (t_new - trans).abs().max().item() > 1e-3     # it did move


# ------------------------------------------------------------------------------- depthwise 7x7 + LayerNorm kernels
@pytest.mark.parametrize("B,H,C,split", [(2, 64, 128, 0), (3, 32, 256, 1), (8, 16, 512, 1), (64, 16, 512, 0), (5, 64, 128, 1)])
def test_dwconv_ln_pingpong_vs_cluster_kernel_and_torch(dev, lib, B, H, C, split):
    """ConvNeXt block front half (dw 7x7 pad 3 + bias -> LayerNorm(C, 1e-6)): the persistent two-warpgroup ping-pong
    kernel is BIT-identical to the one-tile-per-CTA cluster kernel (same FMA order, same LayerNorm combine) and both
    agree with the torch fp32 reference of the same op; odd tile counts (one warpgroup gets one tile more) included."""
    L = _lib()
    g = torch.Generator().manual_seed(B * 1000 + H + C)
    x = torch.randn(B, H, H, C, generator=g).to(dev)
    w = (torch.randn(C, 1, 7, 7, generator=g) / 7).to(dev)
    bias, lw, lb = (torch.randn(C, generator=g) * 0.1).to(dev), (torch.rand(C, generator=g) + 0.5).to(dev), (torch.randn(C, generator=g) * 0.1).to(dev)
    w49c = w.reshape(C, 49).t().contiguous()
    outs = []
    for variant in (0, 1):
        o = torch.full((B * H * H, (2 if split else 1) * C), float("nan"), dtype=torch.bfloat16, device=dev)
        L.check(lib.gdrn_dwconv_ln(L.ptr(x), L.ptr(w49c), L.ptr(bias), L.ptr(lw), L.ptr(lb), L.ptr(o), B, H, H, C, 1e-6, split, variant,
                                   L.current_stream()), "dwconv_ln")
        outs.append(o)
    torch.cuda.synchronize()
    assert torch.equal(outs[0].view(torch.int16), outs[1].view(torch.int16))
    y = torch.nn.functional.conv2d(x.permute(0, 3, 1, 2), w, bias, padding=3, groups=C).permute(0, 2, 3, 1)
    ref = torch.nn.functional.layer_norm(y, (C,), lw, lb, 1e-6).reshape(B * H * H, C)
    got = outs[1][:, :C].float() + (outs[1][:, C:].float() if split else 0)
    assert (got - ref).abs().max().item() < (2e-4 if split else 0.03)


def test_upnp_vs_vendored_ceres_and_epnp_wrapper(dev):
    """csrc/upnp.cu (batched device LM) and the reference-signature host entry against the REFERENCE's vendored Ceres 2.0
    (ceres::Jet autodiff + ceres::TinySolver on the residual of uncertainty_pnp.cpp:16-34, solutions stored in
    tests/golden/ref_cpu_ops.npz) on noise-free and noisy problems; and native_ops.uncertainty_pnp -- the
    un_pnp_utils.py:11-78 wrapper (EPnP init on the 4 highest-weight points via cv2, then the weighted refine) -- recovers
    a known pose."""
    from test_oracle_pinning import upnp_ref_problems

    from gdrnpp_bop2022_b200 import native_ops

    probs = upnp_ref_problems("upnp_gpu")
    K = probs[0]["K"]
    t = lambda k: torch.from_numpy(np.stack([p[k] for p in probs])).to(dev)
    res = native_ops.uncertainty_pnp_batched(t("p2"), t("p3"), t("w"), torch.from_numpy(np.tile(K[None], (len(probs), 1, 1))).to(dev),
                                             t("init")).cpu().numpy()
    for i, p in enumerate(probs):
        assert np.abs(res[i] - p["ref"]).max() < 1e-6, (i, res[i], p["ref"])
        host = native_ops.uncertainty_pnp_refine(p["p2"], p["w"], p["p3"], K, p["init"])
        assert np.abs(host - p["ref"]).max() < 1e-6
        if i % 2 == 0:
            assert np.abs(res[i] - p["rt"]).max() < 1e-8
    # the EPnP-initialised wrapper (un_pnp_utils.uncertainty_pnp): [3,4] pose, pn == 4 short-cut included
    import cv2

    rt, p2, p3, w = (probs[0][f] for f in ("rt", "p2", "p3", "w"))
    pose = native_ops.uncertainty_pnp(p2, w, p3, K)
    Rgt = cv2.Rodrigues(rt[:3])[0]
    assert pose.shape == (3, 4) and np.abs(pose[:, :3] - Rgt).max() < 1e-6 and np.abs(pose[:, 3] - rt[3:]).max() < 1e-6
    pose4 = native_ops.uncertainty_pnp(p2[:4], w[:4], p3[:4], K)
    assert pose4.shape == (3, 4) and np.abs(pose4[:, :3] @ pose4[:, :3].T - np.eye(3)).max() < 1e-6


def test_uncertainty_pnp_v2_covariance_form(dev):
    """un_pnp_utils.uncertainty_pnp_v2 (un_pnp_utils.py:81-158): per-point 2x2 covariances -> weight = 1 / largest eigenvalue
    (0 for a degenerate covariance), EPnP on the four best points, weighted refine.  Must equal uncertainty_pnp called with
    those weights as [w, 0, w] rows (the reference builds exactly that), and recover a noise-free pose."""
    import cv2
    from test_oracle_pinning import _upnp_problem

    from gdrnpp_bop2022_b200 import native_ops

    rs = np.random.RandomState(33)
    K, rt, p2, p3, _, _ = _upnp_problem(rs, 12, 0.0)
    sig = rs.uniform(0.5, 3.0, size=12)
    rot = rs.uniform(0, np.pi, size=12)
    covars = np.zeros((12, 2, 2))
    for i in range(12):   # anisotropic covariances: eigenvalues sig^2 and (0.3 sig)^2, rotated
        c, s_ = np.cos(rot[i]), np.sin(rot[i])
        Rm = np.array([[c, -s_], [s_, c]])
        covars[i] = Rm @ np.diag([sig[i] ** 2, (0.3 * sig[i]) ** 2]) @ Rm.T
    covars[3] = 0.0            # degenerate covariance -> weight 0 (covars[i,0,0] < 1e-5)
    w = np.where(covars[:, 0, 0] >= 1e-5, 1.0 / np.maximum(sig ** 2, 1e-30), 0.0)
    pose = native_ops.uncertainty_pnp_v2(p2, covars, p3, K)
    same = native_ops.uncertainty_pnp(p2, np.stack([w, np.zeros(12), w], 1), p3, K)
    assert pose.shape == (3, 4) and np.abs(pose - same).max() < 1e-9
    Rgt = cv2.Rodrigues(rt[:3])[0]
    assert np.abs(pose[:, :3] - Rgt).max() < 1e-6 and np.abs(pose[:, 3] - rt[3:]).max() < 1e-6
    pose4 = native_ops.uncertainty_pnp_v2(p2[:4], covars[[0, 1, 2, 4]], p3[:4], K)   # pn == 4: EPnP result only
    assert pose4.shape == (3, 4) and np.abs(pose4[:, :3] @ pose4[:, :3].T - np.eye(3)).max() < 1e-6


# --------------------------------------------------------------------- online training targets (SURVEY 8f-3)
def _ref_calc_xyz_bp_batch(depth, R, T, K):
    """lib/pysixd/misc.py:412-446 (fmt="BHWC"), restated verbatim in torch (pure-torch reference code)."""
    bs, height, width = depth.shape
    grid_y, grid_x = torch.meshgrid(torch.arange(height, device=depth.device, dtype=depth.dtype),
                                    torch.arange(width, device=depth.device, dtype=depth.dtype), indexing="ij")
    X = grid_x.expand(bs, height, width) - K[:, 0, 2].view(bs, 1, 1)
    Y = grid_y.expand(bs, height, width) - K[:, 1, 2].view(bs, 1, 1)
    xyz_cam = torch.stack((X * depth / K[:, 0, 0].view(bs, 1, 1), Y * depth / K[:, 1, 1].view(bs, 1, 1), depth), dim=-1)
    xyz_cam = xyz_cam.view(bs, height, width, 3, 1)
    Rinv_expand = R.permute(0, 2, 1).view(bs, 1, 1, 3, 3).expand(bs, height, width, 3, 3)
    T_expand = T.view(bs, 1, 1, 3, 1).expand(bs, height, width, 3, 1)
    mask = (depth != 0).to(depth).view(bs, height, width, 1)
    return torch.einsum("bhwij,bhwjk->bhwi", Rinv_expand, xyz_cam - T_expand) * mask


def test_online_targets_vs_reference_recipe(dev):
    """engine_utils.py:131-187 (XYZ_BP branch) on the GPU: ONE rasteriser launch over the mesh registry + ONE fused
    kernel, against the reference recipe restated in torch: calc_xyz_bp_batch (lib/pysixd/misc.py:412-457), roi_mask_obj
    (engine_utils.py:171-173), xyz_to_region_batch with the explicit mask (data_utils.py:283-301), roi_xyz = xyz / extent
    + 0.5 (:183).  Masks and region labels identical (up to distance ties), xyz to fp32 rounding; the back-projected
    points of an icosphere lie on its surface."""
    from gdrnpp_bop2022_b200 import native_ops
    from gdrnpp_bop2022_b200.online_targets import calc_xyz_bp_batch, render_roi_targets, xyz_to_region_batch
    from gdrnpp_bop2022_b200.renderer import Model3D
    from gdrnpp_bop2022_b200.synthetic import make_icosphere_mesh

    n = 6
    _, _, poses, Ks = _mesh_and_poses(n, seed=8)
    exts = [(0.12, 0.08, 0.1), (0.07, 0.11, 0.09)]
    models = [Model3D(*make_icosphere_mesh(3, e), device=dev) for e in exts]
    cls = torch.tensor([0, 1, 1, 0, 1, 0])
    ext_t = torch.tensor([exts[int(c)] for c in cls], dtype=torch.float32, device=dev)
    # 64 FPS points per object (the reference stores them with the dataset): our own bit-exact FPS
    fps = [native_ops.farthest_point_sampling(m.vertices.cpu().numpy(), 64, init_center=True) for m in models]
    fps_t = torch.from_numpy(np.stack([fps[int(c)] for c in cls])).to(dev)
    P, Kt = torch.from_numpy(poses).to(dev), torch.from_numpy(Ks).to(dev)
    R, T = P[:, :, :3].contiguous(), P[:, :, 3].contiguous()
    out = render_roi_targets(models, cls, R, T, Kt, ext_t, roi_fps_points=fps_t, out_res=64)
    depth = out["roi_depth"]
    ref_xyz = _ref_calc_xyz_bp_batch(depth, R, T, Kt)
    ref_mask = ((ref_xyz[..., 0] != 0) & (ref_xyz[..., 1] != 0) & (ref_xyz[..., 2] != 0)).to(torch.float32)
    ref_region = (torch.cdist(ref_xyz.view(n, -1, 3), fps_t, p=2).argmin(-1).view(n, 64, 64) + 1) * ref_mask
    ref_roi_xyz = ref_xyz.permute(0, 3, 1, 2) / ext_t.view(n, 3, 1, 1) + 0.5
    torch.cuda.synchronize()
    assert torch.equal(out["roi_mask_obj"], ref_mask) and 100 < float(ref_mask[0].sum()) < 3000
    assert (out["roi_xyz"] - ref_roi_xyz).abs().max().item() < 1e-5
    assert (out["roi_region"] != ref_region.long()).float().mean().item() < 1e-3      # equal up to nearest-point ties
    assert int(out["roi_region"].max()) <= 64 and out["roi_region"].dtype == torch.int64
    # API-level mirrors of the two reference helpers
    xyz = calc_xyz_bp_batch(depth, R, T, Kt)
    assert (xyz - ref_xyz).abs().max().item() < 1e-6
    assert torch.equal(xyz_to_region_batch(xyz, fps_t, mask=out["roi_mask_obj"]), (torch.cdist(xyz.view(n, -1, 3), fps_t).argmin(-1).view(n, 64, 64) + 1).long()
                       * out["roi_mask_obj"].long())
    # geometry: foreground points lie on the ellipsoid surface (mesh facets: a little inside)
    e = ext_t.view(n, 1, 1, 3) / 2
    rad = ((xyz / e) ** 2).sum(-1).sqrt()
    fg = out["roi_mask_obj"] > 0
    assert 0.85 < float(rad[fg].min()) and float(rad[fg].max()) < 1.1   # integer-pixel back-projection (the helper's convention) vs centre-sampled render


# ------------------------------------------------------------------------- YOLOX head post-processing (SURVEY 8f-4)
def _ref_yolox_postprocess(det_preds, num_classes, conf_thre, nms_thre, class_agnostic):
    """det/yolox/utils/boxes.py:34-80 restated verbatim (pure torch + torchvision reference code)."""
    import torchvision

    det_preds = det_preds.clone()
    box_corner = det_preds.new(det_preds.shape)
    box_corner[:, :, 0] = det_preds[:, :, 0] - det_preds[:, :, 2] / 2
    box_corner[:, :, 1] = det_preds[:, :, 1] - det_preds[:, :, 3] / 2
    box_corner[:, :, 2] = det_preds[:, :, 0] + det_preds[:, :, 2] / 2
    box_corner[:, :, 3] = det_preds[:, :, 1] + det_preds[:, :, 3] / 2
    det_preds[:, :, :4] = box_corner[:, :, :4]
    output = [None for _ in range(len(det_preds))]
    for i, image_pred in enumerate(det_preds):
        class_conf, class_pred = torch.max(image_pred[:, 5:5 + num_classes], 1, keepdim=True)
        conf_mask = (image_pred[:, 4] * class_conf.squeeze() >= conf_thre).squeeze()
        detections = torch.cat((image_pred[:, :5], class_conf, class_pred.float()), 1)[conf_mask]
        if not detections.size(0):
            continue
        if class_agnostic:
            keep = torchvision.ops.nms(detections[:, :4], detections[:, 4] * detections[:, 5], nms_thre)
        else:
            keep = torchvision.ops.batched_nms(detections[:, :4], detections[:, 4] * detections[:, 5], detections[:, 6], nms_thre)
        output[i] = detections[keep]
    return output


@pytest.mark.parametrize("class_agnostic", [False, True])
def test_yolox_postprocess_vs_reference_recipe(dev, class_agnostic):
    """GPU decode + confidence filter + NMS (one library call per batch, no sync) against the reference's postprocess
    (det/yolox/utils/boxes.py:34-80 with torchvision.ops.batched_nms / nms) and decode_outputs (yolo_head.py:239-255) on
    synthetic head outputs: clustered boxes around a few objects, 21 classes, one image with nothing above threshold."""
    pytest.importorskip("torchvision")
    from gdrnpp_bop2022_b200.yolox_post import postprocess, postprocess_padded

    g = torch.Generator().manual_seed(3)
    nc, B = 21, 3
    hw, strides = [(80, 80), (40, 40), (20, 20)], [8, 16, 32]
    A = sum(h * w for h, w in hw)
    raw = torch.zeros(B, A, 5 + nc)
    raw[..., :2] = torch.rand(B, A, 2, generator=g)                     # cell-relative centre
    raw[..., 2:4] = torch.randn(B, A, 2, generator=g) * 0.4 + 1.0       # log size
    raw[..., 4] = torch.rand(B, A, generator=g) ** 6                    # objectness: few confident anchors
    raw[..., 5:] = torch.rand(B, A, nc, generator=g) ** 3
    # plant clusters of near-duplicate confident boxes (what NMS is for)
    for b in range(2):
        for k in range(6):
            a0 = int(torch.randint(0, 6000, (1,), generator=g))
            raw[b, a0:a0 + 3, 4] = torch.tensor([0.95, 0.9, 0.85])
            raw[b, a0:a0 + 3, 5:] = 0.01
            raw[b, a0:a0 + 3, 5 + (k % nc)] = 0.9
            raw[b, a0:a0 + 3, :2] = 0.5
            raw[b, a0:a0 + 3, 2:4] = 1.5
    raw[2, :, 4] = 0.01                                                  # image 2: nothing survives the threshold
    raw = raw.to(dev)
    # reference: decode_outputs then postprocess
    grids, strs = [], []
    for (h, w), s in zip(hw, strides):
        yv, xv = torch.meshgrid([torch.arange(h), torch.arange(w)], indexing="ij")
        grids.append(torch.stack((xv, yv), 2).view(1, -1, 2))
        strs.append(torch.full((1, h * w, 1), s))
    grids, strs = torch.cat(grids, 1).float().to(dev), torch.cat(strs, 1).float().to(dev)
    dec = raw.clone()
    dec[..., :2] = (dec[..., :2] + grids) * strs
    dec[..., 2:4] = torch.exp(dec[..., 2:4]) * strs
    ref = _ref_yolox_postprocess(dec, nc, 0.3, 0.45, class_agnostic)
    for source, kwargs in ((raw, dict(hw=hw, strides=strides)), (dec, {})):          # raw head outputs / already-decoded boxes
        got = postprocess(source, nc, conf_thre=0.3, nms_thre=0.45, class_agnostic=class_agnostic, **kwargs)
        assert got[2] is None and ref[2] is None
        for b in range(2):
            assert got[b].shape == ref[b].shape, (b, got[b].shape, ref[b].shape)
            # same detections in the same (descending score) order; equal scores may swap
            sg, sr = got[b][:, 4] * got[b][:, 5], ref[b][:, 4] * ref[b][:, 5]
            assert torch.equal(sg, sr)
            assert (torch.sort(got[b], dim=0)[0] - torch.sort(ref[b], dim=0)[0]).abs().max().item() < 1e-4
            assert 6 <= got[b].shape[0] < 5000
    dets, n_det = postprocess_padded(raw, nc, 0.3, 0.45, class_agnostic, hw=hw, strides=strides, max_out=4)
    assert n_det.cpu().tolist()[:2] == [4, 4] and int(n_det[2]) == 0        # capped, still the top-scoring ones
    assert torch.equal(dets[0, :4], postprocess(raw, nc, 0.3, 0.45, class_agnostic, hw=hw, strides=strides)[0][:4])
