"""tcgen05 implicit-GEMM conv kernel (through the C ABI) vs a plain PyTorch fp32 conv of the same op."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

# name: (B,H,W,Cin,Cout,R,stride,dil,pad(t,b,l,r),bias,relu,res,res_shift)
CASES = {
    "1x1_small":         (1, 16, 24, 64, 64, 1, 1, 1, (0, 0, 0, 0), 0, 0, 0, 0),
    "1x1_bias_relu_res": (1, 16, 24, 256, 128, 1, 1, 1, (0, 0, 0, 0), 1, 1, 1, 0),
    "3x3_same_batch2":   (2, 20, 28, 64, 64, 3, 1, 1, (1, 1, 1, 1), 1, 1, 0, 0),      # M=1120: ragged last tile
    "3x3_s2_pad10":      (1, 24, 32, 64, 64, 3, 2, 1, (1, 0, 1, 0), 1, 1, 0, 0),      # nn.py:487-492
    "3x3_dil2":          (1, 23, 40, 128, 128, 3, 1, 2, (2, 2, 2, 2), 1, 1, 0, 0),    # res5 blocks 1,2
    "3x3_s2_dil2":       (1, 46, 80, 64, 64, 3, 2, 2, (1, 0, 1, 0), 1, 1, 0, 0),      # res5 block 0
    "1x1_s2_crop":       (2, 24, 32, 128, 256, 1, 2, 1, (0, -1, 0, -1), 1, 0, 0, 0),  # nn.py:555-560 shortcut
    "1x1_upsample_res":  (1, 24, 32, 128, 256, 1, 1, 1, (0, 0, 0, 0), 1, 0, 1, 1),    # FPN lateral + 2x nearest
    "3x3_bigK_N256":     (1, 23, 40, 512, 256, 3, 1, 1, (1, 1, 1, 1), 1, 1, 0, 0),    # 72 K-blocks: ring wraps
    "1x1_many_tiles":    (1, 200, 200, 64, 64, 1, 1, 1, (0, 0, 0, 0), 1, 0, 0, 0),    # 313 tiles > 148 SMs
    "1x1_N1024":         (1, 46, 80, 256, 1024, 1, 1, 1, (0, 0, 0, 0), 1, 1, 1, 0),
    "tiny_M":            (1, 3, 5, 64, 80, 1, 1, 1, (0, 0, 0, 0), 1, 0, 0, 0),        # M=15 < one tile, N=80
    "cout15":            (1, 12, 20, 256, 15, 1, 1, 1, (0, 0, 0, 0), 1, 0, 0, 0),     # RPN class+box fused N
}


def reference(spec, seed):
    B, H, W, Cin, Cout, R, stride, dil, pad, use_bias, relu, use_res, res_shift = spec
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((B, H, W, Cin)).astype(np.float32)
    w = (rng.standard_normal((R, R, Cin, Cout)) / np.sqrt(R * R * Cin)).astype(np.float32)
    bias = rng.standard_normal(Cout).astype(np.float32) if use_bias else None
    pt, pb, pl, pr = pad
    xt = torch.from_numpy(x).permute(0, 3, 1, 2)
    if pb < 0:
        xt = xt[:, :, :H + pb, :]
    if pr < 0:
        xt = xt[:, :, :, :W + pr]
    xt = F.pad(xt, (pl, max(pr, 0), pt, max(pb, 0)))
    ref = F.conv2d(xt, torch.from_numpy(w).permute(3, 2, 0, 1).contiguous(),
                   None if bias is None else torch.from_numpy(bias), stride=stride, dilation=dil)
    Ho, Wo = ref.shape[2:]
    res = None
    if use_res:
        rh, rw = ((Ho + 1) // 2, (Wo + 1) // 2) if res_shift else (Ho, Wo)
        res = rng.standard_normal((B, rh, rw, Cout)).astype(np.float32)
        rt = torch.from_numpy(res).permute(0, 3, 1, 2)
        if res_shift:
            rt = rt.repeat_interleave(2, 2).repeat_interleave(2, 3)[:, :, :Ho, :Wo]
        ref = ref + rt
    if relu:
        ref = torch.relu(ref)
    return x, w, bias, res, ref.permute(0, 2, 3, 1).contiguous().numpy()


@pytest.mark.parametrize("name", sorted(CASES))
@pytest.mark.parametrize("split,tol", [(True, 2e-5), (False, 3e-3)])
def test_conv_tc_matches_torch_fp32(name, split, tol):
    from object_detection_tracking_b200 import engine
    spec = CASES[name]
    x, w, bias, res, ref = reference(spec, seed=len(name))
    out = engine.op_conv2d(x, w, bias, res, stride=spec[6], dil=spec[7], pad=spec[8], relu=bool(spec[10]),
                           res_shift=spec[12], impl="tcgen05", split=split)
    assert out.shape == ref.shape
    assert np.isfinite(out).all()
    assert np.abs(out - ref).max() <= tol * np.abs(ref).max()     # tolerance: split ~fp32, fp16 operands ~2^-11


@pytest.mark.parametrize("name", ["1x1_small", "1x1_N1024", "1x1_upsample_res"])
def test_plain_1x1_through_im2col_tma_equals_tiled_tma(name):
    """The same GEMM with the A operand fetched by the im2col tensor map vs the plain 2-D map: identical bits."""
    from object_detection_tracking_b200 import engine
    spec = CASES[name]
    x, w, bias, res, _ = reference(spec, seed=3)
    kw = dict(stride=1, dil=1, pad=(0, 0, 0, 0), relu=bool(spec[10]), res_shift=spec[12], impl="tcgen05", split=True)
    a = engine.op_conv2d(x, w, bias, res, a_mode=0, **kw)
    b = engine.op_conv2d(x, w, bias, res, a_mode=1, **kw)
    np.testing.assert_array_equal(a, b)


@pytest.mark.parametrize("name", ["3x3_same_batch2", "3x3_s2_dil2", "1x1_s2_crop"])
def test_tensor_core_kernel_vs_cuda_core_kernel_same_operands(name):
    """Same fp16 (hi, lo) operands through tcgen05 and through the CUDA-core kernel: only the fp32
    accumulation order differs."""
    from object_detection_tracking_b200 import engine
    spec = CASES[name]
    x, w, bias, res, ref = reference(spec, seed=5)
    kw = dict(stride=spec[6], dil=spec[7], pad=spec[8], relu=bool(spec[10]), res_shift=spec[12], split=True)
    a = engine.op_conv2d(x, w, bias, res, impl="tcgen05", **kw)
    b = engine.op_conv2d(x, w, bias, res, impl="simt", **kw)
    assert np.abs(a - b).max() <= 5e-6 * np.abs(ref).max()


def test_direct_epilogue_path_equals_tma_staged_epilogue():
    """Both epilogue implementations (per-thread global access vs TMA-staged shared memory) give the same bits."""
    from object_detection_tracking_b200 import engine
    rng = np.random.default_rng(0)
    x = rng.standard_normal((2, 20, 28, 64)).astype(np.float32)
    w = (rng.standard_normal((3, 3, 64, 128)) / 24).astype(np.float32)
    b = rng.standard_normal(128).astype(np.float32)
    r = rng.standard_normal((2, 20, 28, 128)).astype(np.float32)
    kw = dict(pad=(1, 1, 1, 1), relu=True, split=True)
    staged = engine.op_conv2d(x, w, b, r, epi_mode=-1, **kw)
    direct = engine.op_conv2d(x, w, b, r, epi_mode=0, **kw)
    np.testing.assert_array_equal(staged, direct)


@pytest.mark.parametrize("name", ["1x1_bias_relu_res", "3x3_bigK_N256", "1x1_N1024", "3x3_dil2"])
def test_cta_pair_path_is_bit_identical(name):
    """The opt-in CTA-pair path (B2_PAIR: cta_group::2, two CTAs share 256-row tiles and the B operand) does the same
    arithmetic in the same order as the single-CTA kernel: identical bits, including the odd m-block count of the first
    case (the last pair's second block lies past M) and residual / ragged tiles."""
    import os
    from object_detection_tracking_b200 import engine
    spec = CASES[name]
    x, w, bias, res, _ = reference(spec, seed=11)
    kw = dict(stride=spec[6], dil=spec[7], pad=spec[8], relu=bool(spec[10]), res_shift=spec[12], impl="tcgen05", split=True)
    from object_detection_tracking_b200 import _lib
    lib = _lib.load()
    base = engine.op_conv2d(x, w, bias, res, **kw)
    n0 = lib.b2_conv_pair_launches()
    os.environ["B2_PAIR"] = "1"
    try:
        pair = engine.op_conv2d(x, w, bias, res, **kw)
    finally:
        os.environ.pop("B2_PAIR", None)
    assert lib.b2_conv_pair_launches() == n0 + 1      # the pair kernel really ran
    np.testing.assert_array_equal(base, pair)
