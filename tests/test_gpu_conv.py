"""csrc/conv.cu, the MinAtar embedding (channels-last frame -> Conv2d(C, OC, 3) + bias + ReLU + flatten), against
float64 autograd of torch's conv2d, at every path its backward dispatches to:

- the 3xTF32 tensor-core backward (``conv3x3_relu_bwd_mma_kernel<NT>``, NT = (9C + 8) / 8): every reachable NT,
- the FMA backward (``conv3x3_relu_bwd_kernel``): too few taps, an output plane that is not a multiple of 8 or
  exceeds 64, OC != 16, and PB_CONV_MMA=0 at the tensor-core shapes,
- batches past 296, where one CTA accumulates more than one sample before the fixed-order reduction.

Frames are real-valued: a binary frame splits exactly into its TF32 high part, so it cannot notice a missing
3xTF32 term (one binary case is kept as the MinAtar control).  Bars are fp32-level, 2e-5 of the tensor's max: a
single-pass TF32 product sits near 1e-3 and a dropped low-part product near 1e-4.

Also here: pb_conv3x3_relu_supported against a Python mirror of the kernel's limits (no GPU needed), and
MinAtarModel's cuDNN path for the frames the kernel refuses."""
import ctypes as C
import json
import os
import re
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

from helpers import rel_err

DEV = "cuda:0"
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

FWD_BAR = 2e-5
GRAD_BAR = 2e-5             # also at B 4096 (14 samples per CTA): dW 6.9e-6, db 3.0e-6 measured on a B200 at 1000 W
KINK = 1e-5                 # fp32 and fp64 ReLU gates may disagree only this close to 0, relative to the output's max


# ------------------------------------------------------------------------------------------------------------------
# Python mirror of the kernel's limits and dispatch
# ------------------------------------------------------------------------------------------------------------------
SMEM = 48 * 1024
MAX_X, MAX_W, MAX_OUT = 16 * 16 * 16, 32 * 16 * 9, 32 * 14 * 14


def frame_pitch(W):
    return ((W + 7) // 16) * 16 + 8


def mirror_supported(H, W, C_, OC):
    """check_dims in conv.cu: the dimension limits, then the forward's and the FMA backward's shared memory."""
    OH, OW = H - 2, W - 2
    if H < 3 or W < 3 or C_ <= 0 or OC <= 0:
        return False
    if H * W * C_ > MAX_X or OC * C_ * 9 > MAX_W or OC * OH * OW > MAX_OUT or OC * C_ * 9 + OC > 8 * 256:
        return False
    ocp = (OC + 7) // 8 * 8
    return 4 * (H * frame_pitch(W) * C_ + ocp * C_ * 9) <= SMEM and 4 * (H * W * C_ + OC * OH * OW) <= SMEM


def backward_path(H, W, C_, OC):
    """The backward pb_conv3x3_relu_bwd launches (PB_CONV_MMA unset), as the tensor-core condition in that entry
    (conv.cu) decides it: 'mma_nt<NT>' for the tensor-core kernel, 'fma_<reason>' for the FMA kernel."""
    plane, nt = (H - 2) * (W - 2), (9 * C_ + 1 + 7) // 8
    if OC != 16:
        return "fma_oc"
    if plane % 8 or plane > 64:
        return "fma_plane"
    if not 5 <= nt <= 12:
        return "fma_taps"
    if 4 * (H * frame_pitch(W) * C_ + 16 * 68 + plane + nt * 8) > SMEM:
        return "fma_smem"
    return "mma_nt%d" % nt


# ------------------------------------------------------------------------------------------------------------------
# inputs, reference, kernel
# ------------------------------------------------------------------------------------------------------------------
def make_inputs(B, H, W, C_, OC, frames="randn", bias=True, seed=0):
    g = torch.Generator().manual_seed(seed * 7919 + B * 31 + H * 17 + W * 13 + C_ * 5 + OC)
    if frames == "randn":
        x = torch.randn(B, H, W, C_, generator=g)
    elif frames == "u8":
        x = torch.randint(0, 256, (B, H, W, C_), generator=g, dtype=torch.uint8).float() / 255.0
    else:                                                                          # binary, as MinAtar emits
        x = (torch.rand(B, H, W, C_, generator=g) < 0.3).float()
    w = torch.randn(OC, C_, 3, 3, generator=g) / (9 * C_) ** 0.5
    b = torch.randn(OC, generator=g) * 0.1 if bias else None
    gy = torch.randn(B, OC * (H - 2) * (W - 2), generator=g)
    return x, w, b, gy


def reference(x, w, b, gy, out):
    """fp64 conv2d on the NCHW view.  Returns (pre-activation, ReLU output, dW, db); the gradients use the ReLU gate
    the kernel produced (out > 0): the gate is discontinuous, and the two precisions may differ right at 0."""
    wr = w.double().requires_grad_(True)
    br = None if b is None else b.double().requires_grad_(True)
    pre = F.conv2d(x.double().permute(0, 3, 1, 2), wr, br).flatten(1)
    (pre * (out.detach().cpu() > 0)).backward(gy.double())
    return pre.detach(), torch.relu(pre.detach()), wr.grad, None if br is None else br.grad


def run_kernel(x, w, b, gy):
    from prism_b200.agents import ops
    wd = w.to(DEV).requires_grad_(True)
    bd = None if b is None else b.to(DEV).requires_grad_(True)
    out = ops.conv3x3_relu_flatten(x.to(DEV), wd, bd)
    assert "ConvEmbed" in type(out.grad_fn).__name__
    out.backward(gy.to(DEV))
    torch.cuda.synchronize()
    return out.detach().cpu(), wd.grad.cpu(), None if bd is None else bd.grad.cpu()


def assert_gate_flips_near_zero(out, pre):
    """Every unit whose fp32 (kernel) and fp64 ReLU gates disagree has an fp64 pre-activation within KINK of 0."""
    flipped = (out > 0) != (pre > 0)
    if flipped.any():
        assert float(pre[flipped].abs().max()) < KINK * float(torch.relu(pre).abs().max())


def check_against_fp64(x, w, b, gy):
    """Kernel vs fp64 reference: forward within FWD_BAR, dW / db within GRAD_BAR, and every unit whose fp32 and fp64
    gates disagree within KINK of 0.  Returns the three relative errors."""
    out, dw, db = run_kernel(x, w, b, gy)
    pre, ref, dw_r, db_r = reference(x, w, b, gy, out)
    assert_gate_flips_near_zero(out, pre)
    errs = (rel_err(out.numpy(), ref.numpy()), rel_err(dw.numpy(), dw_r.numpy()),
            0.0 if b is None else rel_err(db.numpy(), db_r.numpy()))
    assert errs[0] < FWD_BAR, errs
    assert errs[1] < GRAD_BAR, errs
    assert errs[2] < GRAD_BAR, errs
    return errs


def backward_kernels(fn):
    """Names of the conv backward kernels that fn() launches, from the CUDA profiler: 'mma_nt<NT>' / 'fma'."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    got = set()
    for e in prof.events():
        m = re.search(r"conv3x3_relu_bwd_mma_kernel<(\d+)>", e.name)
        if m:
            got.add("mma_nt" + m.group(1))
        elif "conv3x3_relu_bwd_kernel" in e.name:
            got.add("fma")
    return got


# (B, H, W, C, OC, frames)
CASES = (
    [(256, 10, 10, c, 16, "randn") for c in range(4, 11)]                  # every reachable tensor-core instantiation
    + [(64, 6, 10, 6, 16, "randn"), (64, 3, 10, 4, 16, "randn")]          # tensor cores, planes of 32 and 8
    + [(64, 10, 10, c, 16, "randn") for c in (1, 2, 3)]                    # FMA: NT < 5
    + [(64, 7, 7, 4, 16, "randn"), (64, 11, 11, 6, 16, "randn"),           # FMA: plane 25, plane 81
       (32, 16, 16, 14, 16, "randn")]                                      # ... plane 196, the largest C taken
    + [(64, 10, 10, 4, oc, "randn") for oc in (1, 8, 12, 32)]              # FMA: OC != 16 (1, 12: padded to 8, 16)
    + [(b, 10, 10, 6, 16, "randn") for b in (1, 7, 272, 296, 297, 593, 4096)]   # one and several samples per CTA
    + [(256, 10, 10, 6, 16, "u8"), (256, 10, 10, 3, 16, "u8"), (256, 10, 10, 6, 16, "binary")])


def case_id(case):
    B, H, W, C_, OC, frames = case
    return "%s-B%d-%dx%dx%d-oc%d-%s" % (backward_path(H, W, C_, OC), B, H, W, C_, OC, frames)


# ------------------------------------------------------------------------------------------------------------------
# no GPU needed
# ------------------------------------------------------------------------------------------------------------------
def test_supported_query_matches_the_kernel_limits():
    """pb_conv3x3_relu_supported == the mirror of check_dims over every small frame; both entries refuse the shapes it
    refuses before touching their (dummy) pointers or the stream."""
    from prism_b200 import _lib
    lib = _lib.load()
    dummy = C.c_void_p(256)
    shapes = [(h, w, c, oc) for h in range(3, 17) for w in range(3, 17) for c in range(1, 17) for oc in (1, 8, 16, 32)]
    # 3x3x128 is the largest 3x3 frame the forward's shared memory takes (96 floats per channel for one filter), 129
    # channels pass every count of check_dims; the last two sit near the 4096-float frame limit
    shapes += [(3, 3, 128, 1), (3, 3, 129, 1), (3, 64, 21, 1), (66, 3, 20, 1)]
    refused = 0
    for H, W, C_, OC in shapes:
        want = mirror_supported(H, W, C_, OC)
        assert lib.pb_conv3x3_relu_supported(H, W, C_, OC) == int(want), (H, W, C_, OC)
        if not want:
            refused += 1
            assert lib.pb_conv3x3_relu_fwd(1, H, W, C_, OC, dummy, dummy, dummy, dummy, None) != 0, (H, W, C_, OC)
            assert lib.pb_conv3x3_relu_bwd(1, H, W, C_, OC, dummy, dummy, dummy, dummy, dummy, dummy, None) != 0
    assert refused > 1000
    assert lib.pb_conv3x3_relu_supported(10, 10, 14, 16) == 1 and lib.pb_conv3x3_relu_supported(10, 10, 15, 16) == 0
    assert mirror_supported(3, 3, 128, 1) and not mirror_supported(3, 3, 129, 1)
    assert 129 * 9 + 1 <= 8 * 256 and 3 * 3 * 129 <= MAX_X
    for bad in ((2, 10, 4, 16), (10, 2, 4, 16), (10, 10, 0, 16), (10, 10, 4, 0), (1 << 20, 1 << 20, 1 << 20, 16)):
        assert lib.pb_conv3x3_relu_supported(*bad) == 0, bad


def test_case_ids_cover_every_path():
    paths = {backward_path(*c[1:5]) for c in CASES}
    assert {"mma_nt%d" % nt for nt in (5, 6, 7, 8, 10, 11, 12)} <= paths       # NT 9: no C reaches it
    assert {"fma_taps", "fma_plane", "fma_oc"} <= paths
    assert 9 not in {(9 * c + 8) // 8 for c in range(1, 15)}


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_conv_matches_fp64(case):
    B, H, W, C_, OC, frames = case
    x, w, b, gy = make_inputs(B, H, W, C_, OC, frames)
    errs = check_against_fp64(x, w, b, gy)
    print("conv rel_err %s: fwd %.2e dW %.2e db %.2e" % ((case_id(case),) + errs))


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_backward_takes_the_expected_kernel(case):
    B, H, W, C_, OC, frames = case
    x, w, b, gy = make_inputs(B, H, W, C_, OC, frames)
    path = backward_path(H, W, C_, OC)
    assert backward_kernels(lambda: run_kernel(x, w, b, gy)) == {"fma" if path.startswith("fma") else path}


@pytest.mark.gpu
@pytest.mark.parametrize("case", [(256, 10, 10, 6, 16, "randn"), (64, 7, 7, 4, 16, "randn"),
                                  (64, 10, 10, 4, 8, "randn")], ids=case_id)
def test_conv_without_bias(case):
    """bias=None: the forward adds nothing, the backward writes no db (None) and a correct dW."""
    from prism_b200.agents import ops
    B, H, W, C_, OC, frames = case
    x, w, _, gy = make_inputs(B, H, W, C_, OC, frames, bias=False)
    check_against_fp64(x, w, None, gy)
    out = ops.conv3x3_relu_flatten(x.to(DEV), w.to(DEV).requires_grad_(True), None)
    _, dw, db = ops._ConvEmbed.backward(out.grad_fn, gy.to(DEV))
    torch.cuda.synchronize()
    assert db is None and dw.shape == (OC, C_, 3, 3)


FMA_CHILD_CASES = [(256, 10, 10, c, 16, "randn") for c in (4, 6, 10)]


def fma_child_main():
    """Body of the PB_CONV_MMA=0 child: the FMA backward at the tensor-core shapes (the switch is read once per
    process, so it cannot be flipped inside the parent)."""
    assert os.environ.get("PB_CONV_MMA") == "0"
    res = []
    for case in FMA_CHILD_CASES:
        x, w, b, gy = make_inputs(*case)
        kernels = backward_kernels(lambda: run_kernel(x, w, b, gy))
        res.append({"case": case_id(case), "kernels": sorted(kernels), "errs": check_against_fp64(x, w, b, gy)})
    print("FMA_CHILD " + json.dumps(res))


@pytest.mark.gpu
def test_fma_backward_at_tensor_core_shapes():
    env = dict(os.environ, PB_CONV_MMA="0")
    code = "import sys; sys.path[:0] = [%r, %r]; import test_gpu_conv; test_gpu_conv.fma_child_main()" % (HERE, ROOT)
    p = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                       timeout=300, env=env)
    assert p.returncode == 0, p.stdout[-3000:]
    line, = [l for l in p.stdout.splitlines() if l.startswith("FMA_CHILD ")]
    res = json.loads(line[len("FMA_CHILD "):])
    assert len(res) == len(FMA_CHILD_CASES)
    for r in res:
        print("conv rel_err PB_CONV_MMA=0 %s: fwd %.2e dW %.2e db %.2e" % ((r["case"],) + tuple(r["errs"])))
        assert r["kernels"] == ["fma"], r
        assert r["errs"][0] < FWD_BAR and max(r["errs"][1:]) < GRAD_BAR, r


@pytest.mark.gpu
@pytest.mark.parametrize("case", [(297, 10, 10, 6, 16, "randn"), (297, 10, 10, 3, 16, "randn")], ids=case_id)
def test_conv_is_deterministic_and_graph_replay_is_bit_exact(case):
    """Fixed-order reductions: two calls give the same bits, and so does a CUDA graph of forward + autograd.grad."""
    from prism_b200.agents import ops
    x, w, b, gy = (t.to(DEV) for t in make_inputs(*case))
    w.requires_grad_(True)
    b.requires_grad_(True)

    def step():
        out = ops.conv3x3_relu_flatten(x, w, b)
        dw, db = torch.autograd.grad(out, (w, b), gy)
        return out.detach(), dw, db

    first = [t.clone() for t in step()]
    second = step()
    torch.cuda.synchronize()
    assert all(torch.equal(a, c) for a, c in zip(first, second))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = step()
    for _ in range(2):
        for t in captured:
            t.fill_(float("nan"))
        graph.replay()
        torch.cuda.synchronize()
        assert all(torch.equal(a, c) for a, c in zip(first, captured))


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["uint8", "channels_last_view"])
def test_minatar_model_input_layouts(layout):
    """MinAtarModel(6) on CUDA takes uint8 frames and non-contiguous channels-last views through the kernel and
    matches the fp64 copy of its own nn.Sequential."""
    import copy
    from prism_b200.agents.models.cnn_models import MinAtarModel
    torch.manual_seed(3)
    model = MinAtarModel(6, device=DEV)
    g = torch.Generator().manual_seed(11)
    B = 256
    if layout == "uint8":
        x = torch.randint(0, 256, (B, 10, 10, 6), generator=g, dtype=torch.uint8)
        xd = x.to(DEV)
    else:
        x = torch.randn(B, 6, 10, 10, generator=g).permute(0, 2, 3, 1)
        xd = x.permute(0, 3, 1, 2).contiguous().to(DEV).permute(0, 2, 3, 1)
        assert not xd.is_contiguous()
    gy = torch.randn(B, model.output_dim, generator=g)
    out = model(xd)
    assert "ConvEmbed" in type(out.grad_fn).__name__
    out.backward(gy.to(DEV))
    torch.cuda.synchronize()
    ref = copy.deepcopy(model.model).cpu().double()
    xr = x.double().permute(0, 3, 1, 2)
    out = out.detach().cpu()
    assert rel_err(out.numpy(), ref(xr).detach().numpy()) < FWD_BAR
    ref.zero_grad()
    pre = ref[0](xr).flatten(1)
    assert_gate_flips_near_zero(out, pre.detach())
    (pre * (out > 0)).backward(gy.double())
    assert rel_err(model.model[0].weight.grad.cpu().numpy(), ref[0].weight.grad.numpy()) < GRAD_BAR
    assert rel_err(model.model[0].bias.grad.cpu().numpy(), ref[0].bias.grad.numpy()) < GRAD_BAR


@pytest.mark.gpu
@pytest.mark.parametrize("C_", [6, 3], ids=["mma_nt7", "fma_taps"])
def test_zero_windows_give_exact_zeros_and_no_gradient(C_):
    """Sparse init (zero bias, zero weights, one all-zero filter) on frames with all-zero 3x3 windows: the output is
    exactly 0 there, and an upstream gradient on those units reaches neither dW nor db."""
    import torch.nn as nn
    from prism_b200.agents.models.cnn_models import _sparse_conv_init
    B, H, W, OC = 64, 10, 10, 16
    torch.manual_seed(5)
    net = nn.Sequential(nn.Conv2d(C_, OC, 3))
    _sparse_conv_init(net, 0.5)
    w, b = net[0].weight.detach().clone(), net[0].bias.detach().clone()
    w[3] = 0.0
    assert not b.any()
    g = torch.Generator().manual_seed(C_)
    x = torch.randn(B, H, W, C_, generator=g)
    x[:, :5, :5, :] = 0.0                       # the windows at origins (0..2, 0..2)
    x[7] = 0.0                                  # a whole frame
    zero = torch.zeros(B, OC, H - 2, W - 2, dtype=torch.bool)
    zero[:, :, :3, :3] = True
    zero[7] = True
    zero[:, 3] = True
    zero = zero.flatten(1)
    gy = torch.randn(B, OC * (H - 2) * (W - 2), generator=g)
    out, dw, db = run_kernel(x, w, b, gy * zero)
    assert not out[zero].any()
    assert not dw.any() and not db.any()
    out, dw, db = run_kernel(x, w, b, gy)
    assert not out[zero].any() and not dw[3].any() and db[3] == 0
    check_against_fp64(x, w, b, gy)


@pytest.mark.gpu
@pytest.mark.parametrize("C_", [14, 15, 16], ids=["kernel-c14", "cudnn-c15", "cudnn-c16"])
def test_minatar_model_falls_back_to_fp32_cudnn(C_, monkeypatch):
    """Frames the kernel refuses (C > 14 at 10x10) take nn.Conv2d on cuDNN, still at fp32 accuracy although TF32 is
    torch's default for cuDNN convolutions."""
    from prism_b200.agents.models.cnn_models import MinAtarModel
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", True)
    model = MinAtarModel(C_, device=DEV)
    x, w, b, gy = make_inputs(64, 10, 10, C_, 16)
    conv = model.model[0]
    with torch.no_grad():
        conv.weight.copy_(w)
        conv.bias.copy_(b)
    out = model(x.to(DEV))
    assert ("ConvEmbed" in type(out.grad_fn).__name__) == (C_ <= 14)
    out.backward(gy.to(DEV))
    torch.cuda.synchronize()
    out = out.detach().cpu()
    _, ref, dw_r, db_r = reference(x, w, b, gy, out)
    errs = (rel_err(out.numpy(), ref.numpy()), rel_err(conv.weight.grad.cpu().numpy(), dw_r.numpy()),
            rel_err(conv.bias.grad.cpu().numpy(), db_r.numpy()))
    print("conv rel_err MinAtarModel(%d): fwd %.2e dW %.2e db %.2e" % ((C_,) + errs))
    assert errs[0] < FWD_BAR and errs[1] < GRAD_BAR and errs[2] < GRAD_BAR, errs


@pytest.mark.gpu
def test_minatar_model_rejects_a_frame_with_other_channels():
    """A frame whose channel count differs from the layer's is nn.Conv2d's shape error, as on the CPU, not a kernel
    call that would read (OC, C, 3, 3) weights the layer does not have."""
    from prism_b200.agents.models.cnn_models import MinAtarModel
    model = MinAtarModel(4, device=DEV)
    for c in (3, 6):
        with pytest.raises(RuntimeError, match="channels"):
            model(torch.zeros(8, 10, 10, c, device=DEV))
        with pytest.raises(RuntimeError, match="channels"):
            model.cpu()(torch.zeros(8, 10, 10, c))
        model.to(DEV)
