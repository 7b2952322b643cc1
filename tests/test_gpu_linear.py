"""csrc/linear.cu, the cluster split-K GEMM behind the learner-batch dense layers (pb_linear_fwd / bwd_input /
bwd_weight), against float64 math at every kernel, split factor and pipeline depth ``launch_gemm`` dispatches to:

- ``gemm_async_kernel<AK, BK, ROWSUM, STAGES>`` (cp.async tiles, 16-byte aligned operands): STAGES 2 (a split of at
  most 2 chunks of 32 along the inner dimension), STAGES 4 with the whole split in flight, and STAGES 4 with the ring
  wrapping (more than 4 chunks per split),
- ``gemm_kernel<AK, BK, ROWSUM>`` (register-staged tiles): unaligned shapes and pointers, at split factors 1, 2, 4 and 8,
- split-K factors 1, 2, 4 and 8, including a split that gets no chunks (272 rows = the padded data-parallel batch),
- the fused epilogue and operand work: bias, ReLU, the ReLU mask as a third operand, the bias gradient (ROWSUM),
  heads as a batch and heads as inner-dimension segments (``sum_heads``).

The entries are called directly, not through the ops routing, so each table shape reaches linear.cu whatever its
FLOP count.  Inputs are real-valued: a binary or integer operand splits exactly into its TF32 high part and cannot
notice a dropped 3xTF32 term.  The bar is 2e-5 of the tensor's max; ``test_bar_catches_a_missing_tf32_term`` shows on
the CPU that single-pass TF32 and 3xTF32 without its lo.hi term both exceed it on these inputs.

Which kernel runs is mirrored in Python (``plan``, no GPU needed) and checked against the kernel names and grids the
CUDA profiler records."""
import json
import re

import numpy as np
import pytest
import torch

from helpers import rel_err

DEV = "cuda:0"

BAR = 2e-5
SMS_B200 = 148
TAIL = 67                    # sentinel floats after every output: a store past M / N lands here
SENTINEL = 1234.5

# ------------------------------------------------------------------------------------------------------------------
# Python mirror of launch_gemm (linear.cu)
# ------------------------------------------------------------------------------------------------------------------
TM = TN = 64
TK = 32
NS = 4                       # cp.async stages of a split with more than 2 chunks
ENTRIES = ("fwd", "bwd_input", "bwd_weight")


def pick_splits(tiles, chunks, sms):
    s = 1
    while s < 8 and tiles * (s * 2) <= 2 * sms and chunks // (s * 2) >= 2:
        s *= 2
    return s


def async_eligible(ptrs_aligned, lda, ldb, strides, ak, bk, M, N, K):
    if not ptrs_aligned or (lda | ldb) & 3 or any(s & 3 for s in strides):
        return False
    return not ((K if ak else M) & 3) and not ((K if bk else N) & 3)


def gemm_args(entry, case, masked=False):
    """The GemmArgs an entry builds: (M, N, K, n_seg, batch, aligned) of the GEMM it launches."""
    K, M, N, J, shared, off = case
    xhs = 0 if shared else M * J
    x_ok, mask_ok = off != "x+1", not (masked and off == "mask+1")
    if entry == "fwd":                                    # A = X (k-major), B = W (k-major)
        return M, N, J, 1, K, async_eligible(x_ok, J, J, (xhs, N * J), True, True, M, N, J)
    if entry == "bwd_input":                              # A = dY (k-major), B = W (row-major along J)
        aligned = async_eligible(mask_ok, N, J, (M * N, N * J), True, False, M, J, N)
        return (M, J, N, K, 1, aligned) if shared else (M, J, N, 1, K, aligned)
    # bwd_weight: A = dY read as its transpose, B = X, neither contiguous along the inner dimension M
    return N, J, M, 1, K, async_eligible(x_ok and mask_ok, N, J, (M * N, xhs), False, False, N, J, M)


def plan(entry, case, sms=SMS_B200, masked=False):
    """What launch_gemm launches for `entry` on `case`: kernel ('async2', 'async4', 'reg'), split factor, chunks per
    split, grid and label."""
    gM, gN, gK, n_seg, batch, aligned = gemm_args(entry, case, masked)
    m_tiles, n_tiles = -(-gM // TM), -(-gN // TN)
    cps = -(-gK // TK)
    chunks = n_seg * cps
    splits = pick_splits(m_tiles * n_tiles * batch, chunks, sms)
    per = -(-chunks // splits)
    kernel = ("async2" if per <= 2 else "async4") if aligned else "reg"
    ranges = [(s * per, min(chunks, s * per + per)) for s in range(splits)]
    return {"kernel": kernel, "splits": splits, "per": per, "chunks": chunks, "cps": cps, "n_seg": n_seg,
            "ranges": ranges, "grid": [n_tiles, m_tiles * batch, splits],
            "label": "%s_s%d_per%d" % (kernel, splits, per)}


# (K heads, M rows, N outputs, J inputs, X shared by the heads, misaligned pointer)
TABLE = [
    (1, 256, 256, 1024, True, ""),        # the configs[1] layer
    (1, 272, 256, 1024, True, ""),        # the data-parallel padded batch: 16 live rows in the last M tile, an empty split
    (10, 64, 256, 1024, True, ""),        # forward ring wraps; input gradient over 10 head segments on s8
    (10, 64, 256, 1024, False, ""),
    (1, 64, 64, 4096, True, ""),          # forward: 16 chunks per split
    (10, 512, 256, 256, False, ""),       # weight gradient + ROWSUM with 16 chunks per split (ops would take tcgen05)
    (1, 512, 64, 64, True, ""),           # weight gradient on s8
    (2, 130, 96, 200, False, ""),         # ragged M / N / K
    (3, 64, 64, 36, False, ""),           # s1 everywhere
    (1, 100, 36, 68, True, ""),           # ragged K tail inside a 16-byte group
    (1, 256, 30, 256, True, ""),          # N % 4 != 0: scalar-store epilogue, both gradients register-staged
    (1, 64, 64, 1023, True, ""),          # register-staged forward on s8
    (3, 37, 19, 50, False, ""),           # fully unaligned
    (4, 5, 7, 3, True, ""),
    (1, 256, 256, 1024, True, "x+1"),     # X one float past a 16-byte boundary: only the input gradient stays on cp.async
    (1, 256, 256, 1024, True, "mask+1"),  # the ReLU mask one float past a 16-byte boundary, dY aligned
]

# (bias, act, Ymask, db): every option given and not given
VARIANTS = {"bias-relu-mask-db": (True, 1, True, True), "plain": (False, 0, False, False),
            "bias-db": (True, 0, False, True), "relu-mask": (False, 1, True, False)}

def case_id(case):
    K, M, N, J, shared, off = case
    return "K%d-M%d-N%d-J%d-%s%s" % (K, M, N, J, "shared" if shared else "perhead", "-" + off if off else "")


def coverage(table, sms=SMS_B200):
    """Required dispatch item -> id of the first table case that reaches it."""
    hit = {}

    def mark(item, case):
        hit.setdefault(item, case_id(case))

    for case in table:
        for entry in ENTRIES:
            p = plan(entry, case, sms, masked=True)
            k = p["kernel"]
            if k == "async2":
                mark("%s: async STAGES 2" % entry, case)
            if k == "async4":
                mark("%s: async STAGES 4, %s" % (entry, "ring wraps" if p["per"] > NS else "<= 4 chunks per split"), case)
            mark("%s: %d splits" % (entry, p["splits"]), case)
            if k == "reg":
                mark("reg kernel, %d splits" % p["splits"], case)
            if any(a >= b for a, b in p["ranges"]):
                mark("a split with zero chunks", case)
            if entry == "bwd_input" and p["n_seg"] > 1 and any(
                    a < b and a // p["cps"] != (b - 1) // p["cps"] for a, b in p["ranges"]):
                mark("bwd_input sum_heads: segments cross a split boundary", case)
            if entry == "bwd_weight":
                mark("bwd_weight with db on %s" % ("async" if k.startswith("async") else "register-staged"), case)
    return hit


REQUIRED = ([e + ": " + s for e in ENTRIES for s in ("async STAGES 2", "async STAGES 4, <= 4 chunks per split",
                                                      "async STAGES 4, ring wraps")]
            + [e + ": %d splits" % s for e in ENTRIES for s in (1, 2, 4, 8)]
            + ["reg kernel, %d splits" % s for s in (1, 2, 4, 8)]
            + ["a split with zero chunks",
               "bwd_input sum_heads: segments cross a split boundary",
               "bwd_weight with db on async", "bwd_weight with db on register-staged"])


# ------------------------------------------------------------------------------------------------------------------
# inputs, reference, kernel
# ------------------------------------------------------------------------------------------------------------------
def make_inputs(case, seed=0):
    """Real-valued X, W, b, dY and a ReLU mask holding exact 0.0, -0.0, negatives, a positive denormal (> 0 without
    flush-to-zero) and NaN (not > 0)."""
    K, M, N, J, shared, _ = case
    g = torch.Generator().manual_seed(seed * 7919 + K * 1009 + M * 31 + N * 7 + J)
    x = torch.randn((M, J) if shared else (K, M, J), generator=g)
    w = torch.randn(K, N, J, generator=g) / J ** 0.5
    b = torch.randn(K, N, generator=g)
    dy = torch.randn(K, M, N, generator=g)
    mask = torch.randn(K, M, N, generator=g)
    kind = torch.randint(0, 10, (K, M, N), generator=g)
    mask[kind == 0] = 0.0
    mask[kind == 1] = -0.0
    mask[kind == 2] = 1e-40
    mask[kind == 3] = float("nan")
    assert mask[kind == 2].min() > 0                      # the denormal survives on the host side
    return x, w, b, dy, mask


def reference(case, x, w, b, dy, mask, bias, act, masked, with_db):
    K, M, N, J, shared, _ = case
    x64, w64, dy64 = x.double(), w.double(), dy.double()
    xe = x64.unsqueeze(0).expand(K, M, J) if shared else x64
    y = xe @ w64.transpose(1, 2)
    if bias:
        y = y + b.double().unsqueeze(1)
    if act:
        y = torch.relu(y)
    dz = dy64 * (mask.double() > 0) if masked else dy64
    dx = dz @ w64
    if shared:
        dx = dx.sum(0)
    dw = dz.transpose(1, 2) @ xe
    return {"Y": y, "dX": dx, "dW": dw, "db": dz.sum(1) if with_db else None}


def _out(n):
    """n NaNs (every element must be written) followed by TAIL sentinels (none may be)."""
    t = torch.full((n + TAIL,), float("nan"), device=DEV)
    t[n:] = SENTINEL
    return t


def _device(t, off):
    """t on the device; off: one float past a 16-byte boundary (a legal, misaligned float pointer)."""
    if not off:
        return t.to(DEV).contiguous(), None
    buf = torch.empty(t.numel() + 4, device=DEV)
    view = buf[1:1 + t.numel()]
    view.copy_(t.flatten())
    assert view.data_ptr() % 16 == 4
    return view, buf


def run_entries(case, x, w, b, dy, mask, bias, act, masked, with_db):
    """pb_linear_fwd, _bwd_input (sum_heads = X shared) and _bwd_weight on freshly NaN-filled outputs."""
    from prism_b200 import _lib
    lib = _lib.load()
    K, M, N, J, shared, off = case
    xd, _keep_x = _device(x, off == "x+1")
    md, _keep_m = _device(mask, off == "mask+1")
    wd, bd, dyd = w.to(DEV), b.to(DEV), dy.to(DEV)
    xhs = 0 if shared else M * J
    stream = torch.cuda.current_stream().cuda_stream
    n = {"Y": K * M * N, "dX": (1 if shared else K) * M * J, "dW": K * N * J, "db": K * N}
    out = {k: _out(v) for k, v in n.items()}
    _lib.check(lib.pb_linear_fwd(K, M, N, J, xd.data_ptr(), xhs, wd.data_ptr(), bd.data_ptr() if bias else None, act,
                                 out["Y"].data_ptr(), stream), "pb_linear_fwd")
    mp = md.data_ptr() if masked else None
    _lib.check(lib.pb_linear_bwd_input(K, M, N, J, dyd.data_ptr(), mp, wd.data_ptr(), int(shared), out["dX"].data_ptr(),
                                       stream), "pb_linear_bwd_input")
    _lib.check(lib.pb_linear_bwd_weight(K, M, N, J, dyd.data_ptr(), mp, xd.data_ptr(), xhs, out["dW"].data_ptr(),
                                        out["db"].data_ptr() if with_db else None, stream), "pb_linear_bwd_weight")
    torch.cuda.synchronize()
    res = {}
    for k, t in out.items():
        t = t.cpu()
        body, tail = t[:n[k]], t[n[k]:]
        assert torch.equal(tail, torch.full((TAIL,), SENTINEL)), "%s: store past the end of the output" % k
        if k == "db" and not with_db:
            assert torch.isnan(body).all(), "db written although NULL was passed"
            continue
        assert not torch.isnan(body).any(), "%s: %d elements never written" % (k, int(torch.isnan(body).sum()))
        res[k] = body
    return res


def check_case(case, variant):
    """Every entry against fp64 within BAR; a second identical call gives the same bits.  Returns the errors."""
    bias, act, masked, with_db = VARIANTS[variant]
    x, w, b, dy, mask = make_inputs(case)
    got = run_entries(case, x, w, b, dy, mask, bias, act, masked, with_db)
    again = run_entries(case, x, w, b, dy, mask, bias, act, masked, with_db)
    for k in got:
        assert torch.equal(got[k], again[k]), "%s: two identical calls differ" % k
    ref = reference(case, x, w, b, dy, mask, bias, act, masked, with_db)
    errs = {k: rel_err(got[k].numpy(), ref[k].reshape(-1).numpy()) for k in got}
    assert max(errs.values()) < BAR, errs
    return errs


def entry_of(output):
    return {"Y": "fwd", "dX": "bwd_input", "dW": "bwd_weight", "db": "bwd_weight"}[output]


GEMM_NAME = re.compile(r"\b(gemm_async_kernel|gemm_kernel)<([^>]*)>")


def launched_gemms(fn, trace_path):
    """(kernel, ROWSUM, grid) of every linear.cu launch fn() makes, in launch order, from a chrome trace of the CUDA
    profiler: the template arguments name the kernel and its pipeline, gridDim.z is the split factor."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    prof.export_chrome_trace(str(trace_path))
    with open(str(trace_path)) as fh:
        events = json.load(fh)["traceEvents"]
    got = []
    for e in sorted((e for e in events if e.get("cat") == "kernel"), key=lambda e: e["ts"]):
        m = GEMM_NAME.search(e["name"])
        if not m:
            continue
        targs = [a.strip() for a in m.group(2).split(",")]
        kernel = "async%s" % targs[3] if m.group(1) == "gemm_async_kernel" else "reg"
        assert "grid" in e.get("args", {}), "the profiler trace records no grid for %s" % e["name"]
        got.append({"kernel": kernel, "rowsum": targs[2] == "true", "grid": list(e["args"]["grid"])})
    return got


def witness_table(trace_path):
    """Run every table case once (bias, ReLU, mask, db) under the profiler; returns (launched, expected)."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    inputs = [make_inputs(case) for case in TABLE]

    def run_all():
        for case, (x, w, b, dy, mask) in zip(TABLE, inputs):
            run_entries(case, x, w, b, dy, mask, True, 1, True, True)

    run_all()                                             # first launches set the kernels' attributes
    got = launched_gemms(run_all, trace_path)
    want = []
    for case in TABLE:
        for entry in ENTRIES:
            p = plan(entry, case, sms, masked=True)
            want.append({"kernel": p["kernel"], "rowsum": entry == "bwd_weight", "grid": p["grid"]})
    return got, want


# ------------------------------------------------------------------------------------------------------------------
# no GPU needed
# ------------------------------------------------------------------------------------------------------------------
def test_mirror_table_covers_every_dispatch_path():
    """At 148 SMs the table reaches every kernel, pipeline depth and split factor of every entry, an empty split, head
    segments crossing a split, and the bias gradient on both kernels.  Printed: the first shape reaching each item."""
    hit = coverage(TABLE)
    for item in REQUIRED:
        print("linear coverage %-55s %s" % (item, hit.get(item, "MISSING")))
    missing = [item for item in REQUIRED if item not in hit]
    assert not missing, missing
    # the labels the table's design notes rely on, fwd / bwd_input / bwd_weight
    labels = {c: tuple(plan(e, c)["label"] for e in ENTRIES) for c in TABLE}
    assert labels[TABLE[0]] == ("async4_s8_per4", "async2_s4_per2", "async2_s4_per2")
    assert labels[TABLE[1]] == ("async4_s8_per4", "async4_s2_per4", "async4_s4_per3")
    assert plan("bwd_weight", TABLE[1])["ranges"][3] == (9, 9)           # M = 272: 9 chunks on 4 splits of 3
    assert plan("fwd", TABLE[2])["per"] == 8 and plan("bwd_input", TABLE[2])["label"] == "async4_s8_per10"
    assert plan("bwd_input", TABLE[2])["n_seg"] == 10
    assert plan("fwd", TABLE[4])["per"] == 16
    assert plan("bwd_weight", TABLE[5])["label"] == "async4_s1_per16"
    assert plan("bwd_weight", TABLE[6])["splits"] == 8
    assert labels[TABLE[8]] == ("async2_s1_per2", "async2_s1_per2", "async2_s1_per2")
    assert labels[TABLE[10]][0].startswith("async") and labels[TABLE[10]][1:] == ("reg_s1_per1", "reg_s4_per2")
    assert labels[TABLE[11]][0] == "reg_s8_per4"
    x_off = [plan(e, TABLE[14], masked=True)["kernel"] for e in ENTRIES]
    assert x_off[0] == "reg" and x_off[1].startswith("async") and x_off[2] == "reg"
    mask_off = [plan(e, TABLE[15], masked=True)["kernel"] for e in ENTRIES]
    assert mask_off[0].startswith("async") and mask_off[1] == "reg" and mask_off[2] == "reg"


def _tf32(a):
    """The 19 bits the tensor core reads of an fp32 word (split_tf32: hi = word & 0xFFFFE000)."""
    return (np.ascontiguousarray(a, dtype=np.float32).view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)


def _emulated(a, b, terms):
    """a (M x K) . b (K x N) with the products of one 3xTF32 recipe, summed exactly in fp64."""
    ah, bh = _tf32(a), _tf32(b)
    al, bl = _tf32(a - ah), _tf32(b - bh)                 # x - hi is exact in fp32; the residual is read to 19 bits too
    d = lambda t: t.astype(np.float64)
    parts = {"hi.hi": d(ah) @ d(bh), "lo.hi": d(al) @ d(bh), "hi.lo": d(ah) @ d(bl)}
    return sum(parts[t] for t in terms)


def test_bar_catches_a_missing_tf32_term():
    """On the table's inputs, single-pass TF32 and 3xTF32 without lo.hi both miss the 2e-5 bar; the full
    lo.hi + hi.lo + hi.hi recipe stays below it.  Forward of the configs[1] layer, masked weight gradient of the
    data-parallel layer."""
    cases = []
    x, w, _, _, _ = make_inputs(TABLE[0])
    cases.append(("fwd " + case_id(TABLE[0]), x.numpy(), w[0].numpy().T))
    x, _, _, dy, mask = make_inputs(TABLE[1])
    cases.append(("bwd_weight " + case_id(TABLE[1]), (dy[0] * (mask[0] > 0)).numpy().T, x.numpy()))
    for name, a, b in cases:
        ref = a.astype(np.float64) @ b.astype(np.float64)
        err = {k: rel_err(_emulated(a, b, t), ref) for k, t in
               (("tf32", ["hi.hi"]), ("3xtf32 without lo.hi", ["hi.lo", "hi.hi"]), ("3xtf32", ["lo.hi", "hi.lo", "hi.hi"]))}
        print("linear emulated rel_err %s: %s" % (name, ", ".join("%s %.2e" % kv for kv in err.items())))
        assert err["tf32"] > BAR and err["3xtf32 without lo.hi"] > BAR, err
        assert err["3xtf32"] < BAR / 10, err


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("case", TABLE, ids=case_id)
def test_linear_entries_match_fp64(case, variant):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    errs = check_case(case, variant)
    masked = VARIANTS[variant][2]
    print("linear rel_err %s %s: %s" % (case_id(case), variant, ", ".join(
        "%s[%s] %.2e" % (k, plan(entry_of(k), case, sms, masked=masked)["label"], v) for k, v in errs.items())))


@pytest.mark.gpu
def test_profiler_sees_the_mirrored_gemm_kernels(tmp_path):
    """Kernel, pipeline depth, ROWSUM and grid (gridDim.z = split factor) of every launch over the table equal the
    mirror's plan at this GPU's SM count."""
    got, want = witness_table(tmp_path / "linear.pt.trace.json")
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert g == w, (case_id(TABLE[i // 3]), ENTRIES[i % 3], g, w)

