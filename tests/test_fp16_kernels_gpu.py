"""fp16 operand path (the default precision and the one bench.py measures), kernel by kernel, against float64 torch on the
same 16-bit operand values, plus the segmentation engine checked one stage at a time through its debug taps.

fp16 here means IEEE half bits stored in the bf16-typed plane buffers of the ABI, with the kernels' saturation: clamp to
+-65504, then round to nearest even (so 65520 and 1e6 become 65504, never inf).  The one-pass fp16 GEMM reads exact fp16
operand values, whose products are exact in fp32, so its fp32 output differs from the float64 contraction only by fp32
accumulation: the bound is 3e-5 of the output scale (not the 5e-4 the bf16 test needs for its operand rounding).  A 16-bit
output must sit within one 16-bit ulp of the reference (plus that fp32 slack, which matters only for values far below
the output scale)."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from diarizen_b200 import _lib
from gpu_util import act_ref, ptr, run_gemm, rup

pytestmark = pytest.mark.gpu

DEV = "cuda"
F16_MAX = 65504.0
DTYPE16 = {1: torch.float16, 0: torch.bfloat16}


# ------------------------------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------------------------------
def round16(x: torch.Tensor, fp16: int) -> torch.Tensor:
    """fp32 -> 16-bit values as the kernels round them (fp16: clamp to +-65504 first, then round to nearest even).
    NaN is not covered: to16() maps it to -65504 (fmaxf drops it) while pack2_16 keeps it."""
    if fp16:
        return x.clamp(-F16_MAX, F16_MAX).to(torch.float16)
    return x.to(torch.bfloat16)


def split16(x: torch.Tensor, fp16: int):
    """fp32 -> (hi, lo) 16-bit tensors: hi = rn(x), lo = rn(x - hi) with the fp32 subtraction the kernels do."""
    x = x.float()
    hi = round16(x, fp16)
    lo = round16(x - hi.float(), fp16)
    return hi, lo


def planes16(x: torch.Tensor, fp16: int = 1, ld: int = None, planes: int = 2) -> torch.Tensor:
    """fp32 (..., rows, cols) -> 16-bit planes (planes, ..., rows, ld) in the bf16-typed buffers of the ABI, zero padded."""
    cols = x.shape[-1]
    ld = ld or rup(cols, 8)
    out = torch.zeros((planes,) + tuple(x.shape[:-1]) + (ld,), dtype=torch.bfloat16, device=x.device)
    hi, lo = split16(x, fp16)
    out[0, ..., :cols] = hi.view(torch.bfloat16)
    if planes > 1:
        out[1, ..., :cols] = lo.view(torch.bfloat16)
    return out


def val16(p: torch.Tensor, fp16: int) -> torch.Tensor:
    """bf16-typed 16-bit cells -> float64 values under the given interpretation."""
    return p.view(DTYPE16[fp16]).double()


def hi_value(p: torch.Tensor, fp16: int) -> torch.Tensor:
    return val16(p[0], fp16)


def sum_value(p: torch.Tensor, fp16: int) -> torch.Tensor:
    return val16(p[0], fp16) + val16(p[1], fp16)


def ordered(bits16: torch.Tensor) -> torch.Tensor:
    """16-bit float bit patterns -> integers in the order of the values (adjacent representable values differ by 1)."""
    b = bits16.view(torch.int16).int()
    return torch.where(b < 0, -(b & 0x7FFF), b)


def ulp_diff(got16: torch.Tensor, ref: torch.Tensor, fp16: int) -> torch.Tensor:
    """Distance in 16-bit ulps between 16-bit cells and the 16-bit rounding of a float64 reference."""
    r = round16(ref.float(), fp16).view(torch.bfloat16)
    return (ordered(got16) - ordered(r)).abs()


def ulp16(ref: torch.Tensor, fp16: int) -> torch.Tensor:
    """Spacing of the 16-bit format at |ref| (float64)."""
    mant, emin = (10, -14) if fp16 else (7, -126)
    e = torch.floor(torch.log2(ref.abs().clamp_min(2.0 ** emin))).clamp_min(emin)
    return torch.pow(2.0, e - mant)


def check_one_plane(name, got16, ref, fp16, slack):
    """One 16-bit plane: within one ulp of the 16-bit rounding of `ref`, or within `slack` (the fp32-class error bound,
    absolute) where an ulp is smaller than that."""
    err = (val16(got16, fp16) - ref.clamp(-F16_MAX, F16_MAX) if fp16 else val16(got16, fp16) - ref).abs()
    ok = (ulp_diff(got16, ref, fp16) <= 1) | (err <= ulp16(ref, fp16) + slack)
    assert ok.all(), f"{name}: {int((~ok).sum())} cells off by more than 1 ulp, worst |err| {err[~ok].max().item():.3e}"


def check_rel(name, got, ref, tol):
    scale = ref.abs().max().item() + 1e-6
    err = (got.double() - ref).abs().max().item() / scale
    assert err < tol, f"{name}: rel err {err:.3e} (bound {tol:.1e})"
    return err


def lib():
    return _lib.lib()


# ------------------------------------------------------------------------------------------------------------------------
# 1. operand conversion: dz_rows_to_planes (bit-exact) and dz_channel_mean
# ------------------------------------------------------------------------------------------------------------------------
def _edge_values(fp16):
    t = [0.0, -0.0, 1.0, -1.0, F16_MAX, -F16_MAX, 65519.0, 65520.0, -65520.0, 1e6, -1e6, 65505.5, 3e38, -3e38, 1e-40, -1e-40]
    if fp16:
        t += [1 + 2 ** -11, 1 + 3 * 2 ** -11, -(1 + 2 ** -11), 2048 + 1, 2048 + 3,    # round-to-nearest-even ties
              2 ** -24, 2 ** -25, 3 * 2 ** -25, 5 * 2 ** -25, -3 * 2 ** -25, 2 ** -15, 1e-8, 6.1e-5, -2 ** -20]   # subnormals
    else:
        t += [1 + 2 ** -8, 1 + 3 * 2 ** -8, -(1 + 2 ** -8), 256 + 1, 256 + 3, 2 ** -133, 1.5 * 2 ** -133]
    return torch.tensor(t, dtype=torch.float32)


@pytest.mark.parametrize("fp16", [1, 0], ids=["fp16", "bf16"])
@pytest.mark.parametrize("planes", [1, 2])
@pytest.mark.parametrize("rows,C,ldx,ldo", [(37, 64, 64, 72), (300, 1024, 1028, 1024), (29, 100, 100, 104), (41, 13, 16, 16)],
                         ids=["vec8", "vec8_wide", "scalar_C100", "scalar_C13"])
def test_rows_to_planes_bit_exact(fp16, planes, rows, C, ldx, ldo):
    torch.manual_seed(rows + C)
    x = torch.randn(rows, ldx) * torch.pow(10.0, torch.randint(-6, 6, (rows, ldx)).float())
    edge = _edge_values(fp16)
    flat = x[:, :C].reshape(-1)
    flat[: edge.numel()] = edge
    flat[-edge.numel():] = edge.flip(0)
    x[:, :C] = flat.view(rows, C)
    xd = x.to(DEV)
    plane = rows * ldo + 64
    out = torch.full((planes * plane,), -7.0, dtype=torch.bfloat16, device=DEV)
    sentinel = out.clone()
    _lib.check(lib().dz_rows_to_planes(ptr(xd), rows, C, ldx, ptr(out), plane, ldo, planes, fp16, None))
    torch.cuda.synchronize()
    hi, lo = split16(x[:, :C], fp16)
    for p, ref in enumerate([hi, lo][:planes]):
        got = out[p * plane: p * plane + rows * ldo].view(rows, ldo).cpu()
        assert torch.equal(got[:, :C].view(torch.int16), ref.view(torch.int16)), \
            f"plane {p}: {(got[:, :C].view(torch.int16) != ref.view(torch.int16)).sum()} cells differ"
        assert torch.equal(got[:, C:], sentinel[:rows * (ldo - C)].view(rows, ldo - C).cpu()), "pad columns must stay untouched"
        if fp16:   # hi and lo both saturate at the rails, never reach inf
            v = got[:, :C].view(torch.float16).float()
            assert torch.isfinite(v).all(), "fp16 planes must saturate, never reach inf"
            assert (v.abs()[x[:, :C].abs() >= (2 if p == 0 else 3) * F16_MAX] == F16_MAX).all()


@pytest.mark.parametrize("Cn", [1, 2, 7])
def test_channel_mean(Cn):
    torch.manual_seed(Cn)
    B, T, D, ld = 3, 41, 100, 104
    x = torch.randn(B * Cn * T, ld, device=DEV) * 3 + 1
    out = torch.full((B * T, ld), 5.0, device=DEV)
    _lib.check(lib().dz_channel_mean(ptr(x), ptr(out), B, Cn, T, D, ld, None))
    torch.cuda.synchronize()
    ref = x.double().view(B, Cn, T, ld)[..., :D].mean(dim=1).reshape(B * T, D)
    assert (out[:, :D].double() - ref).abs().max().item() < 4e-6
    assert (out[:, D:] == 5.0).all(), "columns past D must stay untouched"


# ------------------------------------------------------------------------------------------------------------------------
# 2. dz_layernorm vs F.layer_norm in float64
# ------------------------------------------------------------------------------------------------------------------------
def _ln_call(x, rows, C, ldx, pre, gamma, beta, act, y=None, ldy=0, yb=None, bf_plane=0, ldb=0, planes=1, mix=None, mix_w=0.0,
             mix_src=0, mix_init=0, fp16=0):
    return lib().dz_layernorm(ptr(x), rows, C, ldx, ptr(pre), ptr(gamma), ptr(beta), act, ptr(y), ldy, ptr(yb), bf_plane, ldb,
                              planes, ptr(mix), mix_w, mix_src, mix_init, fp16, None)


def _ln_ref(x, C, pre, gamma, beta, act):
    xv = x[:, :C].double()
    if pre is not None:
        xv = xv * pre[:C].double()
    return act_ref(F.layer_norm(xv, (C,), gamma[:C].double(), beta[:C].double(), 1e-5), act)


def _ln_inputs(rows, C, ldx, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn(rows, ldx, device=DEV, generator=g) * 3 + 0.5
    gamma = 1 + 0.2 * torch.randn(C, device=DEV, generator=g)
    beta = 0.3 * torch.randn(C, device=DEV, generator=g)
    pre = 1 + 0.2 * torch.randn(C, device=DEV, generator=g)
    return x, gamma, beta, pre


BIG_ROWS = 60000   # > grid cap (148 SMs x 3 CTAs x 4) x rows per CTA pass (at most 32): the grid-stride loop iterates


@pytest.mark.parametrize("rows", [1, 7, 33, 1001, BIG_ROWS])
@pytest.mark.parametrize("C,ldx", [(130, 132), (256, 256), (384, 388), (512, 512), (1021, 1024), (1024, 1024)])
def test_layernorm_outputs(C, ldx, rows):
    """fp32 output and 16-bit planes (fp16 / bf16, one / two planes) for every activation, with and without prescale.
    NV = 2 / 4 / 8 float4 chunks per lane; C = 130, 1021 leave a chunk that straddles C."""
    x, gamma, beta, pre = _ln_inputs(rows, C, ldx, C + rows)
    ldy, ldb = rup(C, 4) + 4, rup(C, 8)
    for i in range(8):
        act, p = i % 4, (pre if i >= 4 else None)
        fp16, planes = [(1, 1), (1, 2), (0, 1), (0, 2)][(i + rows + C) % 4]
        y = torch.full((rows, ldy), 9.0, device=DEV)
        yb = torch.full((planes, rows, ldb), 9.0, device=DEV, dtype=torch.bfloat16)
        _lib.check(_ln_call(x, rows, C, ldx, p, gamma, beta, act, y, ldy, yb, rows * ldb, ldb, planes, fp16=fp16))
        torch.cuda.synchronize()
        ref = _ln_ref(x, C, p, gamma, beta, act)
        tag = f"act {act} prescale {p is not None} fp16 {fp16} planes {planes}"
        assert (y[:, :C].double() - ref).abs().max().item() < 2e-5, tag
        # the straddling float4 chunk is written with zeros in [C, rup(C, 4)); nothing past it is touched
        assert (y[:, C:rup(C, 4)] == 0).all() and (y[:, rup(C, 4):] == 9.0).all(), tag
        assert (yb[:, :, C:] == 0).all(), f"{tag}: pad columns of the planes must be zero"
        if planes == 1:
            check_one_plane(tag, yb[0, :, :C], ref, fp16, 2e-5)
        else:
            err = (sum_value(yb, fp16)[:, :C] - ref).abs() - ref.abs() * 2.0 ** -16
            assert err.max().item() < 2e-5, f"{tag}: hi + lo err {err.max().item():.3e}"


@pytest.mark.parametrize("planes", [1, 2])
def test_layernorm_fp16_saturates(planes):
    rows, C = 100, 384
    x, gamma, beta, _ = _ln_inputs(rows, C, C, 3)
    gamma = gamma * 1e5
    yb = torch.zeros((planes, rows, C), device=DEV, dtype=torch.bfloat16)
    _lib.check(_ln_call(x, rows, C, C, None, gamma, beta, 0, yb=yb, bf_plane=rows * C, ldb=C, planes=planes, fp16=1))
    torch.cuda.synchronize()
    ref = _ln_ref(x, C, None, gamma, beta, 0)
    h = val16(yb, 1)
    assert torch.isfinite(h).all(), "fp16 planes must saturate, never reach inf"
    big = ref.abs() > F16_MAX + 16
    assert big.sum() > 1000
    assert (h[0][big] == torch.sign(ref[big]) * F16_MAX).all()
    small = ref.abs() < 60000          # fp32 LayerNorm error (~2e-5) scaled by gamma ~ 1e5: 2 absolute
    assert ((h[0] - ref).abs()[small] <= ulp16(ref, 1)[small] + 2.0).all()


@pytest.mark.parametrize("mix_src", [1, 2])
@pytest.mark.parametrize("mix_init", [0, 1])
@pytest.mark.parametrize("C,ldx,rows", [(256, 256, 33), (256, 256, BIG_ROWS), (1024, 1024, 1001), (1021, 1024, 77), (130, 136, 5000)])
def test_layernorm_layer_mix(C, ldx, rows, mix_src, mix_init):
    """mix += w * (x | y) next to an fp16 plane output (the pre-norm encoder's LayerNorm); C % 4 != 0 runs the generic
    kernel, which must leave the mix columns past C untouched too."""
    x, gamma, beta, _ = _ln_inputs(rows, C, ldx, C * 3 + rows + mix_src)
    mix = torch.randn(rows, ldx, device=DEV)
    mix0 = mix.clone()
    yb = torch.full((1, rows, rup(C, 8)), 9.0, device=DEV, dtype=torch.bfloat16)
    w = 0.37
    _lib.check(_ln_call(x, rows, C, ldx, None, gamma, beta, 1, yb=yb, bf_plane=0, ldb=rup(C, 8), planes=1, mix=mix, mix_w=w,
                        mix_src=mix_src, mix_init=mix_init, fp16=1))
    torch.cuda.synchronize()
    ref = _ln_ref(x, C, None, gamma, beta, 1)
    src = x[:, :C].double() if mix_src == 1 else ref
    mref = (0 if mix_init else mix0[:, :C].double()) + w * src
    assert (mix[:, :C].double() - mref).abs().max().item() < 2e-5
    assert torch.equal(mix[:, C:], mix0[:, C:]), "mix columns past C must stay untouched"
    check_one_plane("y", yb[0, :, :C], ref, 1, 2e-5)


@pytest.mark.parametrize("case", ["valid", "ldx%4", "ldy%4", "ldb%8", "bf_plane%8", "C=0", "C>1024", "ldx<C"])
def test_layernorm_rejects_bad_arguments(case):
    """Misaligned strides would send the float4 / 8-byte accesses of either kernel off alignment: rejected before launch."""
    rows, C = 16, 1021
    x, gamma, beta, _ = _ln_inputs(rows, 1100, 1100, 1)
    y = torch.full((rows, 1100), 9.0, device=DEV)
    yb = torch.full((2 * rows * 1104 + 64,), 9.0, device=DEV, dtype=torch.bfloat16)
    args = dict(ldx=1024, ldy=1024, ldb=1024, bf_plane=rows * 1024, C=C)
    args.update({"valid": {}, "ldx%4": dict(ldx=1022), "ldy%4": dict(ldy=1022), "ldb%8": dict(ldb=1028), "bf_plane%8": dict(bf_plane=rows * 1024 + 4),
                 "C=0": dict(C=0), "C>1024": dict(C=1025, ldx=1028, ldy=1028, ldb=1032), "ldx<C": dict(ldx=1020)}[case])
    rc = _ln_call(x, rows, args["C"], args["ldx"], None, gamma, beta, 0, y, args["ldy"], yb, args["bf_plane"], args["ldb"], 2, fp16=1)
    torch.cuda.synchronize()
    if case == "valid":   # the same call with aligned strides runs
        assert rc == 0 and not (y[:, :C] == 9.0).all()
        return
    assert rc == -1, f"{case}: expected DZ_ERR_INVALID, got {rc}"
    assert (y == 9.0).all() and (yb == 9.0).all(), "a rejected call must not launch"


# ------------------------------------------------------------------------------------------------------------------------
# 3. GEMM with fp16 operands (one pass)
# ------------------------------------------------------------------------------------------------------------------------
TOL32 = 3e-5


def _lin_desc(Ap, Wp, M, N, K):
    d = _lib.GemmDesc.default()
    d.M, d.N, d.K, d.npass, d.fp16 = M, N, K, 1, 1
    d.a, d.a_plane, d.a_rstride, d.a_kinner, d.a_rows_alloc = ptr(Ap).value, Ap[0].numel(), Ap.shape[-1], K, M
    d.b, d.b_plane, d.ldb, d.b_gstride = ptr(Wp).value, Wp[0].numel(), Wp.shape[-1], Wp[0].numel()
    return d


@pytest.mark.parametrize("impl", [0, 1], ids=["tc", "simt"])
@pytest.mark.parametrize("out", ["f32", "h1", "h2", "r1", "r2"])
@pytest.mark.parametrize("M,N,K,bn", [(300, 200, 136, 0), (128, 64, 64, 64), (257, 666, 768, 128), (513, 1092, 1024, 256),
                                     (96, 11, 256, 0), (1000, 384, 53, 0), (200, 100, 96, 64)])
def test_linear_epilogue_fp16(impl, out, M, N, K, bn):
    """Every activation, alpha != 1, activation before and after the residual.  Outputs: fp32 (+ fp32 residual), one or two
    16-bit planes, and 16-bit planes plus an fp16 residual read from planes of the same count (res16).  These are the
    single-output shapes the TMA-store epilogue takes (tc impl)."""
    torch.manual_seed(M + N + K)
    A = torch.randn(M, K, device=DEV)
    W = torch.randn(N, K, device=DEV) / K ** 0.5
    bias = torch.randn(rup(N, 64) + 64, device=DEV)
    Ap, Wp = planes16(A, 1, planes=1), planes16(W, 1, planes=1)
    ldn = rup(N, 8)
    planes = 2 if out in ("h2", "r2") else 1
    res32 = torch.randn(M, ldn, device=DEV)
    rp = planes16(torch.randn(M, ldn, device=DEV) * 2, 1, ldn, planes)
    acc = hi_value(Ap, 1)[:, :K] @ hi_value(Wp, 1)[:, :K].T + bias[:N].double()
    for act in range(4):
        for after in (0, 1):
            alpha = 0.75
            d = _lin_desc(Ap, Wp, M, N, K)
            d.bias, d.act, d.alpha, d.act_after_res = ptr(bias).value, act, alpha, after
            if out == "f32":
                res = res32[:, :N].double()
                o = torch.full((M, ldn), 7.0, device=DEV)
                d.residual, d.ldr = ptr(res32).value, ldn
                d.out_f32, d.ldo = ptr(o).value, ldn
            else:
                res = (hi_value(rp, 1) + (val16(rp[1], 1) if planes == 2 else 0))[:, :N] if out[0] == "r" else 0.0
                o = torch.full((planes, M, ldn), 7.0, device=DEV, dtype=torch.bfloat16)
                d.out_bf, d.ob_plane, d.ldob, d.out_planes, d.zero_pad_to = ptr(o).value, o[0].numel(), ldn, planes, ldn
                if out[0] == "r":
                    d.res16, d.res16_plane, d.ldr16 = ptr(rp).value, rp[0].numel(), ldn
            run_gemm(d, impl, bn)
            ref = act_ref(alpha * acc + res, act) if after else alpha * act_ref(acc, act) + res
            tag = f"{out} act {act} after_res {after}"
            scale = ref.abs().max().item()
            if out == "f32":
                check_rel(tag, o[:, :N], ref, TOL32)
                # the TMA store moves 16-byte units: it writes zeros into [N, rup(N, 4)) and nothing past that
                assert ((o[:, N:rup(N, 4)] == 7.0) | (o[:, N:rup(N, 4)] == 0)).all() and (o[:, rup(N, 4):] == 7.0).all(), \
                    "fp32 output must not touch pad columns past the 16-byte unit that holds column N - 1"
            elif planes == 1:
                check_one_plane(tag, o[0, :, :N], ref, 1, TOL32 * scale)
                assert (o[:, :, N:] == 0).all(), "pad columns must be zeroed"
            else:
                check_rel(tag, sum_value(o, 1)[:, :N], ref, TOL32)
                assert (o[:, :, N:] == 0).all(), "pad columns must be zeroed"


@pytest.mark.parametrize("impl", [0, 1], ids=["tc", "simt"])
@pytest.mark.parametrize("planes", [1, 2])
@pytest.mark.parametrize("generic", [False, True], ids=["tma_store", "generic"])
def test_gemm_fp16_output_saturates(impl, planes, generic):
    """Outputs beyond 65504 are stored as exactly +-65504 in the hi plane (and never as inf in either plane)."""
    torch.manual_seed(11)
    M, N, K = 256, 192, 128
    A, W = torch.randn(M, K, device=DEV), torch.randn(N, K, device=DEV) / K ** 0.5
    Ap, Wp = planes16(A, 1, planes=1), planes16(W, 1, planes=1)
    o = torch.zeros((planes, M, N), device=DEV, dtype=torch.bfloat16)
    of = torch.zeros((M, N), device=DEV)
    d = _lin_desc(Ap, Wp, M, N, K)
    d.alpha = 4e4
    d.out_bf, d.ob_plane, d.ldob, d.out_planes = ptr(o).value, o[0].numel(), N, planes
    if generic:   # a second (fp32) output takes the generic epilogue
        d.out_f32, d.ldo = ptr(of).value, N
    run_gemm(d, impl)
    ref = 4e4 * (hi_value(Ap, 1)[:, :K] @ hi_value(Wp, 1)[:, :K].T)
    v = val16(o, 1)
    assert torch.isfinite(v).all()
    big = ref.abs() > F16_MAX * 1.01
    assert big.sum() > 100
    assert (v[0][big] == torch.sign(ref[big]) * F16_MAX).all()
    inside = ref.abs() < F16_MAX * 0.99
    assert ((v[0] - ref).abs()[inside] <= ulp16(ref, 1)[inside] + TOL32 * F16_MAX).all()


@pytest.mark.parametrize("impl", [0, 1], ids=["tc", "simt"])
@pytest.mark.parametrize("planes", [1, 2])
def test_transposed_output_fp16(impl, planes):
    """q|k row-major + v^T planes from one projection GEMM, fp16 operands and outputs."""
    torch.manual_seed(5)
    B, T, D, h = 2, 99, 256, 3
    M, N = B * T, 3 * h * 64
    A, W = torch.randn(M, D, device=DEV), torch.randn(N, D, device=DEV) / D ** 0.5
    Ap, Wp = planes16(A, 1, planes=1), planes16(W, 1, planes=1)
    Tp = rup(T, 8)
    qk = torch.zeros(planes, M, 2 * h * 64, device=DEV, dtype=torch.bfloat16)
    vt = torch.zeros(planes, B, h * 64, Tp, device=DEV, dtype=torch.bfloat16)
    d = _lin_desc(Ap, Wp, M, N, D)
    d.out_bf, d.ob_plane, d.ldob, d.out_planes = ptr(qk).value, qk[0].numel(), 2 * h * 64, planes
    d.out_t, d.ot_plane, d.ot_bstride, d.ldt, d.tr_col0, d.seq_len = ptr(vt).value, vt[0].numel(), h * 64 * Tp, Tp, 2 * h * 64, T
    run_gemm(d, impl)
    ref = hi_value(Ap, 1) @ hi_value(Wp, 1).T
    vref = ref[:, 2 * h * 64:].reshape(B, T, h * 64).permute(0, 2, 1)
    scale = ref.abs().max().item()
    if planes == 1:
        check_one_plane("qk", qk[0], ref[:, :2 * h * 64], 1, TOL32 * scale)
        check_one_plane("vt", vt[0, ..., :T], vref, 1, TOL32 * scale)
    else:
        check_rel("qk", sum_value(qk, 1), ref[:, :2 * h * 64], TOL32)
        check_rel("vt", sum_value(vt, 1)[..., :T], vref, TOL32)
    assert (vt[..., T:] == 0).all()


def _conv1d_operands(B, Tin, Cin, Cout, k, seed):
    torch.manual_seed(seed)
    x = torch.randn(B, Tin, Cin, device=DEV)
    w = torch.randn(Cout, Cin, k, device=DEV) / (Cin * k) ** 0.5
    Cp = rup(Cin, 8)
    xp = planes16(x, 1, Cp, planes=1)
    wr = torch.zeros(Cout, k, Cp, device=DEV)
    wr[:, :, :Cin] = w.permute(0, 2, 1)
    wp = planes16(wr.reshape(Cout, k * Cp), 1, planes=1)
    Tout = (Tin - k) // 2 + 1
    d = _lib.GemmDesc.default()
    d.M, d.N, d.K, d.npass, d.batches, d.fp16 = Tout, Cout, k * Cp, 1, B, 1
    d.a, d.a_plane, d.a_rstride, d.a_kinner, d.a_bstride, d.a_rows_alloc = ptr(xp).value, xp[0].numel(), 2 * Cp, k * Cp, Tin * Cp, Tout
    d.b, d.b_plane, d.ldb, d.b_gstride = ptr(wp).value, wp[0].numel(), wp.shape[-1], wp[0].numel()
    xv = hi_value(xp, 1)[..., :Cin].permute(0, 2, 1)
    wv = hi_value(wp, 1).reshape(Cout, k, Cp)[:, :, :Cin].permute(0, 2, 1)
    y = F.conv1d(xv, wv, stride=2).permute(0, 2, 1)
    return d, (xp, wp), y, Tout


@pytest.mark.parametrize("impl", [0, 1], ids=["tc", "simt"])
@pytest.mark.parametrize("B,Tin,Cin,Cout,k", [(3, 401, 24, 40, 3), (2, 1000, 153, 224, 3), (2, 300, 90, 161, 2)])
def test_conv1d_as_strided_gemm_fp16(impl, B, Tin, Cin, Cout, k):
    d, keep, y, Tout = _conv1d_operands(B, Tin, Cin, Cout, k, Tin)
    ldo = rup(Cout, 8)
    out = torch.zeros(B, Tout, ldo, device=DEV)
    d.act, d.out_f32, d.ldo, d.of_bstride = 1, ptr(out).value, ldo, Tout * ldo
    run_gemm(d, impl)
    check_rel("conv", out[..., :Cout], F.gelu(y), TOL32)


@pytest.mark.parametrize("planes", [1, 2])
@pytest.mark.parametrize("B,Tin,Cin,Cout", [(2, 1000, 153, 224), (2, 777, 512, 153), (3, 401, 24, 40), (1, 300, 224, 255)])
def test_conv1d_with_fused_layernorm_gelu_fp16(planes, B, Tin, Cin, Cout):
    """conv1d -> LayerNorm(channels) -> GELU in one launch, fp16 operands and 16-bit outputs (the conv stack of the
    benchmarked layer-norm extractor)."""
    d, keep, y, Tout = _conv1d_operands(B, Tin, Cin, Cout, 3, Tin + Cout)
    gamma, beta = torch.zeros(rup(Cout, 32), device=DEV), torch.zeros(rup(Cout, 32), device=DEV)
    gamma[:Cout] = 1.0 + 0.2 * torch.randn(Cout, device=DEV)
    beta[:Cout] = 0.3 * torch.randn(Cout, device=DEV)
    ldo = rup(Cout, 8)
    out = torch.full((planes, B, Tout, ldo), 7.0, device=DEV, dtype=torch.bfloat16)
    d.act, d.ln_gamma, d.ln_beta, d.ln_eps = 1, ptr(gamma).value, ptr(beta).value, 1e-5
    d.out_bf, d.ob_plane, d.ldob, d.ob_bstride, d.out_planes, d.zero_pad_to = ptr(out).value, out[0].numel(), ldo, Tout * ldo, planes, ldo
    run_gemm(d, 0)
    ref = F.gelu(F.layer_norm(y, (Cout,), gamma[:Cout].double(), beta[:Cout].double(), 1e-5))
    # the accumulator error (TOL32 of the conv output scale) is amplified by scale / std of the row when normalised
    if planes == 1:
        check_one_plane("ln+gelu", out[0, ..., :Cout], ref, 1, 5e-5)
    else:
        check_rel("ln+gelu planes", sum_value(out, 1)[..., :Cout], ref, 5e-5)
    assert (out[..., Cout:ldo] == 0).all(), "pad columns must be zeroed"


@pytest.mark.parametrize("impl", [0, 1], ids=["tc", "simt"])
@pytest.mark.parametrize("planes", [1, 2])
@pytest.mark.parametrize("B,H,W,Cin,Cout,ks,stride,res", [(2, 10, 50, 32, 32, 3, 1, True), (1, 20, 199, 32, 64, 3, 2, False),
                                                         (2, 8, 130, 64, 128, 1, 2, False), (1, 6, 300, 128, 128, 3, 1, True),
                                                         (1, 5, 77, 256, 256, 3, 1, True)])
def test_conv2d_as_gemm_fp16(impl, planes, B, H, W, Cin, Cout, ks, stride, res):
    """ResNet conv2d (+ folded BN bias, fp16 residual planes, ReLU after the add) with fp16 operands."""
    torch.manual_seed(W + planes)
    x = torch.randn(B, Cin, H, W, device=DEV)
    w = torch.randn(Cout, Cin, ks, ks, device=DEV) / (Cin * ks * ks) ** 0.5
    bias = torch.randn(rup(Cout, 64) + 64, device=DEV)
    pad = 1 if ks == 3 else 0
    Ho, Wo = (H + 2 * pad - ks) // stride + 1, (W + 2 * pad - ks) // stride + 1
    Wp, Wop = W + 2, Wo + 2
    xin = torch.zeros(B, H, Wp, Cin, device=DEV)
    xin[:, :, 1:W + 1] = x.permute(0, 2, 3, 1)
    xp = planes16(xin.reshape(B * H * Wp, Cin), 1, planes=1)
    xp = torch.cat([xp, torch.zeros(1, 64, Cin, device=DEV, dtype=xp.dtype)], dim=1).contiguous()
    run_len = ks * Cin
    krun = rup(run_len, 64)
    wr = torch.zeros(Cout, ks, krun, device=DEV)
    wr[:, :, :run_len] = w.permute(0, 2, 3, 1).reshape(Cout, ks, ks * Cin)
    wp = planes16(wr.reshape(Cout, ks * krun), 1, planes=1)
    resid = torch.randn(B, Ho, Wop, Cout, device=DEV)
    resid[:, :, 0] = 0; resid[:, :, -1] = 0
    rp = planes16(resid.reshape(B * Ho * Wop, Cout), 1, planes=planes)
    out = torch.zeros(planes, B * Ho * Wop, Cout, device=DEV, dtype=torch.bfloat16)
    d = _lib.GemmDesc.default()
    d.M, d.N, d.K, d.npass, d.batches, d.fp16 = Wo, Cout, ks * krun, 1, B * Ho, 1
    d.a, d.a_plane, d.a_rstride, d.a_bstride, d.a_hstride = ptr(xp).value, xp[0].numel(), stride * Cin, H * Wp * Cin, Wp * Cin
    d.a_kinner = d.K
    d.conv_runs, d.conv_run_len, d.conv_x0, d.conv_h0, d.conv_hs, d.conv_Ho, d.conv_H = ks, run_len, (0 if ks == 3 else Cin), -pad, stride, Ho, H
    d.b, d.b_plane, d.ldb, d.b_gstride = ptr(wp).value, wp[0].numel(), ks * krun, wp[0].numel()
    d.bias, d.act, d.act_after_res = ptr(bias).value, 3, 1
    if res:
        d.res16, d.res16_plane, d.res16_bstride, d.ldr16, d.res16_row_off = ptr(rp).value, rp[0].numel(), Wop * Cout, Cout, 1
    d.out_bf, d.ob_plane, d.ob_bstride, d.ldob, d.out_row_off, d.out_planes = ptr(out).value, out[0].numel(), Wop * Cout, Cout, 1, planes
    run_gemm(d, impl)
    xv = hi_value(xp, 1)[:B * H * Wp].view(B, H, Wp, Cin)[:, :, 1:W + 1].permute(0, 3, 1, 2)
    wv = hi_value(wp, 1).view(Cout, ks, krun)[:, :, :run_len].reshape(Cout, ks, ks, Cin).permute(0, 3, 1, 2)
    ref = F.conv2d(xv, wv, bias[:Cout].double(), stride=stride, padding=pad)
    if res:
        rv = hi_value(rp, 1) + (val16(rp[1], 1) if planes == 2 else 0)
        ref = ref + rv.view(B, Ho, Wop, Cout)[:, :, 1:Wo + 1].permute(0, 3, 1, 2)
    ref = torch.relu(ref).permute(0, 2, 3, 1)
    scale = ref.abs().max().item()
    if planes == 1:
        got = out[0].view(B, Ho, Wop, Cout)
        check_one_plane("conv2d", got[:, :, 1:Wo + 1], ref, 1, TOL32 * scale)
        g = hi_value(out, 1).view(B, Ho, Wop, Cout)
    else:
        g = sum_value(out, 1).view(B, Ho, Wop, Cout)
        check_rel("conv2d planes", g[:, :, 1:Wo + 1], ref, TOL32)
    assert (g[:, :, 0] == 0).all() and (g[:, :, -1] == 0).all(), "zero border must stay untouched"


@pytest.mark.parametrize("impl", [0, 1], ids=["tc", "simt"])
@pytest.mark.parametrize("B,T,D", [(2, 49, 128), (2, 249, 768), (1, 300, 1024)])
def test_grouped_posconv_fp16(impl, B, T, D):
    """Grouped conv1d(k=128, pad=64, groups=16) + bias + GELU + residual through the GEMM, fp16 operands."""
    torch.manual_seed(T)
    G, KT = 16, 128
    Dg = D // G
    x = torch.randn(B, T, D, device=DEV)
    w = torch.randn(D, Dg, KT, device=DEV) / (Dg * KT) ** 0.5
    bias = torch.randn(D + 64, device=DEV)
    stage = torch.zeros(B, T + 128, G, 64, device=DEV)
    stage[:, 64:64 + T, :, :Dg] = x.view(B, T, G, Dg)
    sp = planes16(stage.view(B, T + 128, G * 64), 1, planes=1)
    wr = torch.zeros(G, Dg, KT, 64, device=DEV)
    wr[:, :, :, :Dg] = w.view(G, Dg, Dg, KT).permute(0, 1, 3, 2)
    wp = planes16(wr.view(G * Dg, KT * 64), 1, planes=1)
    res = x.clone().view(B * T, D).contiguous()
    d = _lib.GemmDesc.default()
    d.M, d.N, d.K, d.npass, d.batches, d.groups, d.fp16 = T, Dg, KT * 64, 1, B, G, 1
    d.a, d.a_plane, d.a_rstride, d.a_kinner, d.a_kouter, d.a_gstride = ptr(sp).value, sp[0].numel(), G * 64, 64, G * 64, 64
    d.a_bstride, d.a_rows_alloc = (T + 128) * G * 64, T
    d.b, d.b_plane, d.ldb, d.b_gstride = ptr(wp).value, wp[0].numel(), KT * 64, Dg * KT * 64
    d.bias, d.act, d.group_cols = ptr(bias).value, 1, Dg
    d.residual, d.res_bstride, d.ldr = ptr(res).value, T * D, D
    d.out_f32, d.of_bstride, d.ldo = ptr(res).value, T * D, D
    run_gemm(d, impl)
    xv = hi_value(sp, 1).view(B, T + 128, G, 64)[:, 64:64 + T, :, :Dg].reshape(B, T, D)
    wv = hi_value(wp, 1).view(G, Dg, KT, 64)[..., :Dg].permute(0, 1, 3, 2).reshape(D, Dg, KT)
    pc = F.conv1d(xv.permute(0, 2, 1), wv, bias[:D].double(), padding=64, groups=G)[..., :-1]
    ref = x.double() + F.gelu(pc).permute(0, 2, 1)
    check_rel("posconv", res.view(B, T, D), ref, TOL32)


# ------------------------------------------------------------------------------------------------------------------------
# 4. attention with fp16 operands
# ------------------------------------------------------------------------------------------------------------------------
# tc: P is rounded to the 16-bit format before P.V (fp16: 2^-11 relative, bf16: 2^-8); simt: fp32 throughout
ATT_TOL = {("tc", 1): 4e-3, ("tc", 0): 1.5e-2, ("simt", 1): 2e-4, ("simt", 0): 2e-4}


def _run_attention(q, k, v, tab, gate, impl, vrow, fp16):
    """q, k, v (B, T, h, 64) fp32 -> (kernel output (B*T, h*64) float64, float64 reference on the 16-bit operand values)."""
    B, T, h, _ = q.shape
    cols = [q.reshape(B * T, h * 64), k.reshape(B * T, h * 64)] + ([v.reshape(B * T, h * 64)] if vrow else [])
    qkp = planes16(torch.cat(cols, dim=1), fp16, planes=1)
    Tp = rup(T, 8)
    vtp = planes16(v.permute(0, 2, 3, 1).reshape(B, h * 64, T), fp16, Tp, planes=1)
    out = torch.zeros(2, B * T, h * 64, device=DEV, dtype=torch.bfloat16)
    a = _lib.AttnArgs()
    a.T, a.nheads, a.fp16 = T, h, fp16
    a.q = a.k = ptr(qkp).value
    a.qk_plane, a.ldqk, a.q_col, a.k_col = qkp[0].numel(), (3 if vrow else 2) * h * 64, 0, h * 64
    a.planes = 1
    if vrow:
        a.v, a.v_col = ptr(qkp).value, 2 * h * 64
    else:
        a.vt, a.vt_plane, a.ldvt = ptr(vtp).value, vtp[0].numel(), Tp
    a.bias_tab = ptr(tab).value if tab is not None else None
    a.gate = ptr(gate).value if gate is not None else None
    a.out, a.out_plane, a.ldo, a.out_planes = ptr(out).value, out[0].numel(), h * 64, 2
    _lib.check(lib().dz_attention(ctypes.byref(a), B, {"tc": 0, "simt": 1}[impl], None))
    torch.cuda.synchronize()
    x = hi_value(qkp, fp16)
    qv = x[:, :h * 64].view(B, T, h, 64).permute(0, 2, 1, 3)
    kv = x[:, h * 64:2 * h * 64].view(B, T, h, 64).permute(0, 2, 1, 3)
    vv = hi_value(vtp, fp16)[..., :T].view(B, h, 64, T).permute(0, 1, 3, 2)
    s = qv @ kv.transpose(-1, -2)
    if tab is not None:
        idx = (torch.arange(T, device=DEV)[None, :] - torch.arange(T, device=DEV)[:, None]) + T - 1
        s = s + gate.double()[..., None] * tab.double()[:, idx][None]
    ref = (torch.softmax(s, dim=-1) @ vv).permute(0, 2, 1, 3).reshape(B * T, h * 64)
    return sum_value(out, fp16), ref


@pytest.mark.parametrize("impl,vrow", [("tc", 0), ("tc", 1), ("simt", 1)], ids=["tc-vT", "tc-vrow", "simt"])
@pytest.mark.parametrize("bias", [True, False], ids=["bias", "nobias"])
@pytest.mark.parametrize("h", [1, 3, 5])
@pytest.mark.parametrize("T", [49, 63, 64, 65, 127, 128, 129, 249, 799])
def test_attention_fp16(impl, vrow, T, h, bias):
    """attention_tc2_kernel<1, 0> / <1, 1> and the CUDA-core kernel with fp16 operands."""
    torch.manual_seed(T * 7 + h)
    B = 2
    q = torch.randn(B, T, h, 64, device=DEV) * 0.5
    k, v = torch.randn(B, T, h, 64, device=DEV), torch.randn(B, T, h, 64, device=DEV)
    tab = torch.randn(h, 2 * T - 1, device=DEV) if bias else None
    gate = (1.0 + torch.rand(B, h, T, device=DEV)) if bias else None
    got, ref = _run_attention(q, k, v, tab, gate, impl, vrow, 1)
    err = (got - ref).abs().max().item()
    assert err < ATT_TOL[(impl, 1)], f"max err {err:.3e}"


@pytest.mark.parametrize("fp16", [1, 0], ids=["fp16", "bf16"])
@pytest.mark.parametrize("impl,vrow", [("tc", 0), ("tc", 1), ("simt", 1)], ids=["tc-vT", "tc-vrow", "simt"])
@pytest.mark.parametrize("profile,T", [("rising", 249), ("rising", 799), ("falling", 249), ("falling", 799), ("last_key", 65),
                                       ("last_key", 129), ("huge", 129), ("huge", 799)])
def test_attention_online_softmax_profiles(profile, T, impl, vrow, fp16):
    """Score profiles aimed at the online softmax bookkeeping of the tensor-core kernel:
    rising   - bias climbing along the keys: the row maximum moves by far more than 2^8 every key block, so every block
               re-references and rescales O and its ones-column denominator;
    falling  - the maximum sits in block 0 and later blocks underflow (nothing re-references);
    last_key - the row maximum is the last valid key of a partial last block;
    huge     - raw scores of a few hundred in magnitude."""
    torch.manual_seed(T + len(profile))
    B, h = 2, 2
    q = torch.randn(B, T, h, 64, device=DEV) * 0.1
    k, v = torch.randn(B, T, h, 64, device=DEV), torch.randn(B, T, h, 64, device=DEV)
    tab = gate = None
    rel = torch.arange(-(T - 1), T, device=DEV, dtype=torch.float32)     # k - q
    if profile in ("rising", "falling"):
        tab = (0.25 if profile == "rising" else -0.25) * rel.repeat(h, 1).contiguous()
        gate = torch.ones(B, h, T, device=DEV)
    elif profile == "last_key":
        q[..., 0] = 1.0
        k[:, T - 1, :, 0] = 30.0
    else:
        q, k = q * 50, k * 5          # |q.k| ~ 150 typical, a few hundred at the row maximum
    got, ref = _run_attention(q, k, v, tab, gate, impl, vrow, fp16)
    err = (got - ref).abs().max().item()
    # scores of a few hundred carry fp32 rounding (~|s| * 2^-24 per term) into the exponent: 2.5e-4 measured for simt
    tol = max(ATT_TOL[(impl, fp16)], 5e-4) if profile == "huge" else ATT_TOL[(impl, fp16)]
    assert err < tol, f"max err {err:.3e}"


# ------------------------------------------------------------------------------------------------------------------------
# 5. segmentation engine, one stage at a time
# ------------------------------------------------------------------------------------------------------------------------
def _stage_errors(arch_name, precision, seconds=16.0, windows=2):
    """Runs the engine once and compares every stage with the float64 oracle of that stage fed with the engine's own
    input to it (its tap), so that errors do not compound from stage to stage.  -> {stage: error}: max |err| over
    max |ref| (absolute for the log-probs)."""
    from diarizen_b200.archs import get_arch, init_state_dict
    from diarizen_b200.segmentation import SegmentationModel
    from oracle import seg_oracle as O
    a = get_arch(arch_name)
    sd32 = init_state_dict(a, 1)
    sd = {k: v.to(DEV, torch.float64) for k, v in sd32.items()}
    N = int(seconds * 16000)
    wav = 0.1 * torch.randn(windows, N, generator=torch.Generator().manual_seed(1234))
    m = SegmentationModel(a, sd32, precision=precision, gemm_impl="tc", attn_impl="tc")
    logp, _ = m.hard(wav.unsqueeze(1))
    torch.cuda.synchronize()
    T = a.num_frames(N)
    B = windows

    def tap(name, cols):
        return m.tap(name).view(B, -1, cols).double()

    def rel(got, ref):
        return ((got - ref).abs().max() / ref.abs().max()).item()

    errs = {}
    with torch.no_grad():
        w = wav.to(DEV, torch.float64)
        x0 = F.layer_norm(w, w.shape[-1:]) if a.large else w
        c0 = O.conv_layer(a, sd, 0, x0.unsqueeze(1)).transpose(1, 2)
        errs["conv0"] = rel(tap("conv0", a.conv_channels[0]), c0)
        D = a.embed_dim
        errs["proj->rep0"] = rel(tap("rep0", D), O.pos_conv(a, sd, tap("proj", D)))
        bias = O.encoder_bias(a, sd, T)
        reps = [tap("rep0", D)]
        for l in range(a.num_layers):
            x = reps[l]
            if a.heads[l]:
                pre = f"wavlm_model.encoder.transformer.layers.{l}."
                xin = F.layer_norm(x, (D,), sd[pre + "layer_norm.weight"], sd[pre + "layer_norm.bias"]) if a.large else x
                ctx = O.wavlm_attention_context(a, sd, pre + "attention.", xin, a.heads[l], bias)
                errs[f"rep{l}->L{l}_ctx"] = rel(tap(f"L{l}_ctx", 64 * len(a.heads[l])), ctx)
            reps.append(tap(f"rep{l + 1}", D))
            errs[f"rep{l}->rep{l + 1}"] = rel(reps[l + 1], O.wavlm_layer(a, sd, l, x, bias))
        mix = tap("mix", D)
        wsum = sum(sd["weight_sum.weight"][0, l] * reps[l] for l in range(a.num_layers + 1))
        errs["reps->mix"] = rel(mix, wsum)
        A = a.head_dim_model
        x = tap("head_in", A)
        errs["mix->head_in"] = rel(x, O.head_input(sd, mix))
        for i in range(a.head_layers):
            y = tap(f"C{i}_out", A)
            errs[f"C{i - 1}_out->C{i}_out" if i else "head_in->C0_out"] = rel(y, O.conformer_block(a, sd, f"conformer.conformer_layer.{i}.", x))
            x = y
        errs["head->logp"] = (logp.double() - O.classify(sd, x)).abs().max().item()
    return errs


def _kind(stage):
    """Stages of the same kind share one bound."""
    if stage.startswith("rep") and "_ctx" in stage:
        return "ctx"
    if stage.startswith("rep") and stage.split("->")[1].startswith("rep"):
        return "layer"
    if stage.startswith("C") or stage.startswith("head_in->"):
        return "conformer"
    return stage


# Bounds per stage kind (max |err| / max |ref|; log-probs absolute): twice the worst value measured over both
# architectures (wavlm_large_s80_md: 2 x 16 s windows, tiny_base: 2 x 4 s, init_state_dict seed 1) on an NVIDIA B200
# (1000 W power limit).  The measured values are listed in test_engine_stages.__doc__.  bf16x3 is the control: it sits
# at fp32-class error, one to two orders of magnitude below fp16 on every stage that rounds operands to 16 bits.
STAGE_BOUNDS = {
    "fp16": {"conv0": 1.1e-3, "proj->rep0": 3.3e-4, "ctx": 1.2e-3, "layer": 4.1e-4, "reps->mix": 4e-7, "mix->head_in": 6.8e-4,
             "conformer": 3.1e-4, "head->logp": 1.1e-6},
    "bf16x3": {"conv0": 1.4e-5, "proj->rep0": 4.6e-5, "ctx": 2.8e-5, "layer": 1.1e-5, "reps->mix": 4e-7, "mix->head_in": 1.3e-5,
               "conformer": 4.6e-6, "head->logp": 1.1e-6},
}


@pytest.mark.parametrize("precision", ["fp16", "bf16x3"])
@pytest.mark.parametrize("arch,seconds", [("wavlm_large_s80_md", 16.0), ("tiny_base", 4.0)])
def test_engine_stages(arch, seconds, precision):
    """Every stage of the engine (tc GEMMs, tc attention) against the float64 oracle of that stage on the engine's own
    stage input: waveform -> conv0 (wave_stats + conv0_tc for large, conv0_moments + gn_coef for base), proj -> rep0
    (pos-conv), rep<l> -> L<l>_ctx (LayerNorm, QKV, gate, attention), rep<l> -> rep<l+1>, reps -> mix, mix -> head_in,
    conformer blocks (GLU depthwise conv, SiLU and alpha = 0.5 GEMMs), last block -> log-probs.

    Worst value per stage kind measured on a B200 (large / tiny_base):
                    fp16                  bf16x3
      conv0         4.71e-4 / 5.45e-4     6.89e-6 / 5.82e-6
      proj->rep0    8.51e-5 / 1.61e-4     2.27e-5 / 9.47e-6
      L<l>_ctx      5.56e-4 / 5.58e-4     1.39e-5 / 6.98e-6
      rep<l+1>      2.02e-4 / 1.12e-4     5.35e-6 / 1.58e-6
      mix           1.77e-7 / 6.62e-8     1.78e-7 / 5.93e-8
      head_in       3.20e-4 / 3.38e-4     5.12e-6 / 6.15e-6
      C<i>_out      1.54e-4 / 8.16e-5     2.29e-6 / 1.41e-6
      log-probs     5.01e-7 / 4.79e-7     5.12e-7 / 4.74e-7   (absolute; the classifier runs in fp32)"""
    errs = _stage_errors(arch, precision, seconds)
    bounds = STAGE_BOUNDS[precision]
    bad = {s: e for s, e in errs.items() if not e < bounds[_kind(s)]}
    assert not bad, f"{arch}/{precision}: stages over their bound: " + ", ".join(f"{s} {e:.2e} (bound {bounds[_kind(s)]:.0e})"
                                                                               for s, e in bad.items())
