"""The engine's GEMM argument forms on every kernel route, element by element against an fp64 reference (B200).

Each case runs one call-site form of csrc/engine.cu (tests/_gemm_sites.py) through bw_test_gemm -- batched (Z), broadcast
(zero z-stride) operands / bias / residual, z-strided bias, padded operands (a_rows / b_rows), swap-AB, in place on the
residual stream, operands that start inside a larger buffer -- and checks:
  * every written element: |C - ref| <= gamma * S + rho(ref), S = |A|.|B|^T + |bias| + |residual| (the magnitudes that
    the fp32 accumulation and the fp32 epilogue round), rho = half a bf16 ulp of the rounded reference for bf16 output,
    0 for fp32 output; ref in fp64 on the stored (bf16 or fp32) operands with exact erf-GELU;
  * rows behind M / N (a_rows / b_rows), columns behind K (lda > K in the forced-route cases) and everything around
    the operands hold NaN, so any read of them shows up in the result;
  * C is pre-filled with a NaN pattern, and every element outside the written extent -- before and after C, behind ldc,
    behind c_zstride -- must keep that pattern bit for bit;
  * route_taken is the route the CPU table (tests/test_gemm_routes_cpu.py) expects.
The exact-epilogue test multiplies by one-hot B rows (exact accumulator), so bias / GELU / residual order and the GELU
approximation are compared to fp64 at fp32 precision on every route."""
import ctypes as C
import zlib

import pytest

from tests import _gemm_sites as G

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]

torch = pytest.importorskip("torch")

# Per-element bound |C - ref| <= GAMMA * S + rho, calibrated once on an NVIDIA B200 (1000 W power limit) over every case
# of this file: worst observed (err - rho) / S of the tcgen05 kernels 7.75e-7 (large-v3 enc_w2, K = 5120, tile128), of
# the SIMT kernel 3.65e-7 (fp32 validation mode); GAMMA is 4x that or less.
GAMMA_TC = 3.0e-6
GAMMA_SIMT = 1.4e-6

GUARD = {torch.float32: 0x7FC0DEAD, torch.bfloat16: 0x7FAD}  # NaN bit patterns (quiet NaN with a payload)
INT_VIEW = {torch.float32: torch.int32, torch.bfloat16: torch.int16}
LEAD = 64  # guard elements in front of every buffer


def _lib():
    from b200_whisper import _lib as L

    return L, L.load()


def _nan_buffer(n, dtype):
    buf = torch.empty(n, device="cuda", dtype=dtype)
    buf.view(INT_VIEW[dtype]).fill_(GUARD[dtype])
    return buf


class Operand:
    """`slices` matrices [rows, cols] with leading dimension ld and slice stride zs inside a NaN-filled flat buffer that
    starts `lead` elements before the first one; rows >= `live` of each slice stay NaN (a_rows / b_rows padding).
    values: [slices, live, cols] (default random * scale); False leaves every element NaN."""

    def __init__(self, dtype, slices, rows, cols, ld, zs, lead=LEAD, live=None, gen=None, scale=1.0, values=None, tail=LEAD):
        self.dtype, self.slices, self.rows, self.cols, self.ld, self.zs, self.lead = dtype, slices, rows, cols, ld, zs, lead
        self.live = rows if live is None else live
        extent = (slices - 1) * zs + (rows - 1) * ld + cols
        self.buf = _nan_buffer(lead + extent + tail, dtype)
        if values is None:
            values = torch.randn((slices, self.live, cols), device="cuda", generator=gen, dtype=torch.float32) * scale
        if values is not False:
            self.view(self.buf)[:, :self.live, :] = values.to(dtype)

    def view(self, buf):
        return torch.as_strided(buf, (self.slices, self.rows, self.cols), (self.zs, self.ld, 1), self.lead)

    def ptr(self):
        return self.buf.data_ptr() + self.lead * self.buf.element_size()

    def values64(self):
        return self.view(self.buf)[:, :self.live, :].double()


def _half_ulp_bf16(x):
    r = x.to(torch.bfloat16).double().abs()
    _, e = torch.frexp(r)
    return torch.where(r > 0, torch.ldexp(torch.ones_like(r), (e - 9).to(torch.int32)), torch.zeros_like(r))


def run_case(form, *, dtype=0, route=None, expect=None, lead_windows=0, c_pad=(0, 0), a_pad_cols=0, seed=0):
    """Runs `form` through bw_test_gemm and checks it; returns (worst err / S, route taken).  route: forced route name
    (None = dispatcher), expect: the route that must run.  lead_windows: operands (except weights and the positional
    embedding) start that many of their own extents into a larger buffer.  c_pad: (extra columns behind ldc, extra rows
    behind c_zstride)."""
    L, lib = _lib()
    f = dict(form)
    M, N, K, Z, tr = f["M"], f["N"], f["K"], f["Z"], bool(f["transposed"])
    gen = torch.Generator(device="cuda").manual_seed(seed)
    op_t = torch.float32 if dtype == 1 else torch.bfloat16
    c_t = torch.float32 if (dtype == 1 or f["out_fp32"]) else torch.bfloat16
    crows, ccols = (N, M) if tr else (M, N)
    f["lda"] += a_pad_cols
    if c_pad != (0, 0):
        f["ldc"] += c_pad[0]
        if Z > 1:
            f["c_zstride"] = (crows + c_pad[1]) * f["ldc"]
        if f["inplace"]:
            f["ldres"], f["res_zstride"] = f["ldc"], f["c_zstride"]

    za = 1 if (Z > 1 and f["a_zstride"] == 0) else Z
    zb = 1 if (Z > 1 and f["b_zstride"] == 0) else Z
    a_rows = max(f["a_rows"], M)
    b_rows = max(f["b_rows"], N)
    a_zs = f["a_zstride"] if za > 1 else a_rows * f["lda"]
    b_zs = f["b_zstride"] if zb > 1 else b_rows * f["ldb"]

    def lead_of(extent):
        return LEAD + lead_windows * extent

    A = Operand(op_t, za, a_rows, K, f["lda"], a_zs, lead=lead_of(za * a_zs), live=M, gen=gen, scale=0.5)
    # the weight operand of swap-AB is A; B (the activations) of the vocabulary projection has b_rows allocated
    B = Operand(op_t, zb, b_rows, K, f["ldb"], b_zs, live=N, gen=gen, scale=0.5)
    c_zs = f["c_zstride"] if Z > 1 else crows * f["ldc"]
    # unwritten = NaN; a full row of guard behind C catches a store one row (one column of a transposed C) too far
    Cop = Operand(c_t, Z, crows, ccols, f["ldc"], c_zs, lead=lead_of(Z * c_zs), values=False, tail=LEAD + f["ldc"])
    bias = None
    if f["bias"]:  # per column of the stored C: N, or M when transposed
        zbias = 1 if (Z > 1 and f["bias_zstride"] == 0) else Z
        bias_zs = f["bias_zstride"] if zbias > 1 else ccols
        bias = Operand(torch.float32, zbias, 1, ccols, ccols, bias_zs, gen=gen)
    if f["inplace"]:
        Cop.view(Cop.buf)[:] = torch.randn((Z, crows, ccols), device="cuda", generator=gen)
        res_view = Cop.view(Cop.buf).double().clone()
        res_ptr = Cop.ptr()
        f["ldres"], f["res_zstride"] = f["ldc"], (c_zs if Z > 1 else 0)
    elif f["residual"]:
        zr = 1 if (Z > 1 and f["res_zstride"] == 0) else Z
        r_zs = f["res_zstride"] if zr > 1 else crows * f["ldres"]
        # a separate residual is the positional embedding (conv2): a weight, not offset like the activations
        R = Operand(torch.float32, zr, crows, ccols, f["ldres"], r_zs, gen=gen)
        res_view, res_ptr = R.values64(), R.ptr()
    before = Cop.buf.clone()

    desc = G.desc_of(f, A=A.ptr(), B=B.ptr(), C_=Cop.ptr(), bias=bias.ptr() if bias else None,
                     residual=res_ptr if f["residual"] else None)
    taken = C.c_int32(-1)
    torch.cuda.synchronize()
    L.check(lib.bw_test_gemm(C.byref(desc), dtype, G.route_code(route) if route else 0, C.byref(taken), None), "bw_test_gemm")
    torch.cuda.synchronize()
    taken = G.route_name(taken.value)
    if expect is not None:
        assert taken == expect, f"route {taken}, expected {expect}"

    # ---- fp64 reference per z-slice ----
    a64, b64 = A.values64(), B.values64()
    worst = 0.0
    out = Cop.view(Cop.buf)
    for z in range(Z):
        a, b = a64[0 if za == 1 else z], b64[0 if zb == 1 else z]
        acc = a @ b.t()  # [M, N]
        S = a.abs() @ b.abs().t()
        if bias is not None:
            bz = bias.values64()[0 if bias.slices == 1 else z, 0]
            acc = acc + (bz[:, None] if tr else bz[None, :])
            S = S + (bz.abs()[:, None] if tr else bz.abs()[None, :])
        if f["gelu"]:
            acc = 0.5 * acc * (1.0 + torch.special.erf(acc / 2.0 ** 0.5))
        if f["residual"]:
            rz = res_view[0 if res_view.shape[0] == 1 else z]
            rz = rz.t() if tr else rz
            acc = acc + rz
            S = S + rz.abs()
        got = out[z].double()
        got = got.t() if tr else got
        err = (got - acc).abs()
        rho = _half_ulp_bf16(acc) if c_t == torch.bfloat16 else torch.zeros_like(acc)
        gamma = GAMMA_SIMT if taken == "simt" else GAMMA_TC
        bad = ~(err <= gamma * S + rho)  # NaN counts as bad
        if bool(bad.any()):
            i, j = [int(v) for v in bad.nonzero()[0]]
            raise AssertionError(f"z {z} [{i}, {j}] of {M}x{N}x{K} on {taken}: got {float(got[i, j])} ref {float(acc[i, j])} "
                                 f"bound {float(gamma * S[i, j] + rho[i, j]):.3e}; {int(bad.sum())} bad elements")
        worst = max(worst, float(((err - rho).clamp_min(0) / S.clamp_min(1e-300)).max()))

    # ---- guards: every element outside the written extent keeps its bits ----
    written = torch.zeros(Cop.buf.numel(), dtype=torch.bool, device="cuda")
    torch.as_strided(written, (Z, crows, ccols), (c_zs, f["ldc"], 1), Cop.lead).fill_(True)
    iv = INT_VIEW[c_t]
    changed = (Cop.buf.view(iv) != before.view(iv)) & ~written
    assert not bool(changed.any()), f"{int(changed.sum())} elements outside C changed (first at flat offset " \
                                    f"{int(changed.nonzero()[0]) - Cop.lead} from C) on {taken}"
    return worst, taken


def _report(kind, name, worst, taken):
    print(f"\n[gemm-layouts] {kind} {name} route {taken}: worst err/S {worst:.3e}")


@pytest.mark.parametrize("model,site,batch,route", G.GPU_DISPATCH_CASES,
                         ids=[f"{m}-{s}-{b}-{r}" for m, s, b, r in G.GPU_DISPATCH_CASES])
def test_call_site_on_dispatched_route(model, site, batch, route):
    form = G.site_form(model, site, batch)
    # the activations of a second encoder sub-batch start `batch` windows into their buffers (engine.cu:130), cross K/V
    # reads window bi of the encoder output and writes slot q of the cross cache (engine.cu:199)
    lead = 1 if site in G.ENCODER_SITES or site == "cross_kv" else 0
    worst, taken = run_case(form, expect=route, lead_windows=lead, seed=zlib.crc32(f"{model}/{site}/{batch}".encode()) % 1000)
    _report("dispatch", f"{model}/{site}/{batch}", worst, taken)


@pytest.mark.parametrize("model,site,batch,route", G.GPU_FORCED_CASES,
                         ids=[f"{m}-{s}-{b}-{r}" for m, s, b, r in G.GPU_FORCED_CASES])
def test_call_site_on_forced_route(model, site, batch, route):
    """Routes the dispatcher does not pick for these rows, with C padded behind ldc and c_zstride (guards there) and A
    padded behind K (NaN columns)."""
    form = G.site_form(model, site, batch)
    worst, taken = run_case(form, route=route, expect=route, c_pad=(8, 3), a_pad_cols=8, seed=7)
    _report("forced", f"{model}/{site}/{batch}", worst, taken)


FP32_FORMS = {
    "conv2": G.site_form("test-tiny", "conv2", 2),
    "cross_kv": G.site_form("test-tiny", "cross_kv", 0),
    "dec_w2": G.site_form("tiny", "dec_w2", 37),
    "enc_w1": G.site_form("test-tiny", "enc_w1", 1),
    # the fp32 mode never swaps A and B: logits [R, n_vocab] with LR_max rows behind the activations
    "vocab": G._form(37, 51865, 384, a_rows=G.LR_MAX, out_fp32=True),
}


@pytest.mark.parametrize("name", sorted(FP32_FORMS))
def test_fp32_validation_mode_forms(name):
    # the fp32 mode keeps every activation in fp32
    worst, taken = run_case(dict(FP32_FORMS[name], out_fp32=1), dtype=1, expect="simt", lead_windows=1, seed=11)
    _report("fp32", name, worst, taken)


# ---- exact epilogue: one-hot B, so acc[i, j] = A[i, k(j)] exactly (zeros add exactly on every split) ----
SWEEP = [0.0, -0.0, 1e-39, -1e-39, 1e-30, -1e-30, 13.5, -13.5, 14.0, -14.0] + [x / 8.0 for x in range(-96, 97)]


def _exact_case(route, transposed):
    ks = int(route[len("splitk"):]) if route.startswith("splitk") else int(route[4:]) if route.startswith("rows") else 1
    K = 64 * ks
    M, N, Z = 300, 320, 2
    gen = torch.Generator(device="cpu").manual_seed(3)
    sweep = torch.tensor(SWEEP, dtype=torch.float32)
    idx = torch.randint(0, len(SWEEP), (1, M, K), generator=gen)
    A = sweep[idx]
    A[0, :, 0] = sweep[torch.arange(M) % len(SWEEP)]  # every sweep value lands in column 0 of some rows
    onehot = torch.zeros((1, N, K))
    kj = (torch.arange(N) * 5) % K
    kj[: N // 2] = 0  # half the columns read column 0 of A
    onehot[0, torch.arange(N), kj] = 1.0
    ncol = M if transposed else N
    bias = torch.stack([((torch.arange(ncol) % 3) - 1).float() * 0.25 * (z + 1) for z in range(Z)])[:, None, :]
    rows, cols = (N, M) if transposed else (M, N)
    res = (0.5 + torch.rand((Z, rows, cols), generator=gen)) * torch.where(torch.rand((Z, rows, cols), generator=gen) < 0.5, -1.0, 1.0)
    if transposed:  # swap-AB: A is the weight side (M rows), B the activations; the sweep stays in the accumulator
        form = G._form(M, N, K, Z=Z, a_zstride=0, b_zstride=0, c_zstride=rows * cols, bias_zstride=ncol,
                       res_zstride=rows * cols, gelu=True, out_fp32=True, transposed=True, bias=True, residual=True)
    else:
        form = G._form(M, N, K, Z=Z, a_zstride=0, b_zstride=0, c_zstride=M * N, bias_zstride=N, res_zstride=M * N,
                       gelu=True, out_fp32=True, bias=True, residual=True)
    vals = {"A": A.cuda(), "B": onehot.cuda(), "bias": bias.cuda(), "res": res.cuda()}
    return form, vals


def _check_exact(form, vals, route, dtype):
    """Epilogue at fp32 precision: |C - ref| <= 2e-6 (|gelu(x)| + |res|) + 1e-7 -- relative to the terms the epilogue
    rounds, not to their sum, which cancels where gelu(x) ~ -res (the GELU approximation and three fp32 roundings)."""
    L, lib = _lib()
    f = dict(form)
    M, N, K, Z, tr = f["M"], f["N"], f["K"], f["Z"], bool(f["transposed"])
    op_t = torch.float32 if dtype == 1 else torch.bfloat16
    A = vals["A"].to(op_t).contiguous()
    B = vals["B"].to(op_t).contiguous()
    bias, res = vals["bias"].contiguous(), vals["res"].contiguous()
    rows, cols = (N, M) if tr else (M, N)
    out = torch.full((Z * rows + 1, cols), float("nan"), device="cuda")[: Z * rows].view(Z, rows, cols)  # + a guard row
    desc = G.desc_of(f, A=A.data_ptr(), B=B.data_ptr(), C_=out.data_ptr(), bias=bias.data_ptr(), residual=res.data_ptr())
    taken = C.c_int32(-1)
    torch.cuda.synchronize()
    L.check(lib.bw_test_gemm(C.byref(desc), dtype, G.route_code(route), C.byref(taken), None), "bw_test_gemm")
    torch.cuda.synchronize()
    assert G.route_name(taken.value) == route
    acc = A[0].double() @ B[0].double().t()  # exact: one product per element
    for z in range(Z):
        x = acc + (bias[z, 0][:, None] if tr else bias[z, 0][None, :]).double()
        g = 0.5 * x * (1.0 + torch.special.erf(x / 2.0 ** 0.5))
        r = res[z].double().t() if tr else res[z].double()
        ref = g + r
        got = out[z].double().t() if tr else out[z].double()
        bad = ~((got - ref).abs() <= 2e-6 * (g.abs() + r.abs()) + 1e-7)
        if bool(bad.any()):
            i, j = [int(v) for v in bad.nonzero()[0]]
            raise AssertionError(f"{route} z {z} [{i}, {j}]: x {float(x[i, j])} bias {float(bias[z, 0, i if tr else j])} got "
                                 f"{float(got[i, j])} ref {float(ref[i, j])}; {int(bad.sum())} bad elements")


@pytest.mark.parametrize("route", G.EXACT_EPILOGUE_ROUTES)
def test_exact_epilogue_bias_gelu_residual(route):
    form, vals = _exact_case(route, False)
    _check_exact(form, vals, route, 0)


@pytest.mark.parametrize("route", ["tile32", "tile64", "tile128", "splitk2", "splitk4", "simt"])
def test_exact_epilogue_transposed(route):
    form, vals = _exact_case(route, True)
    _check_exact(form, vals, route, 0)


def test_exact_epilogue_fp32_mode():
    form, vals = _exact_case("simt", False)
    _check_exact(form, vals, "simt", 1)
