"""GPU suite (-m gpu): every kernel path at the numeric edges, against the oracle, with a PER-ELEMENT error bound.

The parity tests bound max|dC| by a fraction of max|C_ref| over the whole output; one token or weight row whose values are
small next to the rest can be wrong inside that bound.  Here every element is held to the dot-product error bound

    |C - C_ref| <= tol * (|x| @ |W|^T)[n][m]            (W dequantised as in T.dense_reference, fp64)

in addition to the tensor-wide check.  Exact paths (fp32 re-association only) hold TIGHT_TOL; the fp16-operand prefill tile
holds P16_ELEM_TOL.  Inputs: tokens and rows scaled by powers of two across fp32's range (outputs must then scale by exactly
the same power of two, bit for bit), a token whose 128-activation sums pass fp16's 65504, activations whose LUT entries are
all exact round-half-even ties, zero and -0.0 groups, all-zero tokens, and the prefill tiles' shape edges."""
import numpy as np
import pytest

import tmac_b200 as tb
import tmac_oracle as T

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

TIGHT_TOL = 2e-5       # exact paths: fp32 re-association only
P16_TOL = 5e-4         # fp16-operand tile, tensor-wide (as test_gpu_parity.py)
P16_ELEM_TOL = 2.5e-4  # fp16-operand tile, per element: operands rounded to fp16 (2^-12 relative each), fp32 accumulation

CFG = T.Config(256, 1024, 2, zero_point=True).resolved()         # W2 g128 act64 zp: every path, both prefill tiles
BITNET = T.Config(640, 3200, 2, one_scale=True).resolved()       # the integer (int32) path: one activation group per row
FP_PATHS = ["two_call", "fused", "grouped", "int8_tile", "fp16_tile", "seq0", "seq2"]
INT_PATHS = ["two_call", "fused", "grouped"]
TOKEN_K = (-24, -16, -8, 0, 8, 14)
ROW_K = (-20, -12, -8, 0, 6)
WORST = {}


@pytest.fixture(scope="module")
def lib():
    if not torch.cuda.is_available():
        pytest.fail("-m gpu tests need a CUDA device; libtmac_b200 has no CPU fallback")
    lib = tb.load()
    tb.check(lib.tmac_b200_init(0), "init")
    st = torch.cuda.Stream()
    torch.cuda.set_stream(st)
    tb.check(lib.tmac_b200_set_stream(st.cuda_stream), "set_stream")
    yield lib
    torch.cuda.synchronize()
    tb.check(lib.tmac_b200_set_stream(None), "set_stream")
    for k in sorted(WORST):
        print("worst |dC| / elem_bound  %-40s %.3g" % (k, WORST[k]))


def kc(cfg):
    return tb.make_kcfg(cfg.Mout, cfg.K, cfg.bits, cfg.bm, cfg.kfactor, cfg.group_size, cfg.act_group_size, cfg.zero_point, cfg.one_scale)


def elem_bound(w, sc, z, x, cfg):
    """(|x| @ |W|^T) in fp64: the scale of every output element's rounding error."""
    cfg = cfg.resolved()
    wf = w.astype(np.float64) - (1 << (cfg.bits - 1))
    if cfg.one_scale:
        W = wf * float(np.asarray(sc).reshape(-1)[0])
    else:
        gs = cfg.group_size
        W = wf.reshape(cfg.Mout, cfg.K // gs, gs) * np.asarray(sc, np.float64)[:, :, None]
        if cfg.zero_point:
            W = W - np.asarray(z, np.float64)[:, :, None]
        W = W.reshape(cfg.Mout, cfg.K)
    return np.abs(np.asarray(x, np.float64)) @ np.abs(W).T


def oracle_out(oracle, cfg, w, sc, z, x):
    A, S = T.pack_reference_layout(w, sc, z, cfg)
    q, ls, lb = oracle.preprocessor(x, cfg.act_group_size)
    return oracle.qgemm(cfg, A, S, q, ls, lb)


def assert_close(got, ref, eb, path, what, extra=None):
    """Tensor-wide AND per-element check; `extra` is an additional per-element allowance (fp16 output rounding)."""
    tol = P16_ELEM_TOL if path == "fp16_tile" else TIGHT_TOL
    wide = P16_TOL if path == "fp16_tile" else TIGHT_TOL
    got = np.asarray(got, np.float64)
    ref = np.asarray(ref, np.float64)
    d = np.abs(got - ref)
    allow = tol * eb + (0 if extra is None else extra)
    assert np.all(np.isfinite(got)), "%s %s: non-finite outputs at %s" % (path, what, np.argwhere(~np.isfinite(got))[:4].tolist())
    assert d.max() <= (wide + (0 if extra is None else 2.0 ** -11)) * np.abs(ref).max(), "%s %s: tensor-wide" % (path, what)
    bad = ~(d <= allow)
    if bad.any():
        n, m = np.argwhere(bad)[0]
        raise AssertionError("%s %s: %d elements over the element bound; first [%d][%d]: |dC| %.3g, bound %.3g, worst ratio %.3g"
                             % (path, what, bad.sum(), n, m, d[n, m], allow[n, m], (d / np.maximum(eb, 1e-300)).max()))
    r = float((d / np.where(eb > 0, eb, 1.0)).max())
    WORST[path + " " + what.split("[")[0]] = max(WORST.get(path + " " + what.split("[")[0], 0.0), r)


def pad_tokens(x, n_min, seed=99):
    N, K = x.shape
    if N >= n_min:
        return x
    extra = np.random.default_rng(seed).standard_normal((n_min - N, K)).astype(np.float16).astype(np.float32)
    return np.concatenate([x, extra])


def run(path, wts, cfg, x):
    """Outputs [N][Mout] (fp32) of one kernel path for activation rows x (host fp32), on tensor wts[0]."""
    N = x.shape[0]
    xr = pad_tokens(x, 64) if path.endswith("_tile") else x
    Np = xr.shape[0]
    dx = torch.from_numpy(np.ascontiguousarray(xr, np.float32)).cuda()
    out = torch.zeros((Np, cfg.Mout), device="cuda")
    try:
        if path in ("two_call", "fused", "grouped"):
            tb.debug_set("prefill", 0)                      # the GEMV kernels, whatever N
            if path == "two_call":
                nag = cfg.K // cfg.act_group_size
                q = torch.zeros((Np, cfg.K // 4, 16), dtype=torch.int8, device="cuda")
                ls = torch.zeros((Np, nag), device="cuda"); lb = torch.zeros_like(ls)
                tb.preprocessor(cfg.K, Np, cfg.act_group_size, dx, ls, lb, q)
                tb.qgemm_lut(wts[0], Np, q, ls, lb, out)
            elif path == "fused":
                tb.gemv(wts[0], Np, dx, out)
            else:
                tb.gemv_grouped(wts, Np, dx, [out] + [torch.zeros_like(out) for _ in wts[1:]])
        elif path in ("int8_tile", "fp16_tile"):
            tb.debug_set("prefill16", int(path == "fp16_tile"))
            tb.gemv(wts[0], Np, dx, out)
            ll = tb.last_launch()
            assert ll["batch"] == -Np and ll["cluster"] == (16 if path == "fp16_tile" else 1), "expected the %s, got %r" % (path, ll)
        else:
            tb.debug_set("seq_impl", int(path[-1]))         # 0: the stream-K sequence kernel; 2: the resident chain kernel
            seq = tb.Sequence()
            try:
                for n in range(Np):
                    seq.add(wts[0], x=dx[n], out=out[n])
                seq.build(); seq.launch(); seq.status()
                assert (seq.info()["ring_slots"] == -8) == (path == "seq2"), seq.info()
            finally:
                seq.free()
        torch.cuda.synchronize()
        return out.cpu().numpy()[:N]
    finally:
        tb.debug_set("prefill", 1); tb.debug_set("prefill16", 1); tb.debug_set("seq_impl", 2)


def upload(cfg, w, sc, z, grouped=False):
    wt = tb.upload_plain(kc(cfg), w, sc, z)
    return [wt, tb.clone(wt)] if grouped else [wt]


def assert_pow2_equivariant(base, scaled, ks, axis, what):
    """scaled[.., i, ..] == 2^ks[i] * base[.., i, ..] bit for bit, along `axis` (0: tokens, 1: rows)."""
    e = np.asarray(ks).reshape((-1, 1) if axis == 0 else (1, -1))
    want = np.ldexp(base, e).astype(np.float32)
    diff = want.view(np.uint32) != scaled.view(np.uint32)
    if diff.any():
        i = np.argwhere(diff)[0]
        raise AssertionError("%s: not 2^k-equivariant, first at %s: %r vs %r (k = %d)" % (what, i.tolist(), scaled[tuple(i)], want[tuple(i)],
                                                                                         e.reshape(-1)[i[axis]]))


def tokens(cfg, N, seed):
    return np.random.default_rng(seed).standard_normal((N, cfg.K)).astype(np.float16).astype(np.float32)


# ------------------------------------------------------------------------------------------------------------------------
# 1. dynamic range
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg,path", [(CFG, p) for p in FP_PATHS] + [(BITNET, p) for p in INT_PATHS],
                         ids=["fp-%s" % p for p in FP_PATHS] + ["int-%s" % p for p in INT_PATHS])
def test_tokens_scaled_by_powers_of_two(lib, oracle, cfg, path):
    """Token n scaled by 2^k_n, k in TOKEN_K, plus a token with a DC offset (sums of 128 activations > 65504): every element
    within the element bound, and the scaled tokens' outputs exactly 2^k_n times the unscaled ones."""
    w, sc, z, _ = T.make_problem(cfg, seed=101)
    x = tokens(cfg, len(TOKEN_K) + 1, seed=102)
    xs = x.copy()
    for n, k in enumerate(TOKEN_K):
        xs[n] = np.ldexp(x[n], k)
    xs[-1] = x[-1] + 520.0
    assert np.abs(xs[-1].reshape(-1, 128).sum(1)).max() > 65504
    wts = upload(cfg, w, sc, z, grouped=(path == "grouped"))
    try:
        got0, got = run(path, wts, cfg, x), run(path, wts, cfg, xs)
    finally:
        for wt in wts:
            wt.free()
    assert_close(got0, oracle_out(oracle, cfg, w, sc, z, x), elem_bound(w, sc, z, x, cfg), path, "tokens[unscaled]")
    ref = oracle_out(oracle, cfg, w, sc, z, xs)
    if cfg.one_scale:
        assert np.array_equal(got.view(np.uint32), ref.view(np.uint32)), "integer path must be bit exact"
    assert_close(got, ref, elem_bound(w, sc, z, xs, cfg), path, "tokens[2^k, dc]")
    assert_pow2_equivariant(got0[:len(TOKEN_K)], got[:len(TOKEN_K)], TOKEN_K, 0, path)


@pytest.mark.parametrize("path", FP_PATHS)
def test_rows_scaled_by_powers_of_two(lib, oracle, path):
    """Rows' scales and zeros scaled by 2^k, k in ROW_K, 32 rows each: element bound, and those rows' outputs exactly 2^k
    times the unscaled tensor's."""
    cfg = CFG
    w, sc, z, _ = T.make_problem(cfg, seed=111)
    x = tokens(cfg, 4, seed=112)
    ks = np.zeros(cfg.Mout, np.int64)
    for i, k in enumerate(ROW_K):
        ks[40 * i + 3: 40 * i + 35] = k                     # 32 rows, not aligned to the 128-row tiles
    sc2, z2 = np.ldexp(sc, ks[:, None]).astype(np.float32), np.ldexp(z, ks[:, None]).astype(np.float32)
    grouped = path == "grouped"
    wa, wb = upload(cfg, w, sc, z, grouped), upload(cfg, w, sc2, z2, grouped)
    try:
        got0, got = run(path, wa, cfg, x), run(path, wb, cfg, x)
    finally:
        for wt in wa + wb:
            wt.free()
    assert_close(got0, oracle_out(oracle, cfg, w, sc, z, x), elem_bound(w, sc, z, x, cfg), path, "rows[unscaled]")
    assert_close(got, oracle_out(oracle, cfg, w, sc2, z2, x), elem_bound(w, sc2, z2, x, cfg), path, "rows[2^k]")
    assert_pow2_equivariant(got0, got, ks, 1, path)


def test_fp16_activations_scaled_by_powers_of_two(lib, oracle):
    """fp16 activation rows scaled by 2^k while they stay fp16-normal: the preprocessor's QLUT, LUT_Scales and LUT_Biases
    equal the oracle's on the same values byte for byte, and qgemm_lut on them holds the element bound."""
    cfg = CFG
    ks = (-12, -8, 0, 8)
    x = tokens(cfg, len(ks), seed=121)
    x = (np.sign(x) * (np.abs(x) + 0.25)).astype(np.float16).astype(np.float32)    # |x| >= 0.25: x * 2^-12 is still normal
    xs = np.stack([np.ldexp(x[n], k) for n, k in enumerate(ks)]).astype(np.float32)
    assert np.array_equal(xs.astype(np.float16).astype(np.float32), xs)
    N, nag = xs.shape[0], cfg.K // cfg.act_group_size
    dx = torch.from_numpy(xs).cuda().half()
    q = torch.zeros((N, cfg.K // 4, 16), dtype=torch.int8, device="cuda")
    ls = torch.zeros((N, nag), device="cuda"); lb = torch.zeros_like(ls)
    w, sc, z, _ = T.make_problem(cfg, seed=122)
    wt = tb.upload_plain(kc(cfg), w, sc, z)
    try:
        out = torch.zeros((N, cfg.Mout), device="cuda")
        tb.preprocessor(cfg.K, N, cfg.act_group_size, dx, ls, lb, q, dtype=tb.F16)
        tb.qgemm_lut(wt, N, q, ls, lb, out)
        torch.cuda.synchronize()
    finally:
        wt.free()
    qo, lso, lbo = oracle.preprocessor(xs, cfg.act_group_size)
    assert np.array_equal(q.cpu().numpy(), qo)
    assert np.array_equal(ls.cpu().numpy().view(np.uint32), lso.view(np.uint32))
    assert np.array_equal(lb.cpu().numpy().view(np.uint32), lbo.view(np.uint32))
    assert_close(out.cpu().numpy(), oracle_out(oracle, cfg, w, sc, z, xs), elem_bound(w, sc, z, xs, cfg), "two_call", "fp16 in[2^k]")


# ------------------------------------------------------------------------------------------------------------------------
# 2. round-half-even ties in every LUT builder
# ------------------------------------------------------------------------------------------------------------------------
def tie_tokens(K, N, ags, seed):
    """Dyadic activations whose every LUT entry times ts is an exact .5 tie.  In each activation group one K-group is
    (15.875,)*4: abs-sum 63.5, lut_scale 0.5, ts 2, all exact.  Every other K-group is (i + 0.25, j1, j2, j3) with small
    integers, so every entry i + 0.25 +- j1 +- j2 +- j3 times 2 ends in .5."""
    rng = np.random.default_rng(seed)
    x = rng.integers(-4, 5, size=(N, K // 4, 4)).astype(np.float32)
    x[:, :, 0] += 0.25
    per = ags // 4
    for n in range(N):
        for g in range(K // ags):
            x[n, g * per + (n + 3 * g) % per] = 15.875
    return x.reshape(N, K)


@pytest.mark.parametrize("dtype", ["f32", "f16"])
def test_preprocessor_ties_round_half_even(lib, oracle, dtype):
    cfg = CFG
    x = tie_tokens(cfg.K, 3, cfg.act_group_size, seed=131)
    N, nag = x.shape[0], cfg.K // cfg.act_group_size
    dx = torch.from_numpy(x).cuda()
    if dtype == "f16":
        dx = dx.half()
    q = torch.zeros((N, cfg.K // 4, 16), dtype=torch.int8, device="cuda")
    ls = torch.zeros((N, nag), device="cuda"); lb = torch.zeros_like(ls)
    tb.preprocessor(cfg.K, N, cfg.act_group_size, dx, ls, lb, q, dtype=tb.F16 if dtype == "f16" else tb.F32)
    torch.cuda.synchronize()
    qo, lso, lbo = oracle.preprocessor(x, cfg.act_group_size)
    assert np.all(lso == 0.5)
    assert np.array_equal(q.cpu().numpy(), qo), "QLUT bytes differ on round-half-even ties"
    assert np.array_equal(ls.cpu().numpy().view(np.uint32), lso.view(np.uint32))
    assert np.array_equal(lb.cpu().numpy().view(np.uint32), lbo.view(np.uint32))


@pytest.mark.parametrize("cfg,path", [(CFG, p) for p in ("fused", "grouped", "seq0", "seq2")] + [(BITNET, "fused")],
                         ids=["fp-fused", "fp-grouped", "fp-seq0", "fp-seq2", "int-fused"])
def test_lut_builders_round_ties_to_even(lib, oracle, cfg, path):
    """The LUT builders inside the fused GEMV (fp and integer), the grouped GEMV, the chain and the sequence kernel: on
    all-tie activations the output equals the oracle within TIGHT_TOL of the element bound (one tie rounded away from
    even per group is ~1e-3 there); the integer path bit for bit."""
    w, sc, z, _ = T.make_problem(cfg, seed=141)
    x = tie_tokens(cfg.K, 3, cfg.act_group_size, seed=142)
    wts = upload(cfg, w, sc, z, grouped=(path == "grouped"))
    try:
        got = run(path, wts, cfg, x)
    finally:
        for wt in wts:
            wt.free()
    ref = oracle_out(oracle, cfg, w, sc, z, x)
    if cfg.one_scale:
        assert np.array_equal(got.view(np.uint32), ref.view(np.uint32)), "integer path must be bit exact"
    assert_close(got, ref, elem_bound(w, sc, z, x, cfg), path, "ties")


# ------------------------------------------------------------------------------------------------------------------------
# 3. zero groups and all-zero tokens
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", FP_PATHS)
def test_zero_groups_and_zero_tokens(lib, oracle, path):
    """Token 0: an all-zero activation group mid-row; token 1: a -0.0 group; tokens 2 and 4: all zero (padding inside a
    batch, their outputs must be exactly 0); token 3 ordinary."""
    cfg = CFG
    w, sc, z, _ = T.make_problem(cfg, seed=151)
    x = tokens(cfg, 5, seed=152)
    x[0, 5 * 64:6 * 64] = 0.0
    x[1, 7 * 64:8 * 64] = -0.0
    x[2] = 0.0
    x[4] = -0.0
    wts = upload(cfg, w, sc, z, grouped=(path == "grouped"))
    try:
        got = run(path, wts, cfg, x)
    finally:
        for wt in wts:
            wt.free()
    assert np.all(got[[2, 4]] == 0.0)
    assert_close(got, oracle_out(oracle, cfg, w, sc, z, x), elem_bound(w, sc, z, x, cfg), path, "zero groups")


# ------------------------------------------------------------------------------------------------------------------------
# 4. prefill shape edges
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [31, 32, 33, 63, 64, 65, 255, 256, 257, 513])
def test_prefill_token_counts(lib, oracle, N):
    """The dispatch thresholds (GEMV < 32 <= int8 tile < 64 <= fp16 tile) and the 128/256-token tile tails; from N = 64 on
    the int8 tile is forced as well."""
    cfg = CFG
    w, sc, z, _ = T.make_problem(cfg, seed=161)
    x = tokens(cfg, N, seed=162)
    x[N // 2] = 0.0
    wt = tb.upload_plain(kc(cfg), w, sc, z)
    dx = torch.from_numpy(x).cuda()
    ref, eb = oracle_out(oracle, cfg, w, sc, z, x), elem_bound(w, sc, z, x, cfg)
    try:
        for forced in ([None, 0] if N >= 64 else [None]):
            if forced is not None:
                tb.debug_set("prefill16", forced)
            out = torch.zeros((N, cfg.Mout), device="cuda")
            tb.gemv(wt, N, dx, out)
            ll = tb.last_launch()
            torch.cuda.synchronize()
            tb.debug_set("prefill16", 1)
            path = "gemv" if N < 32 else ("int8_tile" if N < 64 or forced == 0 else "fp16_tile")
            if path == "gemv":
                assert ll["batch"] >= 0, ll
            else:
                assert ll["batch"] == -N and ll["cluster"] == (16 if path == "fp16_tile" else 1), ll
            assert_close(out.cpu().numpy(), ref, eb, path, "N=%d" % N)
    finally:
        tb.debug_set("prefill16", 1)
        wt.free()


@pytest.mark.parametrize("mout,k,tile", [(4096, 11008, "fp16_tile"), (4096, 11008, "int8_tile"), (512, 4224, "fp16_tile"),
                                         (512, 4224, "int8_tile")], ids=["4096x11008-fp16", "4096x11008-int8", "512x4224-fp16", "512x4224-int8"])
def test_prefill_long_k(lib, oracle, mout, k, tile):
    """K = 11008 (the Llama down-projection: 86 weight groups = 3 bias steps of the fp16 tile, the last one partial) and
    K = 4224 (33 groups) at N = 256; 8 sampled tokens against the oracle."""
    cfg = T.Config(mout, k, 2, zero_point=True).resolved()
    N = 256
    w, sc, z, _ = T.make_problem(cfg, seed=171)
    x = tokens(cfg, N, seed=172)
    wt = tb.upload_plain(kc(cfg), w, sc, z)
    try:
        got = run(tile, [wt], cfg, x)
    finally:
        wt.free()
    toks = [0, 1, 63, 64, 127, 128, 200, 255]
    xt = x[toks]
    assert_close(got[toks], oracle_out(oracle, cfg, w, sc, z, xt), elem_bound(w, sc, z, xt, cfg), tile, "K=%d" % k)


def test_prefill16_stream_k_many_cuts(lib, oracle):
    """pf_streamk = 1 on 1280 x 4096 at N = 256: 10 tiles over all SMs, every tile cut among ~15 CTAs whose partial tiles
    the finisher adds in K order.  Deterministic, and 16 sampled tokens within the element bound."""
    cfg = T.Config(1280, 4096, 2, zero_point=True).resolved()
    N = 256
    w, sc, z, _ = T.make_problem(cfg, seed=181)
    x = tokens(cfg, N, seed=182)
    wt = tb.upload_plain(kc(cfg), w, sc, z)
    tb.debug_set("pf_streamk", 1)
    try:
        dx = torch.from_numpy(x).cuda()
        out, out2 = torch.zeros((N, cfg.Mout), device="cuda"), torch.zeros((N, cfg.Mout), device="cuda")
        tb.gemv(wt, N, dx, out)
        ll = tb.last_launch()
        tb.gemv(wt, N, dx, out2)
        torch.cuda.synchronize()
    finally:
        tb.debug_set("pf_streamk", 0)
        wt.free()
    assert ll["batch"] == -N and ll["cluster"] == 16 and ll["min_blocks"] == 1, ll
    assert ll["grid_x"] == torch.cuda.get_device_properties(0).multi_processor_count
    assert torch.equal(out, out2)
    toks = list(range(0, N, 17))
    xt = x[toks]
    assert_close(out.cpu().numpy()[toks], oracle_out(oracle, cfg, w, sc, z, xt), elem_bound(w, sc, z, xt, cfg), "fp16_tile", "stream-K")


@pytest.mark.parametrize("tile", ["int8_tile", "fp16_tile"])
@pytest.mark.parametrize("N", [96, 300])
def test_prefill_fp16_activations_and_outputs(lib, oracle, tile, N):
    """fp16 activations in, fp16 outputs out, through tb.gemv on both tiles: the element bound plus the output's own
    rounding (half an fp16 ulp of C)."""
    cfg = CFG
    w, sc, z, _ = T.make_problem(cfg, seed=191)
    x = tokens(cfg, N, seed=192)                           # fp16-representable: the oracle sees the same values
    wt = tb.upload_plain(kc(cfg), w, sc, z)
    tb.debug_set("prefill16", int(tile == "fp16_tile"))
    try:
        out = torch.zeros((N, cfg.Mout), dtype=torch.float16, device="cuda")
        tb.gemv(wt, N, torch.from_numpy(x).cuda().half(), out, dtype=tb.F16)
        ll = tb.last_launch()
        torch.cuda.synchronize()
    finally:
        tb.debug_set("prefill16", 1)
        wt.free()
    assert ll["batch"] == -N and ll["cluster"] == (16 if tile == "fp16_tile" else 1), ll
    ref = oracle_out(oracle, cfg, w, sc, z, x)
    assert_close(out.float().cpu().numpy(), ref, elem_bound(w, sc, z, x, cfg), tile, "fp16 io N=%d" % N,
                 extra=2.0 ** -11 * np.abs(ref.astype(np.float64)) + 2.0 ** -25)
