"""GPU suite (-m gpu): parity of the sm_100a path against the oracle, through the C ABI.

Gates (SURVEY.md 8c):
  G1 exact   : QLUT bytes, LUT_Scales, LUT_Biases (fp32 bit patterns)
  G2 exact   : integer bit-plane sums (CBits) and the whole int32 (BitNet) path output
  G3 fp path : max|dC| <= 1e-3 * max|C_ref| (north_star tolerance) -- we hold 2e-5 -- and NMSE <= 1e-8
  G4 sanity  : NMSE <= 5e-4 vs dense dequant matmul (python/t_mac/ops/qgemm.py:277-282)
No test here reads /root/reference."""
import ctypes as C
import glob
import os

import numpy as np
import pytest

import tmac_b200 as tb
import tmac_oracle as T

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

REL_TOL = 1e-3      # north_star: within 1e-3 relative for fp16 activations
TIGHT_TOL = 2e-5    # what the kernel actually achieves (fp32 re-association only)


@pytest.fixture(scope="module")
def lib():
    if not torch.cuda.is_available():
        pytest.fail("-m gpu tests need a CUDA device; libtmac_b200 has no CPU fallback")
    lib = tb.load()
    tb.check(lib.tmac_b200_init(0), "init")
    # one stream for torch's allocations/fills AND the library's launches: the library's own stream is
    # non-blocking, i.e. NOT ordered after work that torch enqueues on the legacy default stream
    st = torch.cuda.Stream()
    torch.cuda.set_stream(st)
    tb.check(lib.tmac_b200_set_stream(st.cuda_stream), "set_stream")
    yield lib
    torch.cuda.synchronize()
    tb.check(lib.tmac_b200_set_stream(None), "set_stream")


def kc(cfg):
    return tb.make_kcfg(cfg.Mout, cfg.K, cfg.bits, cfg.bm, cfg.kfactor, cfg.group_size, cfg.act_group_size, cfg.zero_point, cfg.one_scale)


def run_gpu(lib, cfg, A, S, x, N, device_ptrs=True, use_dispatch=False):
    """preprocessor + qgemm through the C ABI; returns (qlut, ls, lb, C, cbits) as numpy."""
    k = kc(cfg)
    wt = tb.upload_reference_layout(k, A, S)
    nag = cfg.K // cfg.act_group_size
    try:
        if device_ptrs:
            dx = torch.from_numpy(x).cuda()
            dq = torch.zeros((N, cfg.K // 4, 16), dtype=torch.int8, device="cuda")
            dls = torch.zeros((N, nag), dtype=torch.float32, device="cuda")
            dlb = torch.zeros_like(dls)
            dC = torch.zeros((N, cfg.Mout), dtype=torch.float32, device="cuda")
            dcb = torch.zeros((N, cfg.Mout * cfg.bits), dtype=torch.int32, device="cuda")
            if use_dispatch:
                tb.check(lib.tmac_b200_register_kcfg(C.byref(k)), "register")
                tb.check(lib.preprocessor_int8(cfg.Mout * cfg.bits, cfg.K, N, cfg.bits, dx.data_ptr(), dls.data_ptr(), dlb.data_ptr(), dq.data_ptr()), "preprocessor_int8")
                tb.check(lib.qgemm_lut_int8(cfg.Mout * cfg.bits, cfg.K, N, cfg.bits, A.ctypes.data, dq.data_ptr(), S.ctypes.data, dls.data_ptr(), dlb.data_ptr(), dC.data_ptr()), "qgemm_lut_int8")
            else:
                tb.preprocessor(cfg.K, N, cfg.act_group_size, dx, dls, dlb, dq)
                tb.qgemm_lut(wt, N, dq, dls, dlb, dC)
            tb.cbits(wt, N, dq, dcb)
            torch.cuda.synchronize()
            return dq.cpu().numpy(), dls.cpu().numpy(), dlb.cpu().numpy(), dC.cpu().numpy(), dcb.cpu().numpy()
        q = np.zeros((N, cfg.K // 4, 16), np.int8); ls = np.zeros((N, nag), np.float32); lb = np.zeros_like(ls)
        Cout = np.zeros((N, cfg.Mout), np.float32); cb = np.zeros((N, cfg.Mout * cfg.bits), np.int32)
        tb.preprocessor(cfg.K, N, cfg.act_group_size, x, ls, lb, q)
        tb.qgemm_lut(wt, N, q, ls, lb, Cout)
        tb.cbits(wt, N, q, cb)
        return q, ls, lb, Cout, cb
    finally:
        wt.free()


def check_against_oracle(cfg, w, sc, z, x, A, S, got, oracle):
    q, ls, lb, Cout, cb = got
    qo, lso, lbo = oracle.preprocessor(x, cfg.act_group_size)
    assert np.array_equal(q, qo), "G1: QLUT bytes differ"
    assert np.array_equal(ls.view(np.uint32), lso.view(np.uint32)), "G1: LUT_Scales differ"
    assert np.array_equal(lb.view(np.uint32), lbo.view(np.uint32)), "G1: LUT_Biases differ"
    assert np.array_equal(cb, oracle.cbits(cfg, A, qo)), "G2: integer plane sums differ"
    Co = oracle.qgemm(cfg, A, S, qo, lso, lbo)
    if cfg.one_scale and cfg.act_group_size == cfg.K:
        assert np.array_equal(Cout.view(np.uint32), Co.view(np.uint32)), "G2/G3: int32 path must be bit exact"
    else:
        err = np.abs(Cout - Co).max() / max(np.abs(Co).max(), 1e-30)
        assert err <= REL_TOL, "G3: rel err %g" % err
        assert err <= TIGHT_TOL, "G3 (tight): rel err %g" % err
        assert T.nmse(Co, Cout) <= 1e-8
    assert T.nmse(T.dense_reference(w, sc, z, x, cfg), Cout) <= 5e-4, "G4"


GOLDEN = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(os.path.dirname(__file__), "golden", "w*.npz")))


@pytest.mark.parametrize("name", GOLDEN)
def test_golden_fixtures(lib, oracle, golden_dir, name):
    """CUDA path vs outputs of the reference's own kernels (committed fixtures)."""
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    Mout, K, bits, bm, kf, gs, ags, zp, os_ = [int(v) for v in g["cfg"]]
    cfg = T.Config(Mout, K, bits, bm, kf, gs, ags, bool(zp), bool(os_))
    x = g["x"]; N = x.shape[0]
    q, ls, lb, Cout, cb = run_gpu(lib, cfg, np.ascontiguousarray(g["A"]), np.ascontiguousarray(g["S"]), x, N)
    assert np.array_equal(q, g["qlut"])
    assert np.array_equal(ls.view(np.uint32), g["lut_scales"].view(np.uint32))
    assert np.array_equal(lb.view(np.uint32), g["lut_biases"].view(np.uint32))
    assert np.array_equal(cb, g["cbits"])
    if os_:
        assert np.array_equal(Cout.view(np.uint32), g["C"].view(np.uint32))
    else:
        assert np.abs(Cout - g["C"]).max() <= TIGHT_TOL * np.abs(g["C"]).max()


SHAPES = [
    # (Config, N)   Llama-2-7B / BitNet-3B / Qwen2-7B layer shapes at reduced row counts + odd cases
    (T.Config(1024, 4096, 2, zero_point=True), 1),
    (T.Config(512, 4096, 4), 1),
    (T.Config(512, 4096, 4, zero_point=True), 2),
    (T.Config(768, 11008, 2, zero_point=True), 1),
    (T.Config(384, 1024, 3, zero_point=True), 1),
    (T.Config(512, 2048, 1), 1),
    (T.Config(640, 3200, 2, one_scale=True), 1),
    (T.Config(1280, 8640, 2, one_scale=True), 2),
    (T.Config(512, 3584, 4), 1),
    (T.Config(256, 1024, 4, kfactor=8, group_size=32, act_group_size=32), 1),
    (T.Config(320, 1024, 2, bm=320, group_size=64, act_group_size=64, zero_point=True), 1),
    (T.Config(192, 512, 2, bm=128, zero_point=True), 1),  # 192 rows = 1.5 super-blocks: ragged last super-block
    (T.Config(512, 18944, 4), 1),                         # Qwen2-7B down-proj K: 148 chunks per super-block
    (T.Config(1024, 3584, 4, zero_point=True), 3),        # Qwen2-7B hidden size, batch 3
    (T.Config(64, 128, 4), 1),                            # smallest legal tensor: one super-block, one chunk
    (T.Config(128, 96, 2, bm=256, kfactor=8, group_size=32, act_group_size=32), 1),  # K = 96: three 32-wide chunks
]


@pytest.mark.parametrize("cfg,N", SHAPES, ids=lambda v: ("w%d_%dx%d" % (v.bits, v.Mout, v.K)) if isinstance(v, T.Config) else "n%d" % v)
def test_parity_device_pointers(lib, oracle, cfg, N):
    cfg = cfg.resolved()
    w, sc, z, x = T.make_problem(cfg, seed=0, N=N)
    A, S = T.pack_reference_layout(w, sc, z, cfg)
    check_against_oracle(cfg, w, sc, z, x, A, S, run_gpu(lib, cfg, A, S, x, N), oracle)


@pytest.mark.parametrize("cfg", [T.Config(512, 2048, 2, zero_point=True), T.Config(256, 1024, 4), T.Config(640, 3200, 2, one_scale=True)],
                         ids=["w2zp", "w4", "bitnet"])
def test_parity_host_pointers_and_dispatchers(lib, oracle, cfg):
    """The reference's call shape: host buffers, qgemm_lut_int8 / preprocessor_int8 names."""
    cfg = cfg.resolved()
    w, sc, z, x = T.make_problem(cfg, seed=3, N=1)
    A, S = T.pack_reference_layout(w, sc, z, cfg)
    check_against_oracle(cfg, w, sc, z, x, A, S, run_gpu(lib, cfg, A, S, x, 1, device_ptrs=False), oracle)
    check_against_oracle(cfg, w, sc, z, x, A, S, run_gpu(lib, cfg, A, S, x, 1, device_ptrs=True, use_dispatch=True), oracle)


@pytest.mark.parametrize("bits", [1, 2, 3, 4])
def test_general_lut_matches_oracle(lib, oracle, bits):
    """Random, NON-symmetric LUT as in the reference's own verification (python/t_mac/ops/qgemm.py:289):
    exercises the 16-entry lookup path."""
    cfg = T.Config(384 if bits == 3 else 512, 1024, bits, zero_point=(bits % 2 == 0)).resolved()
    w, sc, z, x = T.make_problem(cfg, seed=5)
    A, S = T.pack_reference_layout(w, sc, z, cfg)
    rng = np.random.default_rng(9)
    nag = cfg.K // cfg.act_group_size
    q = rng.integers(-127, 128, size=(1, cfg.K // 4, 16)).astype(np.int8)
    ls = np.abs(rng.standard_normal((1, nag))).astype(np.float32); lb = rng.standard_normal((1, nag)).astype(np.float32)
    wt = tb.upload_reference_layout(kc(cfg), A, S)
    try:
        for dev in (False, True):
            Cout = np.zeros((1, cfg.Mout), np.float32)
            # a device QLUT is only known to be odd-symmetric if OUR preprocessor wrote it; a recycled torch buffer may
            # still carry that mark, so a caller with its own device table states it (include/tmac_b200.h)
            tb.check(lib.tmac_b200_set_lut_mode(1 if dev else 0), "set_lut_mode")
            if dev:
                dq, dls, dlb = torch.from_numpy(q).cuda(), torch.from_numpy(ls).cuda(), torch.from_numpy(lb).cuda()
                dC = torch.zeros((1, cfg.Mout), dtype=torch.float32, device="cuda")
                tb.qgemm_lut(wt, 1, dq, dls, dlb, dC)
                Cout = dC.cpu().numpy()
            else:
                tb.qgemm_lut(wt, 1, q, ls, lb, Cout)
            Co = oracle.qgemm(cfg, A, S, q, ls, lb)
            assert np.abs(Cout - Co).max() <= TIGHT_TOL * np.abs(Co).max()
    finally:
        tb.check(lib.tmac_b200_set_lut_mode(0), "set_lut_mode")
        wt.free()


def test_tile_calls_like_ggml(lib, oracle):
    """ggml's per-tile calls (ggml.c:12662-12691): src0 + w_offset, dst + dst_offset, n = chunk_size0."""
    cfg = T.Config(1024, 2048, 2, bm=128, zero_point=True).resolved()
    w, sc, z, x = T.make_problem(cfg, seed=7)
    A, S = T.pack_reference_layout(w, sc, z, cfg)
    k = kc(cfg)
    tb.check(lib.tmac_b200_register_kcfg(C.byref(k)), "register")
    wt = tb.upload_reference_layout(k, A, S)
    try:
        nag = cfg.K // cfg.act_group_size
        q = np.zeros((1, cfg.K // 4, 16), np.int8); ls = np.zeros((1, nag), np.float32); lb = np.zeros_like(ls)
        lib.ggml_tmac_mul_mat_task_init(x.ctypes.data, q.ctypes.data, ls.ctypes.data, lb.ctypes.data, cfg.Mout, cfg.K, 1, cfg.bits)
        out = np.zeros((1, cfg.Mout), np.float32)
        n_tile = cfg.n_tile_num; chunk0 = cfg.Mout // n_tile
        w_chunk = A.size // n_tile; s_chunk = S.size // n_tile
        for t in range(n_tile):
            lib.ggml_tmac_mul_mat_task_compute(A.ctypes.data + t * w_chunk, S.ctypes.data + 4 * t * s_chunk, q.ctypes.data, ls.ctypes.data,
                                               lb.ctypes.data, out.ctypes.data + 4 * t * chunk0, chunk0, cfg.K, 1, cfg.bits)
        qo, lso, lbo = oracle.preprocessor(x, cfg.act_group_size)
        Co = oracle.qgemm(cfg, A, S, qo, lso, lbo)
        assert np.array_equal(q, qo)
        assert np.abs(out - Co).max() <= TIGHT_TOL * np.abs(Co).max()
    finally:
        wt.free()


def test_ggml_caller_emulation_whole_tensor_and_per_tile(lib, oracle):
    """ggml's T-MAC mul_mat branch (ref:ggml.c:12562-12706) emulated in C++ (tmac_b200_debug_ggml_mul_mat): task_init + one
    task_compute for the whole tensor, and task_init + one task_compute per weight tile from 1 and 4 tile-stealing threads.
    Host buffers throughout.  The LUT written to the host workspace is the oracle's byte for byte; outputs match the oracle; a
    new activation row (same pointers, new bytes) and a caller-made LUT (same pointer, new bytes) are never served stale data."""
    cfg = T.Config(1024, 2048, 2, bm=128, zero_point=True).resolved()
    w, sc, z, x = T.make_problem(cfg, seed=33)
    A, S = T.pack_reference_layout(w, sc, z, cfg)
    k = kc(cfg)
    tb.check(lib.tmac_b200_register_kcfg(C.byref(k)), "register")
    wt = tb.upload_reference_layout(k, A, S)
    try:
        nag = cfg.K // cfg.act_group_size
        wdata = np.zeros(cfg.K * 4 + 2 * nag * 4 + 64, np.uint8)
        tile_rows = cfg.bm // cfg.bits
        for trial, (per_tile, threads) in enumerate(((0, 1), (1, 1), (1, 4), (0, 1))):
            xr = np.ascontiguousarray(x[0] * (1.0 + 0.25 * trial), np.float32)       # new bytes at the same addresses every trial
            dst = np.full(cfg.Mout, 7.0, np.float32)
            tb.check(lib.tmac_b200_debug_ggml_mul_mat(A.ctypes.data, S.ctypes.data, xr.ctypes.data, wdata.ctypes.data, dst.ctypes.data,
                                                      cfg.Mout, cfg.K, cfg.bits, tile_rows, per_tile, threads), "ggml emulation")
            qo, lso, lbo = oracle.preprocessor(xr[None], cfg.act_group_size)
            Co = oracle.qgemm(cfg, A, S, qo, lso, lbo)[0]
            assert np.array_equal(wdata[:cfg.K * 4].view(np.int8).reshape(1, -1, 16), qo), "host QLUT bytes"
            assert np.abs(dst - Co).max() <= TIGHT_TOL * np.abs(Co).max(), (per_tile, threads)
        # a caller-made (non-symmetric) LUT written over the same workspace: compute only, per tile
        rng = np.random.default_rng(8)
        q = rng.integers(-127, 128, size=(1, cfg.K // 4, 16)).astype(np.int8)
        ls = np.abs(rng.standard_normal((1, nag))).astype(np.float32); lb = rng.standard_normal((1, nag)).astype(np.float32)
        wdata[:cfg.K * 4] = q.view(np.uint8).ravel()
        wdata[cfg.K * 4:cfg.K * 4 + nag * 4] = ls.view(np.uint8).ravel()
        wdata[cfg.K * 4 + nag * 4:cfg.K * 4 + 2 * nag * 4] = lb.view(np.uint8).ravel()
        Co = oracle.qgemm(cfg, A, S, q, ls, lb)[0]
        dst = np.zeros(cfg.Mout, np.float32)
        n_tile = cfg.Mout // tile_rows; w_chunk = A.size // n_tile; s_chunk = S.size // n_tile
        base = wdata.ctypes.data
        for t in range(n_tile):
            lib.ggml_tmac_mul_mat_task_compute(A.ctypes.data + t * w_chunk, S.ctypes.data + 4 * t * s_chunk, base, base + cfg.K * 4, base + cfg.K * 4 + nag * 4,
                                               dst.ctypes.data + 4 * t * tile_rows, tile_rows, cfg.K, 1, cfg.bits)
        assert np.abs(dst - Co).max() <= TIGHT_TOL * np.abs(Co).max()
    finally:
        wt.free()


def test_ggml_hook_transform_tensor_i2_blob(lib, oracle):
    """The load-time path of the llama.cpp fork: an I2 tensor blob `permuted weights || fp32 scales`
    (python/t_mac/model_utils.py:271, ggml-tmac.cpp:336-345) goes through ggml_tmac_b200_transform_tensor, then the
    whole-tensor task_init / task_compute calls (the TVM-threadpool branch of ggml.c:12610-12630) with host buffers."""
    cfg = T.Config(768, 1024, 2, bm=128, zero_point=True).resolved()
    w, sc, z, x = T.make_problem(cfg, seed=17)
    A, S = T.pack_reference_layout(w, sc, z, cfg)
    blob = np.concatenate([A.reshape(-1).view(np.uint8), S.view(np.uint8)]).copy()
    k = kc(cfg)
    lib.tmac_b200_clear_kcfg()
    tb.check(lib.tmac_b200_register_kcfg(C.byref(k)), "register")
    extra = tb.TensorExtra()
    h = lib.ggml_tmac_b200_transform_tensor(blob.ctypes.data, cfg.K, cfg.Mout, cfg.bits, C.byref(extra))
    assert h > 0, tb.last_error()
    try:
        assert extra.n_tile_num == cfg.n_tile_num and extra.scales_size == cfg.scales_size
        assert extra.lut_scales_size == cfg.K // cfg.act_group_size and extra.qweights == blob.ctypes.data
        assert lib.ggml_tmac_b200_get_nbytes(cfg.K, cfg.Mout, cfg.bits) == blob.nbytes
        nag = cfg.K // cfg.act_group_size
        q = np.zeros((1, cfg.K // 4, 16), np.int8); ls = np.zeros((1, nag), np.float32); lb = np.zeros_like(ls)
        out = np.zeros((1, cfg.Mout), np.float32)
        lib.ggml_tmac_mul_mat_task_init(x.ctypes.data, q.ctypes.data, ls.ctypes.data, lb.ctypes.data, cfg.Mout, cfg.K, 1, cfg.bits)
        lib.ggml_tmac_mul_mat_task_compute(extra.qweights, extra.scales, q.ctypes.data, ls.ctypes.data, lb.ctypes.data, out.ctypes.data,
                                           cfg.Mout, cfg.K, 1, cfg.bits)
        qo, lso, lbo = oracle.preprocessor(x, cfg.act_group_size)
        Co = oracle.qgemm(cfg, A, S, qo, lso, lbo)
        assert np.array_equal(q, qo) and np.array_equal(ls, lso) and np.array_equal(lb, lbo)
        assert np.abs(out - Co).max() <= TIGHT_TOL * np.abs(Co).max()
    finally:
        lib.tmac_b200_free_weights(h)
        lib.tmac_b200_clear_kcfg()


@pytest.mark.parametrize("name,bits,block,ags", [("q4_0", 4, 32, 32), ("tq1_0", 2, 256, 64), ("tq2_0", 2, 256, 64)])
def test_ggml_block_types_through_the_hook(lib, oracle, golden_dir, name, bits, block, ags):
    """Q4_0 / TQ1_0 / TQ2_0 tensors (golden block bytes from the reference's gguf-py) go through
    ggml_tmac_b200_transform_tensor_typed, then ggml's two phases with per-tile calls on extra->qweights + offset
    (ggml.c:12662-12691); result vs the oracle run on the decoded codes / scales in the reference layout."""
    z = np.load(os.path.join(golden_dir, "ggml_blocks.npz"))
    q, deq, qt = np.ascontiguousarray(z[name + "_bytes"]), z[name + "_dequant"], int(z[name + "_type"])
    rows, K = deq.shape
    cfg = T.Config(rows, K, bits, kfactor=min(16, block // 4), group_size=block, act_group_size=ags).resolved()
    k = kc(cfg)
    tb.check(lib.tmac_b200_register_kcfg(C.byref(k)), "register")
    assert lib.ggml_tmac_b200_can_mul_mat(qt, 1, 1, b"blk.0.attn_q.weight") == 1
    extra = tb.TensorExtra()
    h = lib.ggml_tmac_b200_transform_tensor_typed(q.ctypes.data, qt, K, rows, C.byref(extra))
    tb.check(h, "transform_tensor_typed")
    try:
        w = np.zeros((rows, K), np.uint8); sc = np.zeros((rows, K // block), np.float32)
        assert lib.tmac_b200_debug_decode_ggml(qt, q.ctypes.data, K, rows, w.ctypes.data, sc.ctypes.data) == block
        A, S = T.pack_reference_layout(w, sc, None, cfg)
        assert extra.n_tile_num == cfg.n_tile_num and extra.scales_size == S.size
        got_scales = np.ctypeslib.as_array((C.c_float * S.size).from_address(extra.scales))
        assert np.array_equal(got_scales, S.reshape(-1)), "extra->scales must be in the reference's run-time order"
        x = np.random.default_rng(5).standard_normal((1, K)).astype(np.float16).astype(np.float32)
        nag = K // ags
        ql = np.zeros((1, K // 4, 16), np.int8); ls = np.zeros((1, nag), np.float32); lb = np.zeros_like(ls)
        lib.ggml_tmac_mul_mat_task_init(x.ctypes.data, ql.ctypes.data, ls.ctypes.data, lb.ctypes.data, rows, K, 1, bits)
        out = np.zeros((1, rows), np.float32)
        n_tile = cfg.n_tile_num; chunk0 = rows // n_tile
        w_chunk = A.size // n_tile; s_chunk = S.size // n_tile
        base, sbase = extra.qweights, extra.scales
        for t in range(n_tile):
            lib.ggml_tmac_mul_mat_task_compute(base + t * w_chunk, sbase + 4 * t * s_chunk, ql.ctypes.data, ls.ctypes.data, lb.ctypes.data,
                                               out.ctypes.data + 4 * t * chunk0, chunk0, K, 1, bits)
        qo, lso, lbo = oracle.preprocessor(x, ags)
        assert np.array_equal(ql, qo)
        Co = oracle.qgemm(cfg, A, S, qo, lso, lbo)
        assert np.abs(out - Co).max() <= TIGHT_TOL * np.abs(Co).max()
        dense = x @ deq.T                                        # the reference's dequantised weights
        assert T.nmse(dense, out) <= 5e-4
    finally:
        lib.tmac_b200_free_weights(h)


def test_gptq_checkpoint_tensors_to_gemv(lib, oracle, golden_dir):
    """qweight / scales / qzeros as a GPTQ checkpoint stores them -> tmac_b200_upload_gptq -> GEMV, against the oracle run on
    the reference's own unpack (golden) packed by the reference layout rule."""
    z = np.load(os.path.join(golden_dir, "gptq_unpack.npz"))
    for tag in ("w4_v2", "w2_v1"):
        bits, K, M, gs, v2 = [int(v) for v in z[tag + "_meta"]]
        cfg = T.Config(M, K, bits, group_size=gs, act_group_size=min(64, gs), zero_point=True).resolved()
        qw, qz, sc = (np.ascontiguousarray(z[tag + k]) for k in ("_qweight", "_qzeros", "_scales"))
        k = kc(cfg)
        h = lib.tmac_b200_upload_gptq(C.byref(k), qw.ctypes.data, sc.ctypes.data, qz.ctypes.data, v2)
        tb.check(h, "upload_gptq")
        try:
            w, s, zr = z[tag + "_w"], z[tag + "_s"].astype(np.float32), z[tag + "_z"].astype(np.float32)
            A, S = T.pack_reference_layout(w, s, zr, cfg)
            x = np.random.default_rng(8).standard_normal((1, K)).astype(np.float16).astype(np.float32)
            out = np.zeros((1, M), np.float32)
            tb.check(lib.tmac_b200_gemv(h, 1, tb.F32, x.ctypes.data, out.ctypes.data), "gemv")
            qo, lso, lbo = oracle.preprocessor(x, cfg.act_group_size)
            Co = oracle.qgemm(cfg, A, S, qo, lso, lbo)
            assert np.abs(out - Co).max() <= TIGHT_TOL * np.abs(Co).max(), tag
            assert T.nmse(T.dense_reference(w, s, zr, x, cfg), out) <= 5e-4
        finally:
            lib.tmac_b200_free_weights(h)


def test_fused_gemv_fp16_and_plain_upload(lib, oracle):
    """tmac_b200_gemv (init+compute in one call) with fp16 activations/outputs (the ARM `T`), weights
    uploaded from un-permuted quantised values."""
    cfg = T.Config(512, 2048, 4, zero_point=True).resolved()
    w, sc, z, x = T.make_problem(cfg, seed=4)
    A, S = T.pack_reference_layout(w, sc, z, cfg)
    wt = tb.upload_plain(kc(cfg), w, sc, z)
    try:
        dx = torch.from_numpy(x).cuda().half()
        dC = torch.zeros((1, cfg.Mout), dtype=torch.float16, device="cuda")
        tb.gemv(wt, 1, dx, dC, dtype=tb.F16)
        qo, lso, lbo = oracle.preprocessor(x, cfg.act_group_size)   # x is fp16-representable
        Co = oracle.qgemm(cfg, A, S, qo, lso, lbo)
        got = dC.float().cpu().numpy()
        assert np.abs(got - Co).max() <= REL_TOL * np.abs(Co).max()   # fp16 output rounding ~ 5e-4
        hC = np.zeros((1, cfg.Mout), np.float32)
        tb.gemv(wt, 1, x, hC)                                        # host buffers end to end
        assert np.abs(hC - Co).max() <= TIGHT_TOL * np.abs(Co).max()
    finally:
        wt.free()


@pytest.mark.parametrize("K", [3200, 8640, 96], ids=["k3200", "k8640_half_chunks", "k96"])
def test_fused_gemv_integer_path_row_wide_scale(lib, oracle, K):
    """BitNet grouping (ONE activation group = the whole row, reference tools/run_pipeline.py:409-412): tmac_b200_gemv builds the
    LUT inside the GEMV -- every CTA scans the row for the row-wide scale, the cluster leader forms the bias in the reference's
    summation order -- and must equal the oracle bit for bit (int32 path), for N > 1, fp32 and fp16 activations, and equal the
    two-call form."""
    cfg = T.Config(640, K, 2, kfactor=8 if K % 64 else 16, one_scale=True).resolved()
    N = 3
    w, sc, z, x = T.make_problem(cfg, seed=12, N=N)
    x = x.astype(np.float16).astype(np.float32)            # fp16-representable: the fp16 call sees the same values
    x[1] *= 32.0; x[2, : K // 2] = 0.0                      # rows with different maxima; a row with a zero half
    A, S = T.pack_reference_layout(w, sc, z, cfg)
    wt = tb.upload_plain(kc(cfg), w, sc, z)
    try:
        qo, lso, lbo = oracle.preprocessor(x, cfg.act_group_size)
        Co = oracle.qgemm(cfg, A, S, qo, lso, lbo)
        dx = torch.from_numpy(x).cuda()
        one = torch.zeros((N, cfg.Mout), device="cuda"); two = torch.zeros_like(one)
        tb.gemv(wt, N, dx, one)
        assert tb.last_launch()["batch"] >= 1
        tb.debug_set("fused", 0)
        tb.gemv(wt, N, dx, two)
        tb.debug_set("fused", 1)
        torch.cuda.synchronize()
        assert np.array_equal(one.cpu().numpy().view(np.uint32), Co.view(np.uint32)), "fused integer path must be bit exact"
        assert np.array_equal(two.cpu().numpy().view(np.uint32), Co.view(np.uint32))
        h16 = torch.zeros((N, cfg.Mout), dtype=torch.float16, device="cuda")
        tb.gemv(wt, N, dx.half(), h16, dtype=tb.F16)
        torch.cuda.synchronize()
        assert np.array_equal(h16.cpu().numpy(), Co.astype(np.float16)), "fp16 activations / outputs: same table, one rounding at the store"
        zero = torch.zeros((1, K), device="cuda"); oz = torch.ones((1, cfg.Mout), device="cuda")
        tb.gemv(wt, 1, zero, oz)                            # all-zero row: scale 0 -> table 0 (lut_ctor.cc:124)
        assert float(oz.abs().max()) == 0.0
    finally:
        tb.debug_set("fused", 1)
        wt.free()


@pytest.mark.parametrize("cfg", [T.Config(512, 2048, 2, zero_point=True), T.Config(640, 3200, 2, one_scale=True), T.Config(384, 1024, 4)],
                         ids=["w2zp", "bitnet", "w4"])
def test_gemv_grouped_equals_single_launches(lib, oracle, cfg):
    """tmac_b200_gemv_grouped (q/k/v, gate/up: one launch, shared activation rows, LUT built inside) against the oracle; on the
    integer path also bit-identical to tmac_b200_gemv per tensor (the fp path's K split differs between the two launch shapes)."""
    cfg = cfg.resolved()
    N = 2
    probs = [T.make_problem(cfg, seed=70 + i, N=N) for i in range(3)]
    x = probs[0][3]
    wts = [tb.upload_plain(kc(cfg), w, sc, z) for (w, sc, z, _) in probs]
    try:
        dx = torch.from_numpy(x).cuda()
        outs = [torch.zeros((N, cfg.Mout), device="cuda") for _ in wts]
        single = [torch.zeros((N, cfg.Mout), device="cuda") for _ in wts]
        tb.gemv_grouped(wts, N, dx, outs)
        assert tb.last_launch()["batch"] == 3
        for wt, o in zip(wts, single):
            tb.gemv(wt, N, dx, o)
        torch.cuda.synchronize()
        qo, lso, lbo = oracle.preprocessor(x, cfg.act_group_size)
        for (w, sc, z, _), o, s1 in zip(probs, outs, single):
            A, S = T.pack_reference_layout(w, sc, z, cfg)
            Co = oracle.qgemm(cfg, A, S, qo, lso, lbo)
            got = o.cpu().numpy()
            if cfg.one_scale:                               # integer path: exact whatever the K split of the launch
                assert np.array_equal(got.view(np.uint32), s1.cpu().numpy().view(np.uint32))
                assert np.array_equal(got.view(np.uint32), Co.view(np.uint32))
            else:
                assert np.abs(got - Co).max() <= TIGHT_TOL * np.abs(Co).max()
        with pytest.raises(tb.TMACError):
            tb.gemv_grouped(wts, N, x, outs)               # host activation pointer
    finally:
        for wt in wts:
            wt.free()


def test_full_size_properties(lib, oracle):
    """BASELINE.json full size (W2 g128 zp, 11008 x 4096): size-independent properties + a row sample
    against the oracle.  (a) determinism, (b) linearity in the weight scales: doubling every
    scale and zero doubles C exactly (power-of-two scaling commutes with every rounding),
    (c) 256 sampled rows vs the oracle."""
    cfg = T.Config(11008, 4096, 2, zero_point=True).resolved()
    w, sc, z, x = T.make_problem(cfg, seed=1)
    k = kc(cfg)
    wt = tb.upload_plain(k, w, sc, z)
    wt2 = tb.upload_plain(k, w, (2 * sc).astype(np.float32), (2 * z).astype(np.float32))
    try:
        dx = torch.from_numpy(x).cuda()
        c1 = torch.zeros((1, cfg.Mout), dtype=torch.float32, device="cuda"); c2 = torch.zeros_like(c1); c3 = torch.zeros_like(c1)
        tb.gemv(wt, 1, dx, c1); tb.gemv(wt, 1, dx, c2); tb.gemv(wt2, 1, dx, c3)
        torch.cuda.synchronize()
        assert torch.equal(c1, c2)
        assert torch.equal(2 * c1, c3)
        rows = np.sort(np.random.default_rng(0).choice(cfg.Mout // 128, 2, replace=False))  # two 128-row tiles
        sub = np.concatenate([np.arange(r * 128, (r + 1) * 128) for r in rows])
        cfg_s = T.Config(len(sub), cfg.K, 2, zero_point=True).resolved()
        As, Ss = T.pack_reference_layout(w[sub], sc[sub], z[sub], cfg_s)
        qo, lso, lbo = oracle.preprocessor(x, 64)
        Co = oracle.qgemm(cfg_s, As, Ss, qo, lso, lbo)
        got = c1.cpu().numpy()[:, sub]
        assert np.abs(got - Co).max() <= TIGHT_TOL * np.abs(Co).max()
    finally:
        wt.free(); wt2.free()


@pytest.mark.parametrize("cfg", [T.Config(512, 2048, 2, zero_point=True), T.Config(256, 1024, 4), T.Config(384, 1024, 3, zero_point=True),
                                 T.Config(512, 1024, 1), T.Config(256, 1024, 4, kfactor=8, group_size=32, act_group_size=32)],
                         ids=["w2zp", "w4", "w3zp", "w1", "w4g32"])
def test_fused_gemv_is_bit_identical_to_two_call_path(lib, oracle, cfg):
    """tmac_b200_gemv builds the LUT inside the GEMV (one launch); the tables, LUT scales and biases it uses are
    bit-identical to preprocessor_int8's, so the output equals preprocessor + qgemm_lut exactly."""
    cfg = cfg.resolved()
    w, sc, z, x = T.make_problem(cfg, seed=13, N=2)
    wt = tb.upload_plain(kc(cfg), w, sc, z)
    try:
        dx = torch.from_numpy(x).cuda()
        fused = torch.zeros((2, cfg.Mout), device="cuda")
        tb.gemv(wt, 2, dx, fused)
        nag = cfg.K // cfg.act_group_size
        q = torch.zeros((2, cfg.K // 4, 16), dtype=torch.int8, device="cuda")
        ls = torch.zeros((2, nag), device="cuda"); lb = torch.zeros_like(ls)
        two = torch.zeros((2, cfg.Mout), device="cuda")
        tb.preprocessor(cfg.K, 2, cfg.act_group_size, dx, ls, lb, q)
        tb.qgemm_lut(wt, 2, q, ls, lb, two)
        torch.cuda.synchronize()
        assert torch.equal(fused, two)
        A, S = T.pack_reference_layout(w, sc, z, cfg)
        qo, lso, lbo = oracle.preprocessor(x, cfg.act_group_size)
        Co = oracle.qgemm(cfg, A, S, qo, lso, lbo)
        assert np.abs(fused.cpu().numpy() - Co).max() <= TIGHT_TOL * np.abs(Co).max()
    finally:
        wt.free()


P16_TOL = 5e-4     # fp16-operand tile: operands normalised per token and per row by powers of two, then rounded to fp16 (2^-12
                   # relative each), fp32 accumulation; north_star's bar is 1e-3.  Per element it holds 2.5e-4 of sum_k |x_k||W_mk|
                   # at every dynamic range (tests/test_gpu_numerics.py)


@pytest.mark.parametrize("tile", ["int8", "fp16"])
@pytest.mark.parametrize("cfg,N", [(T.Config(256, 1024, 2, zero_point=True), 64), (T.Config(384, 2048, 2), 130),
                                   (T.Config(256, 4096, 2, zero_point=True), 256), (T.Config(192, 512, 2, bm=128, zero_point=True), 300)],
                         ids=["zp_n64", "sym_n130", "zp_k4096_n256", "ragged_n300"])
def test_prefill_tcgen05_tiles_match_oracle(lib, oracle, cfg, N, tile):
    """N >= 32, W2 g128 act64 on the tensor cores.  int8 tile (tmac_prefill.cuh): the int8 contraction over the LUT is the same
    integer arithmetic as the GEMV -> fp re-association tolerance.  fp16 tile (tmac_prefill16.cuh, default for N >= 64): both
    scales folded into fp16 operands, fp32 accumulation over K -> its own tolerance (5e-4 here, north_star 1e-3)."""
    cfg = cfg.resolved()
    tol = TIGHT_TOL if tile == "int8" else P16_TOL
    tb.debug_set("prefill16", 0 if tile == "int8" else 1)
    w, sc, z, x = T.make_problem(cfg, seed=23, N=N)
    A, S = T.pack_reference_layout(w, sc, z, cfg)
    wt = tb.upload_plain(kc(cfg), w, sc, z)
    try:
        dx = torch.from_numpy(x).cuda()
        nag = cfg.K // cfg.act_group_size
        q = torch.zeros((N, cfg.K // 4, 16), dtype=torch.int8, device="cuda")
        ls = torch.zeros((N, nag), device="cuda"); lb = torch.zeros_like(ls)
        out = torch.zeros((N, cfg.Mout), device="cuda")
        tb.preprocessor(cfg.K, N, cfg.act_group_size, dx, ls, lb, q)
        tb.qgemm_lut(wt, N, q, ls, lb, out)
        ll = tb.last_launch()
        assert ll["batch"] == -N and ll["cluster"] == (1 if tile == "int8" else 16), "expected the %s tile, got %r" % (tile, ll)
        torch.cuda.synchronize()
        qo, lso, lbo = oracle.preprocessor(x, cfg.act_group_size)
        Co = oracle.qgemm(cfg, A, S, qo, lso, lbo)
        got = out.cpu().numpy()
        assert np.abs(got - Co).max() <= tol * np.abs(Co).max()
        out2 = torch.zeros_like(out)
        tb.gemv(wt, N, dx, out2)                       # the one-shot API takes the same tile: bit-identical
        torch.cuda.synchronize()
        assert torch.equal(out, out2)
        tb.debug_set("prefill", 0)                     # tiles disabled: the GEMV kernel per activation row
        out3 = torch.zeros_like(out)
        tb.qgemm_lut(wt, N, q, ls, lb, out3)
        assert tb.last_launch()["batch"] >= 0, "the tile was supposed to be disabled"
        torch.cuda.synchronize()
        g3 = out3.cpu().numpy()
        assert np.abs(g3 - Co).max() <= TIGHT_TOL * np.abs(Co).max()
        assert np.abs(g3 - got).max() <= (tol + TIGHT_TOL) * np.abs(Co).max()
    finally:
        tb.debug_set("prefill", 1); tb.debug_set("prefill16", 1)
        wt.free()


@pytest.mark.parametrize("mode", ["fp16_streamk", "fp16_tile_per_cta", "int8"])
def test_prefill_full_size_llama_shape(lib, oracle, mode):
    """BASELINE config 4 at full size: 11008 x 4096 W2 g128 zp, N = 256 (86 tiles < 148 SMs -> the fp16 tile runs stream-K:
    tiles cut between CTAs, partial tiles summed in ascending K order).  Every row of 8 sampled tokens against the oracle;
    run twice: deterministic, and the stream-K flags are clean for the next launch."""
    cfg = T.Config(11008, 4096, 2, zero_point=True).resolved()
    N = 256
    tb.debug_set("prefill16", 0 if mode == "int8" else 1)
    tb.debug_set("pf_streamk", 1 if mode == "fp16_streamk" else 0)
    w, sc, z, x = T.make_problem(cfg, seed=29, N=N)
    A, S = T.pack_reference_layout(w, sc, z, cfg)
    wt = tb.upload_plain(kc(cfg), w, sc, z)
    try:
        dx = torch.from_numpy(x).cuda()
        out = torch.zeros((N, cfg.Mout), device="cuda"); out2 = torch.zeros_like(out)
        tb.gemv(wt, N, dx, out)
        ll = tb.last_launch()
        assert ll["batch"] == -N
        if mode.startswith("fp16"):
            assert ll["min_blocks"] == {"fp16_streamk": 1, "fp16_tile_per_cta": 0}[mode], ll
        if mode == "fp16_streamk":
            assert ll["grid_x"] == torch.cuda.get_device_properties(0).multi_processor_count
        tb.gemv(wt, N, dx, out2)
        torch.cuda.synchronize()
        assert torch.equal(out, out2)
        toks = [0, 1, 63, 64, 127, 128, 200, 255]
        qo, lso, lbo = oracle.preprocessor(x[toks], cfg.act_group_size)
        Co = oracle.qgemm(cfg, A, S, qo, lso, lbo)
        got = out.cpu().numpy()[toks]
        tol = TIGHT_TOL if mode == "int8" else P16_TOL
        assert np.abs(got - Co).max() <= tol * np.abs(Co).max()
    finally:
        tb.debug_set("prefill16", 1); tb.debug_set("pf_streamk", 0)
        wt.free()


# BASELINE.md 3.4 shapes at FULL size (the launch decomposition depends on Mout / K): every row against the oracle.
LLAMA = [(4096, 4096), (11008, 4096), (4096, 11008)]
QWEN2 = [(3584, 3584), (512, 3584), (18944, 3584), (3584, 18944)]
BITNET = [(3200, 3200), (8640, 3200), (3200, 8640)]
FULL_CASES = ([(m, k, 2, True, False) for m, k in LLAMA] + [(m, k, 4, False, False) for m, k in LLAMA] + [(m, k, 4, True, False) for m, k in LLAMA + QWEN2] +
              [(m, k, 2, False, True) for m, k in BITNET])


@pytest.mark.parametrize("mout,k,bits,zp,one_scale", FULL_CASES,
                         ids=["%dx%d_w%d%s" % (m, k, b, "_bitnet" if o else ("_zp" if z else "_sym")) for m, k, b, z, o in FULL_CASES])
def test_full_size_shapes_every_row(lib, oracle, mout, k, bits, zp, one_scale):
    cfg = T.Config(mout, k, bits, zero_point=zp, one_scale=one_scale).resolved()
    w, sc, z, x = T.make_problem(cfg, seed=7)
    A, S = T.pack_reference_layout(w, sc, z, cfg)
    wt = tb.upload_plain(kc(cfg), w, sc, z)
    try:
        nag = cfg.K // cfg.act_group_size
        dx = torch.from_numpy(x).cuda()
        q = torch.zeros((1, cfg.K // 4, 16), dtype=torch.int8, device="cuda")
        ls = torch.zeros((1, nag), device="cuda"); lb = torch.zeros_like(ls)
        two = torch.zeros((1, cfg.Mout), device="cuda"); one = torch.zeros_like(two)
        tb.preprocessor(cfg.K, 1, cfg.act_group_size, dx, ls, lb, q)
        tb.qgemm_lut(wt, 1, q, ls, lb, two)            # the two reference calls
        tb.gemv(wt, 1, dx, one)                        # the one-call form (fused LUT where the grouping allows)
        torch.cuda.synchronize()
        qo, lso, lbo = oracle.preprocessor(x, cfg.act_group_size)
        Co = oracle.qgemm(cfg, A, S, qo, lso, lbo)
        assert np.array_equal(q.cpu().numpy(), qo)
        for got in (two.cpu().numpy(), one.cpu().numpy()):
            if one_scale:
                assert np.array_equal(got.view(np.uint32), Co.view(np.uint32)), "int32 path must be bit exact"
            else:
                assert np.abs(got - Co).max() <= TIGHT_TOL * np.abs(Co).max()
    finally:
        wt.free()


@pytest.mark.parametrize("pinned", [False, True], ids=["pageable", "page_locked"])
def test_host_call_buffers_in_place(lib, oracle, pinned):
    """tmac_b200_gemv with host buffers (the reference's call shape): page-locked caller buffers are used in place (copy
    source / kernel store target), ordinary memory goes through the staging buffers; repeated calls with NEW activations
    in the same buffers see them."""
    cfg = T.Config(512, 2048, 2, zero_point=True).resolved()
    w, sc, z, x = T.make_problem(cfg, seed=31, N=1)
    A, S = T.pack_reference_layout(w, sc, z, cfg)
    wt = tb.upload_plain(kc(cfg), w, sc, z)
    try:
        hin = torch.zeros((1, cfg.K)); hout = torch.zeros((1, cfg.Mout))
        if pinned:
            hin, hout = hin.pin_memory(), hout.pin_memory()
        for rep in range(3):
            xr = (x * (rep + 1)).astype(np.float32)
            hin.copy_(torch.from_numpy(xr))
            hout.fill_(-1.0)
            tb.gemv(wt, 1, hin, hout)
            qo, lso, lbo = oracle.preprocessor(xr, cfg.act_group_size)
            Co = oracle.qgemm(cfg, A, S, qo, lso, lbo)
            assert np.abs(hout.numpy() - Co).max() <= TIGHT_TOL * np.abs(Co).max(), "rep %d" % rep
    finally:
        wt.free()


def test_grouped_launch_equals_single_launches(lib, oracle):
    """tmac_b200_qgemm_lut_grouped (q/k/v-style fused launch) is bit-identical to per-tensor launches."""
    cfg = T.Config(512, 2048, 2, zero_point=True).resolved()
    wts, outs_single, qs, lss, lbs = [], [], [], [], []
    try:
        for seed in range(3):
            w, sc, z, x = T.make_problem(cfg, seed=40 + seed)
            wts.append(tb.upload_plain(kc(cfg), w, sc, z))
            dx = torch.from_numpy(x).cuda()
            q = torch.zeros((1, cfg.K // 4, 16), dtype=torch.int8, device="cuda")
            ls = torch.zeros((1, cfg.K // cfg.act_group_size), device="cuda"); lb = torch.zeros_like(ls)
            tb.preprocessor(cfg.K, 1, cfg.act_group_size, dx, ls, lb, q)
            o = torch.zeros((1, cfg.Mout), device="cuda")
            tb.qgemm_lut(wts[-1], 1, q, ls, lb, o)
            qs.append(q); lss.append(ls); lbs.append(lb); outs_single.append(o)
        outs = [torch.zeros((1, cfg.Mout), device="cuda") for _ in range(3)]
        tb.qgemm_lut_grouped(wts, 1, qs, lss, lbs, outs)
        torch.cuda.synchronize()
        for a, b in zip(outs, outs_single):
            assert torch.equal(a, b)
    finally:
        for wt in wts:
            wt.free()


def test_errors_follow_reference_convention(lib):
    """0 / -1 return codes (kernels.h:27,37), no exceptions across the C ABI."""
    x = torch.zeros((1, 96), device="cuda")
    assert lib.tmac_b200_preprocessor(96, 1, 64, 0, x.data_ptr(), x.data_ptr(), x.data_ptr(), x.data_ptr()) == -1
    assert lib.qgemm_lut_int8(256, 4096, 1, 2, x.data_ptr(), x.data_ptr(), x.data_ptr(), x.data_ptr(), x.data_ptr(), x.data_ptr()) == -1
    assert b"not a registered" in lib.tmac_b200_last_error()
    assert lib.tmac_b200_qgemm_lut(123456, 0, 1, 1, 0, x.data_ptr(), x.data_ptr(), x.data_ptr(), x.data_ptr()) == -1
