#!/usr/bin/env python
"""bench.py -- the hot path's headline benchmark (contract: see the task statement).

Metric (BASELINE.json): W2A16 GEMV achieved HBM GB/s on the Llama-2-7B layer shape
out=11008, K=4096, batch=1, W2 g128 zero-point, act_group_size 64.

A *step* is one pass of the hot path (preprocessor + qgemm_lut, both through the C ABI) over one
batch of synthetic input: LAYERS distinct weight tensors of that shape (LAYERS x 12.7 MB = 407 MB,
more than 3x the 126 MB L2, so every weight byte streams from HBM; that is the L2 policy: inputs
larger than L2), each with its own activation row.  The step is captured once in a CUDA graph and
replayed; time is CUDA events on the launching stream, max over ranks.

  value     = algorithmic bytes of all ranks / step time, inputs resident in HBM          [GB/s]
              (step = the faster of: one tmac_b200_gemv launch per layer in a CUDA graph, or the
              decode sequence -- the layers as a DEPENDENT chain in one persistent launch;
              roofline.submission says which)
  roofline  = the dominant kernel of that step: algorithmic bytes per launch / its average
              duration vs the measured HBM peak in MEASURED_PEAKS.json (chain_kernel: one launch =
              all layers; the gemv3 launch-chain figures are kept beside it)
  e2e       = the same metric through the reference-facing call tmac_b200_gemv with HOST
              activations/outputs (H2D + kernel + result into page-locked memory + sync per GEMV
              inside the timed region); e2e.sequence_step = the decode-loop form (host input row ->
              one persistent launch -> all outputs to host)
  cpu_baseline = the reference's own AVX2 kernels (oracle/_ref, built from /root/reference) on the
              box's host cores, bounded sample of the same workload
  --impl reference : that CPU arm alone, same metric / config.

Inputs are seeded: the same arguments give the same weights and activations in every run.
--dump-outputs DIR writes what the step computed in its last run as float32 .npy files, so that
two builds can be compared output for output:
  launch_chain.npy             [LAYERS][out]  one tmac_b200_gemv per layer, layer i on its own row x[i]
  sequence_dependent_chain.npy [LAYERS][out]  the decode sequence (x[i+1] = first K outputs of layer i)
(with N > 1 ranks: [ranks][LAYERS][out], the gathered outputs as rank 0 holds them)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "t-mac_b200"))

METRIC = "w2a16_gemv_hbm_gbps"
UNIT = "GB/s"
MOUT, K, BITS, GS, AGS, ZP = 11008, 4096, 2, 128, 64, True
LAYERS = 32
PREFETCH_NEXT = os.environ.get("TMAC_BENCH_PREFETCH", "1") != "0"


def algorithmic_bytes(mout=MOUT, k=K, bits=BITS, gs=GS, zp=ZP, act_bytes=4, out_bytes=4, scale_bytes=2):
    """SURVEY.md 8d / DESIGN.md: packed indices + scales(+zeros) + activations + outputs, each byte once."""
    return mout * k * bits // 8 + mout * (k // gs) * scale_bytes * (2 if zp else 1) + k * act_bytes + mout * out_bytes


def synth(seed, mout=MOUT, k=K, bits=BITS, gs=GS, zp=ZP, one_scale=False):
    rng = np.random.default_rng(seed)
    if one_scale:
        w = (rng.integers(-1, 2, size=(mout, k)) + 2).astype(np.uint8)
        return w, np.array([0.037], np.float16).astype(np.float32), None
    w = rng.integers(0, 1 << bits, size=(mout, k), dtype=np.uint8)
    sc = (np.abs(rng.standard_normal((mout, k // gs))) * 0.01 + 1e-4).astype(np.float16).astype(np.float32)
    # zero points centred on the middle of the code range plus noise: (w - 2^(bits-1)) * s - z is then zero-mean, so the dependent
    # chain of the bench (x[i+1] = first K outputs of GEMV i, 32 deep) neither overflows fp32 nor underflows (with z ~ N(0, 0.01)
    # alone the mean entry gives the 4096x4096 block a spectral radius of 16.6: 1e37 at layer 31, inf in some runs)
    z = (-0.5 * sc + rng.standard_normal((mout, k // gs)) * 0.001).astype(np.float16).astype(np.float32) if zp else None
    return w, sc, z


def activations(seed, rows=LAYERS, k=K):
    """Seeded fp16-representable activation rows, one per layer."""
    return np.random.default_rng(seed).standard_normal((rows, k)).astype(np.float16).astype(np.float32)


def dump_outputs(dirname, arrays):
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), np.ascontiguousarray(a, np.float32))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                    if r[col].lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own kernels on the host cores (oracle/_ref), or the oracle port.
# ------------------------------------------------------------------------------------------------
def cpu_arm(budget_s, nbuf=4):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import tmac_oracle as T   # the one place bench.py executes oracle/: as the measured CPU baseline
    ref = T.load_ref()
    cfg = T.Config(MOUT, K, BITS, group_size=GS, act_group_size=AGS, zero_point=ZP).resolved()
    cores = os.cpu_count() or 1
    w, sc, z = synth(0)
    A, S = T.pack_reference_layout(w, sc, z, cfg)
    x = np.random.default_rng(1).standard_normal((1, K)).astype(np.float16).astype(np.float32)
    if ref is not None:
        kind, lib = "reference", ref
        bufs = [(A.copy(), S.copy()) for _ in range(nbuf)]   # distinct buffers: weights stream from DRAM, not L2/L3

        def one(i):
            a, s = bufs[i % nbuf]
            ref.gemv_mt(cfg, a, s, x)
        # threads = cores is the reference's guidance (docs/codegen.md:86); on many-core hosts the tile
        # work-stealing stops scaling earlier, so probe a few pool sizes and keep the fastest.
        best, best_t, by_threads = cores, None, {}
        for nt in sorted({1, 4, 8, 16, 32, 64, cores}):
            if nt > cores:
                continue
            ref.set_threads(nt)
            for i in range(3):
                one(i)
            t = None
            for _rep in range(3):                       # best of 3 batches: thread-pool wake-up noise is large on busy hosts
                t0 = time.perf_counter()
                for i in range(20):
                    one(i)
                dt = time.perf_counter() - t0
                t = dt if t is None else min(t, dt)
            by_threads[str(nt)] = round(algorithmic_bytes() / (t / 20) / 1e9, 2)      # GB/s with nt threads (20 GEMVs)
            if best_t is None or t < best_t:
                best, best_t = nt, t
        cores = best
        ref.set_threads(cores)
    else:
        kind, lib, cores, by_threads = "port", T.load_oracle(), 1, {}

        def one(i):
            q, ls, lb = lib.preprocessor(x, AGS)
            lib.qgemm(cfg, A, S, q, ls, lb)
    for i in range(3):
        one(i)
    t0 = time.perf_counter(); n = 0
    while True:
        one(n); n += 1
        el = time.perf_counter() - t0
        if el > budget_s:
            break
    per = el / n
    gbps = algorithmic_bytes() / per / 1e9
    return {"value": gbps, "unit": UNIT, "cores": cores, "kind": kind, "ms_per_gemv": per * 1e3, "GBps_by_threads": by_threads,
            "sample": "%d GEMVs %dx%d W2 g128 zp over %d distinct weight buffers, preprocessor included, %.1f s" % (n, MOUT, K, nbuf, el)}


def parity_check(w, sc, z, xs, out_chain, out_seq, layers_checked=(0, LAYERS // 2, LAYERS - 1)):
    """BASELINE.md 3.6: the numbers above come from outputs that match the CPU reference (oracle/_ref when built, else the
    oracle port) -- used here as the CHECKER only.  Launch chain: layer i with its own input x[i].  Sequence kernel
    (dependent chain): layer i with the GPU's own previous output as input.  All rows, tolerance 1e-3 of max|C| (north_star)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import tmac_oracle as T
    lib = T.load_ref() or T.load_oracle()
    cfg = T.Config(MOUT, K, BITS, group_size=GS, act_group_size=AGS, zero_point=ZP).resolved()
    A, S = T.pack_reference_layout(w, sc, z, cfg)

    def ref(xrow):
        q, ls, lb = lib.preprocessor(xrow[None], AGS)
        return lib.qgemm(cfg, A, S, q, ls, lb)[0]
    worst = {}
    for i in layers_checked:
        r = ref(xs[i])
        e = float(np.abs(out_chain[i] - r).max() / np.abs(r).max())
        worst["launch_chain"] = max(worst.get("launch_chain", 0.0), e)
        assert e <= 1e-3, "launch chain layer %d: rel err %.3g" % (i, e)
        if out_seq is not None:
            xin = xs[0] if i == 0 else out_seq[i - 1][:K]
            r = ref(xin)
            e = float(np.abs(out_seq[i] - r).max() / np.abs(r).max())
            worst["sequence_dependent_chain"] = max(worst.get("sequence_dependent_chain", 0.0), e)
            assert e <= 1e-3, "sequence kernel layer %d: rel err %.3g" % (i, e)
    return {"checker": lib.kind, "layers": list(layers_checked), "rows": MOUT, "max_rel_err": worst, "tolerance": 1e-3}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    per_step_budget = max(0.5, min(10.0, 60.0 / max(1, args.steps + args.warmup)))
    for _ in range(args.warmup):
        cpu_arm(per_step_budget * 0.25)
    vals = [cpu_arm(per_step_budget) for _ in range(max(1, args.steps))]
    v = float(np.mean([r["value"] for r in vals]))
    cb = dict(vals[-1]); cb["value"] = v
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": float(np.mean([r["ms_per_gemv"] for r in vals])) * LAYERS, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int8 LUT / fp32 accumulate", "data": "synthetic",
            "config": workload_config(args.gpus), "cpu_baseline": cb,
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def workload_config(gpus):
    return {"workload": "Llama-2-7B ffn up/gate shape W2A16 GEMV: out=%d K=%d batch=1, W2 g128 zero-point, act_group 64, "
                        "%d distinct layers per step per GPU" % (MOUT, K, LAYERS),
            "layers_per_step": LAYERS, "l2_policy": "inputs larger than L2 (%.0f MB of weights per step per GPU)" % (LAYERS * algorithmic_bytes() / 1e6),
            "parallelism": ("%d ranks x %d rows per layer; the all-gather of every layer's output is fused into the GEMV epilogue "
                            "(peer stores over NVLink, no collective launch)" % (gpus, MOUT)) if gpus > 1 else "single GPU"}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-extras", action="store_true", help="skip tokens/s extras and the CPU baseline")
    ap.add_argument("--eager", action="store_true", help="no CUDA graph (for ncu kernel-level profiling)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the step's last run to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU step's outputs; --impl reference has none")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import tmac_b200 as tb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback in the product path)")
    torch.manual_seed(rank)                     # the inputs of the extras
    torch.cuda.set_device(local)
    dist = None
    force_sharded = os.environ.get("TMAC_BENCH_FORCE_SHARDED", "0") == "1"      # validate the N > 1 extras on one rank
    if world > 1 or force_sharded:
        import torch.distributed as dist
        if world == 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1"); os.environ.setdefault("MASTER_PORT", "29577")
            os.environ.setdefault("RANK", "0"); os.environ.setdefault("WORLD_SIZE", "1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = tb.load()
    tb.check(lib.tmac_b200_init(local), "init")
    stream = torch.cuda.Stream()
    tb.check(lib.tmac_b200_set_stream(stream.cuda_stream), "set_stream")
    launches = {"n": 0}

    # ---- workload: LAYERS distinct resident tensors (one host encode, LAYERS-1 device clones) ----
    w, sc, z = synth(100 + rank)
    cfg = tb.make_kcfg(MOUT, K, BITS, 128, 16, GS, AGS, ZP, False)
    base = tb.upload_plain(cfg, w, sc, z)
    layers = [base] + [tb.clone(base) for _ in range(LAYERS - 1)]
    nag = K // AGS
    with torch.cuda.stream(stream):
        x = torch.from_numpy(activations(200 + rank)).cuda()
        qlut = torch.zeros((LAYERS, K // 4, 16), dtype=torch.int8, device="cuda")
        ls = torch.zeros((LAYERS, nag), device="cuda"); lb = torch.zeros_like(ls)
        out = torch.zeros((LAYERS, MOUT), device="cuda")
        gathered, sv, nccl_gathered = None, None, None
    if world > 1:
        # the step's all-gather is fused into the GEMV epilogues: every rank's [world][LAYERS][MOUT] buffer is mapped by every
        # other rank (cudaIpc) and each launch stores its finished rows into all of them over NVLink (tmac_b200_peer_outputs)
        sv = tb.SharedVector(world * LAYERS * MOUT, dist, rank, world)
        gathered = sv.local.view(world, LAYERS, MOUT)
        out = gathered[rank]
        with torch.cuda.stream(stream):
            nccl_gathered = torch.zeros((world, LAYERS, MOUT), device="cuda")

    def fused_step_calls(_unused=True):
        for i, wt in enumerate(layers):           # the reference-facing plugin call: init + compute in one (fused LUT build)
            if PREFETCH_NEXT:
                lib.tmac_b200_hint_next_weights(layers[(i + 1) % LAYERS].handle)
            if sv is not None:
                tb.peer_outputs([sv.peer_ptr(q) + 4 * (rank * LAYERS + i) * MOUT for q in range(world) if q != rank])
            tb.gemv(wt, 1, x[i], out[i])
        if sv is not None:
            sv.barrier()                          # one flag exchange per step: every rank's rows of this step are in place everywhere

    def step_calls(with_pre=True):
        for i, wt in enumerate(layers):
            if with_pre:
                tb.preprocessor(K, 1, AGS, x[i], ls[i], lb[i], qlut[i])
            if PREFETCH_NEXT:
                lib.tmac_b200_hint_next_weights(layers[(i + 1) % LAYERS].handle)
            tb.qgemm_lut(wt, 1, qlut[i], ls[i], lb[i], out[i])

    def capture(with_pre, fn=None):
        fn = fn or step_calls
        fn(with_pre)                             # eager warm-up allocates every workspace
        tb.check(lib.tmac_b200_sync(), "sync")
        if args.eager:
            return ("eager", fn, with_pre)
        tb.check(lib.tmac_b200_graph_begin(), "graph_begin")
        fn(with_pre)
        g = lib.tmac_b200_graph_end()
        tb.check(g, "graph_end")
        return g

    g_two = capture(True)                        # two-call path: preprocessor_int8 + qgemm_lut_int8 style
    g_gemv = capture(False)                      # qgemm_lut launches only (dominant kernel)
    lone_cfg = tb.last_launch()
    g_step = capture(True, fused_step_calls)     # one call per layer (tmac_b200_gemv, LUT built inside the GEMV)

    def grouped_calls():
        tb.qgemm_lut_grouped(layers, 1, [qlut[i] for i in range(LAYERS)], [ls[i] for i in range(LAYERS)],
                             [lb[i] for i in range(LAYERS)], [out[i] for i in range(LAYERS)])
    g_grouped = None
    if not args.eager:
        grouped_calls(); tb.check(lib.tmac_b200_sync(), "sync")
        grouped_cfg = tb.last_launch()
        tb.check(lib.tmac_b200_graph_begin(), "graph_begin")
        grouped_calls()
        g_grouped = lib.tmac_b200_graph_end(); tb.check(g_grouped, "graph_end")
    kernels_per_step = LAYERS

    # ---- the same chain as ONE persistent launch (decode sequence kernel, tmac_b200_seq_*): op i+1 reads its input from
    #      op i's output (first K rows) -- a TRUE data dependency carried through HBM -- and, for comparison, with the
    #      independent inputs of the launch chain above.  Both write every layer's output.
    out_seq = torch.zeros((LAYERS, MOUT), device="cuda")
    sv2, gathered2, out_plain = None, None, None
    if world > 1:
        # row-sharded form of the sequence: every op also stores its rows into every rank's [world][LAYERS][MOUT] buffer from its
        # epilogue (tmac_b200_seq_peer_outputs), one flag exchange per step; a second, peer-less copy of the sequence checks it
        sv2 = tb.SharedVector(world * LAYERS * MOUT, dist, rank, world)
        gathered2 = sv2.local.view(world, LAYERS, MOUT)
        out_seq = gathered2[rank]
        out_plain = torch.zeros((LAYERS, MOUT), device="cuda")
    seqs = {}
    try:
        for name, chained in (("dependent", True), ("independent", False), ("dependent_streamk", True)) + ((("dependent_plain", True),) if world > 1 else ()):
            tb.debug_set("seq_impl", 0 if name.endswith("streamk") else 2)     # 2 = resident chain where the sequence qualifies
            sq = tb.Sequence()
            dst = out_plain if name == "dependent_plain" else out_seq
            for i, wt in enumerate(layers):
                if chained and i > 0:
                    sq.add(wt, in_op=i - 1, in_offset=0, out=dst[i])
                else:
                    sq.add(wt, x=x[i], out=dst[i])
                if sv2 is not None and name == "dependent":
                    sq.peer_outputs(i, [sv2.peer_ptr(q) + 4 * (rank * LAYERS + i) * MOUT for q in range(world) if q != rank])
            sq.build()
            seqs[name] = sq
    except Exception as ex:
        seqs = {"error": str(ex)[:160]}
    tb.debug_set("seq_impl", 2)
    if world > 1:       # the timed sequence runs contain collectives: either every rank has its sequences or none uses them
        okt = torch.tensor([0 if "error" in seqs else 1], device="cuda", dtype=torch.int32)
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        if not bool(okt.item()) and "error" not in seqs:
            for sq in seqs.values():
                sq.free()
            seqs = {"error": "another rank failed to build its sequences"}

    def run_steps(graph, n):
        if args.eager:
            for _ in range(n):
                graph[1](graph[2])
            return
        tb.check(lib.tmac_b200_graph_launch(graph, 1) if n == 1 else lib.tmac_b200_graph_launch(graph, n), "graph_launch")

    def timed(graph, steps, collective):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(steps):
                run_steps(graph, 1)
                if collective == "nccl" and world > 1:
                    dist.all_gather_into_tensor(nccl_gathered.view(-1), out.reshape(-1))
            e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
            dist.barrier()
        return ms

    with torch.cuda.stream(stream):
        timed(g_step, max(3, args.warmup), True)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    ms = timed(g_step, args.steps, True)
    # the outputs of the last timed step, before the replays below
    dumps = {"launch_chain": (gathered if world > 1 else out).cpu().numpy()} if args.dump_outputs else {}
    launches["n"] = args.steps * kernels_per_step
    # keep the GPU busy a little longer so that the 100 ms clock sampler sees load
    t_end = time.time() + 1.0
    while time.time() < t_end:
        timed(g_step, args.steps, True)
    clocks = sampler.stop() if rank == 0 else None
    gather_check = None
    nccl_step = None
    if world > 1:
        # the fused gather must have produced the same tensor on every rank, and the same bytes as an NCCL all-gather of the
        # ranks' own outputs
        torch.cuda.synchronize(); dist.barrier()
        with torch.cuda.stream(stream):
            dist.all_gather_into_tensor(nccl_gathered.view(-1), out.reshape(-1))
        torch.cuda.synchronize()
        okt = torch.tensor([1 if torch.equal(gathered, nccl_gathered) else 0], device="cuda", dtype=torch.int32)
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        gather_check = bool(okt.item())
        if not gather_check:
            raise SystemExit("bench.py: the fused gather differs from an NCCL all-gather of the ranks' outputs")
        timed(g_step, 3, "nccl")
        ms_nccl = timed(g_step, args.steps, "nccl") / args.steps
        nccl_step = {"what": "same step followed by one ncclAllGather of the step's outputs (round-1 form)", "ms_per_step": ms_nccl,
                     "GBps": world * LAYERS * algorithmic_bytes() / (ms_nccl * 1e-3) / 1e9}
    ms_per_step = ms / args.steps
    bytes_step = LAYERS * algorithmic_bytes()
    value = world * bytes_step / (ms_per_step * 1e-3) / 1e9
    out_launch_chain = out.clone()
    submission = "one tmac_b200_gemv launch per layer (LUT build fused), %d launches captured in one CUDA graph with programmatic-dependent-launch edges" % LAYERS

    def timed_seq(sq, steps, flags=None):
        for _ in range(3):
            sq.launch()
            if flags is not None:
                flags.barrier()
        sq.status()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(steps):
                sq.launch()
                if flags is not None:
                    flags.barrier()             # one flag exchange per step: every rank's rows of this step are in place everywhere
            e1.record(stream)
        torch.cuda.synchronize()
        sq.status()
        t = e0.elapsed_time(e1) / steps
        if world > 1:
            tt = torch.tensor([t], device="cuda"); dist.all_reduce(tt, op=dist.ReduceOp.MAX); t = float(tt.item())
        return t

    seq_report = None
    step_is_sequence = False
    if "error" in seqs:
        seq_report = seqs
    else:
        ms_dep = timed_seq(seqs["dependent"], args.steps, sv2)
        if args.dump_outputs:
            dumps["sequence_dependent_chain"] = (gathered2 if world > 1 else out_seq).cpu().numpy()
        ms_ind, ms_sk = timed_seq(seqs["independent"], args.steps), timed_seq(seqs["dependent_streamk"], args.steps)
        seqs["dependent"].launch(); seqs["dependent"].status()       # the dependent chain's outputs for the parity check (host copy taken now)
        seq_gather_ok = None
        if world > 1:
            # the sharded sequence must equal its peer-less copy bit for bit, and its fused gather an NCCL all-gather of the ranks' rows
            sv2.barrier()
            seqs["dependent_plain"].launch(); seqs["dependent_plain"].status()
            torch.cuda.synchronize(); dist.barrier()
            with torch.cuda.stream(stream):
                dist.all_gather_into_tensor(nccl_gathered.view(-1), out_seq.reshape(-1))
            torch.cuda.synchronize()
            okt = torch.tensor([1 if (torch.equal(gathered2, nccl_gathered) and torch.equal(out_plain, out_seq)) else 0], device="cuda", dtype=torch.int32)
            dist.all_reduce(okt, op=dist.ReduceOp.MIN)
            seq_gather_ok = bool(okt.item())
        out_seq_host = out_seq.cpu().numpy()
        out_seq_nan_now = bool(np.isnan(out_seq_host).any())
        resident = seqs["dependent"].info()["ring_slots"] < 0
        seq_kind = ("resident chain kernel (tmac_chain.cuh): gemv3's clusters kept resident, inputs arrive as {value, epoch} words, next tensor's blocks requested before the lookups"
                    if resident else "stream-K sequence kernel (tmac_seq.cuh): one CTA per SM, TMA weight ring across ops")
        seq_report = {"what": "the %d GEMVs of the step in ONE persistent launch -- %s" % (LAYERS, seq_kind),
                      "dependent_chain": {"ms_per_step": ms_dep, "GBps": world * bytes_step / (ms_dep * 1e-3) / 1e9, "us_per_gemv": ms_dep * 1e3 / LAYERS,
                                          "dependency": "x[i+1] = first K outputs of GEMV i (true data dependency through HBM {value, epoch} words)"},
                      "independent_inputs": {"ms_per_step": ms_ind, "GBps": world * bytes_step / (ms_ind * 1e-3) / 1e9, "us_per_gemv": ms_ind * 1e3 / LAYERS},
                      "streamk_sequence_kernel_dependent_chain": {"ms_per_step": ms_sk, "us_per_gemv": ms_sk * 1e3 / LAYERS, "what": "same chain through tmac_seq.cuh (the fallback for sequences the resident chain does not take)"},
                      "info": seqs["dependent"].info()}
        if world > 1:
            seq_report["sharded"] = {"what": "every op stores its rows into every rank's output buffer from its epilogue (tmac_b200_seq_peer_outputs) + one flag exchange per step; 0 NCCL launches",
                                     "gather_equals_nccl_all_gather_and_peerless_sequence": seq_gather_ok}
        if ms_dep < ms_per_step and (world == 1 or seq_gather_ok):      # the dependent chain in one launch beats the chain of launches: it is the step
            ms_per_step = ms_dep
            value = world * bytes_step / (ms_per_step * 1e-3) / 1e9
            launches["n"] = args.steps * (2 if world > 1 else 1)       # + the flag exchange
            submission = "ONE persistent launch per step (%s); GEMV i+1 consumes GEMV i's output" % seq_kind.split(":")[0]
            step_is_sequence = resident

    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dumps)
    timed(g_two, 3, False)
    ms_two = timed(g_two, args.steps, False) / args.steps
    # ---- roofline of the dominant kernel: gemv launches only --------------------------------------
    timed(g_gemv, 3, False)
    ms_g = timed(g_gemv, args.steps, False)
    t_gemv = ms_g / args.steps / LAYERS * 1e-3
    peak, peak_src = measured_peak()
    achieved = algorithmic_bytes() / t_gemv / 1e9
    kname = "gemv3_kernel<PB=2,SYM,QCH=8,AGQ=4>"
    roofline = {"bound": "hbm", "kernel": kname, "launch": lone_cfg, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "peak_source": peak_src, "us_per_launch": t_gemv * 1e6,
                "submission": submission, "sequence_kernel": seq_report,
                "two_call_step": {"what": "preprocessor + qgemm_lut as two launches per layer (the reference's init/compute split)",
                                  "ms_per_step": ms_two, "GBps": bytes_step / (ms_two * 1e-3) / 1e9}, "algorithmic_bytes_per_launch": algorithmic_bytes(), "traffic": None}
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):       # not measured in this run: dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture
        try:
            tj = json.load(open(tp))
            roofline["traffic"] = tj.get("gemv_kernel_dram_bytes_per_launch")
            roofline["traffic_source"] = "static: " + str(tj.get("source", "profiles/traffic.json (ncu --set full capture)"))
        except Exception:
            pass

    if step_is_sequence:
        # the step IS one launch of the resident chain kernel: it is the dominant kernel.  One launch processes LAYERS GEMVs
        # (LAYERS x the per-GEMV algorithmic bytes); its duration is the CUDA-event time of the step (one kernel per step).
        roofline["gemv3_launch_chain_kernel"] = {"kernel": kname, "launch": lone_cfg, "achieved": achieved, "frac": achieved / peak, "us_per_launch": t_gemv * 1e6,
                                                 "algorithmic_bytes_per_launch": algorithmic_bytes(), "traffic": roofline.get("traffic"), "traffic_source": roofline.get("traffic_source")}
        a2 = bytes_step / (ms_per_step * 1e-3) / 1e9
        roofline.update({"kernel": "chain_kernel<PB=2,QCH=8,AGQ=4> (tmac_chain.cuh; one persistent launch = %d GEMVs)" % LAYERS, "launch": seq_report["info"],
                         "achieved": a2, "frac": a2 / peak, "us_per_launch": ms_per_step * 1e3, "algorithmic_bytes_per_launch": bytes_step, "traffic": None})
        roofline.pop("traffic_source", None)
        try:
            tj = json.load(open(tp))
            if tj.get("chain_kernel_dram_bytes_per_launch"):
                roofline["traffic"] = tj["chain_kernel_dram_bytes_per_launch"]
                roofline["traffic_source"] = "static: " + str(tj.get("chain_source", "profiles/traffic.json (ncu --set full capture)"))
        except Exception:
            pass

    if g_grouped:
        timed(g_grouped, 3, False)
        ms_gr = timed(g_grouped, args.steps, False)
        t_gr = ms_gr / args.steps * 1e-3
        roofline["grouped_launch"] = {"what": "ONE launch for the step's %d independent GEMVs (tmac_b200_qgemm_lut_grouped)" % LAYERS,
                                      "achieved": LAYERS * algorithmic_bytes() / t_gr / 1e9, "frac": LAYERS * algorithmic_bytes() / t_gr / 1e9 / peak,
                                      "us_per_gemv": t_gr / LAYERS * 1e6, "launch": grouped_cfg}

    # ---- e2e: host buffers through the reference-facing call -----------------------------------
    hx = torch.from_numpy(activations(300 + rank)).pin_memory()
    hout = torch.zeros((LAYERS, MOUT)).pin_memory()
    hx_rows = [hx[i] for i in range(LAYERS)]          # the caller's per-layer host buffers (page-locked)
    hout_rows = [hout[i] for i in range(LAYERS)]

    def e2e_step():
        for i, wt in enumerate(layers):               # synchronous, like the CPU operator: returns with the result in hout
            tb.gemv(wt, 1, hx_rows[i], hout_rows[i])

    for _ in range(3):
        e2e_step()
    e2e_steps = args.steps
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    if world > 1:
        t = torch.tensor([e2e_s], device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX); e2e_s = float(t.item())
    e2e = {"value": world * bytes_step / e2e_s / 1e9, "unit": UNIT, "ms_per_step": e2e_s * 1e3,
           "h2d_bytes_per_step": LAYERS * K * 4, "d2h_bytes_per_step": LAYERS * MOUT * 4,
           "call": "tmac_b200_gemv(handle, 1, F32, host_x, host_out) per layer, synchronous: H2D copy of the activation row straight from the caller's "
                   "page-locked buffer + fused LUT/GEMV kernel storing the result into the caller's page-locked buffer + stream sync"}
    launches["n"] += 0
    # ---- the decode-loop form of the same thing: the step's input row copied from page-locked host memory, the dependent chain as ONE
    #      persistent launch (tmac_b200_seq_launch), every layer's output copied back to page-locked host memory, stream sync -- all inside
    #      the timed region.  Reported beside the per-call figure (e2e.value stays the reference-facing per-op call).
    if world == 1 and "error" not in seqs:
        try:
            sqd = seqs["dependent"]
            hx0 = x[0].detach().cpu().pin_memory()
            hseq = torch.zeros((LAYERS, MOUT)).pin_memory()

            def seq_e2e_step():
                with torch.cuda.stream(stream):
                    x[0].copy_(hx0, non_blocking=True)
                    sqd.launch()
                    hseq.copy_(out_seq, non_blocking=True)
                stream.synchronize()
            for _ in range(3):
                seq_e2e_step()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                seq_e2e_step()
            seq_s = (time.perf_counter() - t0) / e2e_steps
            sqd.status()
            e2e["sequence_step"] = {"value": bytes_step / seq_s / 1e9, "unit": UNIT, "ms_per_step": seq_s * 1e3,
                                    "h2d_bytes_per_step": K * 4, "d2h_bytes_per_step": LAYERS * MOUT * 4,
                                    "equals_device_timed_outputs": bool(np.array_equal(hseq.numpy(), out_seq_host)),
                                    "call": "copy of the step's input row from page-locked host memory + tmac_b200_seq_launch (the %d dependent GEMVs in one persistent "
                                            "launch) + copy of all %d output rows to page-locked host memory + stream sync" % (LAYERS, LAYERS)}
        except Exception as ex:
            e2e["sequence_step"] = {"error": str(ex)[:200]}
    # ---- the same through the REFERENCE's own two hook symbols with host workspaces, as ggml calls them: task_init once, then
    #      task_compute for the whole tensor (ref:ggml.c:12610-12630) or once per 64-row weight tile (ref:ggml.c:12662-12691,
    #      172 tiles), driven by the C++ caller emulation tmac_b200_debug_ggml_mul_mat (no interpreter between the calls).
    #      The weights are random bytes in the reference layout (every byte is a valid pair of LUT indices); parity of this
    #      path is the test suite's job (test_ggml_caller_emulation_whole_tensor_and_per_tile).
    try:
        import ctypes as _C
        rng = np.random.default_rng(3)
        A_ref = rng.integers(0, 256, size=MOUT * K * BITS // 8, dtype=np.uint8)
        S_ref = (np.abs(rng.standard_normal(MOUT * (K // GS) * 2)) * 0.01 + 1e-4).astype(np.float16).astype(np.float32)
        kref = tb.make_kcfg(MOUT, K, BITS, 128, 16, GS, AGS, ZP, False)
        tb.check(lib.tmac_b200_register_kcfg(_C.byref(kref)), "register_kcfg")
        wt_ref = tb.upload_reference_layout(kref, A_ref, S_ref)
        wdata = np.zeros(K * 4 + 2 * (K // AGS) * 4 + 64, np.uint8)
        dst = np.zeros(MOUT, np.float32)
        hx_np = hx.numpy()
        ref_sym = {}
        for label, per_tile, threads in (("whole_tensor", 0, 1), ("per_tile_1_thread", 1, 1), ("per_tile_4_threads", 1, min(4, os.cpu_count() or 1))):
            def one(i):
                tb.check(lib.tmac_b200_debug_ggml_mul_mat(A_ref.ctypes.data, S_ref.ctypes.data, hx_np[i % LAYERS].ctypes.data, wdata.ctypes.data,
                                                          dst.ctypes.data, MOUT, K, BITS, 128 // BITS, per_tile, threads), "ggml emulation")
            for i in range(3):
                one(i)
            t0 = time.perf_counter()
            nrep = 40
            for i in range(nrep):
                one(i)
            dt = (time.perf_counter() - t0) / nrep
            ref_sym[label] = {"us_per_gemv": dt * 1e6, "GBps": algorithmic_bytes() / dt / 1e9}
        ref_sym["note"] = ("ONE resident tensor (L2-warm weights): this measures the call path -- H2D of the row, LUT build, D2H of the LUT into the "
                           "caller's workspace, GEMV, result into page-locked memory, per-tile row copies -- not the HBM stream")
        e2e["reference_symbols"] = ref_sym
        wt_ref.free()
    except Exception as ex:
        e2e["reference_symbols"] = {"error": str(ex)[:200]}

    extras = {}
    cpu = None
    def headline(extras_, cpu_):
        return {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "int8 LUT / int32 dp4a / fp32 scale", "data": "synthetic", "config": workload_config(world),
                "clocks": clocks, "fused_gather_equals_nccl_all_gather": gather_check, "nccl_all_gather_step": nccl_step, "e2e": e2e, "gpu_launches": launches["n"], "roofline": roofline,
                "cpu_baseline": cpu_, "tokens_per_s": extras_}

    if (world > 1 or force_sharded) and not args.no_extras:   # all ranks: the model's linears row-sharded over the ranks
        # The extras use collectives on every rank; a watchdog bounds them so that a stuck collective can never cost the
        # headline line: on expiry rank 0 prints the line without the extras and every rank exits.
        def expire():
            if rank == 0:
                print(json.dumps(headline({"error": "sharded tokens/s extras exceeded their time limit"}, None)), flush=True)
            os._exit(0)
        dog = threading.Timer(float(os.environ.get("TMAC_BENCH_EXTRAS_LIMIT_S", "300")), expire)
        dog.daemon = True
        dog.start()
        try:
            extras = tokens_per_second_sharded(tb, lib, torch, dist, stream, rank, world)
        except Exception as ex:
            extras = {"error": str(ex)[:200]}
        dog.cancel()
    elif rank == 0 and not args.no_extras:
        try:
            extras = tokens_per_second(tb, lib, torch, stream)
        except Exception as ex:  # extras must never kill the headline line
            extras = {"error": str(ex)[:200]}
        if world == 1:
            cpu = cpu_arm(12.0)
            try:
                cpu["parity_check"] = parity_check(w, sc, z, x.cpu().numpy(), out_launch_chain.cpu().numpy(),
                                                   out_seq_host if (seq_report and "error" not in seq_report) else None)
                cpu["parity_check"]["out_seq_device_copy_changed_later"] = bool(seq_report and "error" not in seq_report and
                                                                                not np.array_equal(out_seq_host, out_seq.cpu().numpy(), equal_nan=True))
            except AssertionError as ex:
                raise SystemExit("bench.py: GPU outputs disagree with the CPU reference: %s" % ex)

    if rank == 0:
        print(json.dumps(headline(extras, cpu)), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def tokens_per_second_sharded(tb, lib, torch, dist, stream, rank, world):
    """Matmul-only decode tokens/s with every quantised linear ROW-SHARDED over the ranks (SURVEY 8e: whole reference
    tiles per rank, remainders spread; every rank runs its own LUT build).  No collective launch: every GEMV stores its
    finished rows into every rank's output vector from its epilogue (tmac_b200_peer_outputs) and each fused group
    (q/k/v, o, gate/up, down = 4 per layer) ends with one flag exchange (tmac_b200_peer_barrier), the token step captured in
    one CUDA graph.  Strong scaling: the model is fixed, per-rank weights = 1/world.  Runs on ALL ranks."""
    sys.path.insert(0, os.path.join(ROOT, "t-mac_b200"))
    from shard import row_partition
    models = {
        "llama2_7b_w2_g128_zp": dict(L=32, bits=2, zp=True, os=False, shapes=[("qkv", 4096, 4096, 3), ("o", 4096, 4096, 1), ("gateup", 11008, 4096, 2), ("down", 4096, 11008, 1)]),
        "bitnet_3b_w2": dict(L=26, bits=2, zp=False, os=True, shapes=[("qkv", 3200, 3200, 3), ("o", 3200, 3200, 1), ("gateup", 8640, 3200, 2), ("down", 3200, 8640, 1)]),
        "qwen2_7b_w4_g128_zp": dict(L=28, bits=4, zp=True, os=False, shapes=[("q", 3584, 3584, 1), ("kv", 512, 3584, 2), ("o", 3584, 3584, 1), ("gateup", 18944, 3584, 2), ("down", 3584, 18944, 1)]),
    }

    def all_ok(ok):
        t = torch.tensor([1 if ok else 0], device="cuda", dtype=torch.int32)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item())

    res = {}
    for name, m in models.items():
        handles, plan, local_bytes, err = [], [], 0, None
        sv = None
        try:
            sv = tb.SharedVector(max(cnt * mout for (_, mout, _, cnt) in m["shapes"]), dist, rank, world)
            for (tag, mout, k, cnt) in m["shapes"]:
                bits = m["bits"]
                bm = next(b for b in ((192, 384, 576, 768) if bits == 3 else (256, 128, 512, 1024, 320, 640)) if (mout * bits) % b == 0)
                parts = row_partition(mout, bm // bits, world)
                row0, rows = parts[rank]
                ags = k if m["os"] else 64
                with torch.cuda.stream(stream):
                    xb = torch.randn((1, k), device="cuda")
                    q = torch.zeros((1, k // 4, 16), dtype=torch.int8, device="cuda")
                    l1 = torch.zeros((1, k // ags), device="cuda"); l2 = torch.zeros_like(l1)
                hs = []
                if rows > 0:
                    w, sc, z = synth(7, mout, k, bits, 128, m["zp"], m["os"])
                    cfg = tb.make_kcfg(rows, k, bits, bm, 16, 128, ags, m["zp"], m["os"])
                    base = tb.upload_plain(cfg, np.ascontiguousarray(w[row0:row0 + rows]), sc if m["os"] else np.ascontiguousarray(sc[row0:row0 + rows]),
                                           None if z is None else np.ascontiguousarray(z[row0:row0 + rows]))
                    hs = [base] + [tb.clone(base) for _ in range(m["L"] * cnt - 1)]
                    handles += hs
                    local_bytes += m["L"] * cnt * base.nbytes
                plan.append((hs, cnt, mout, k, ags, xb, q, l1, l2, row0, rows))
        except Exception as ex:
            err = str(ex)[:160]
        if not all_ok(err is None):
            res[name] = {"error": err or "another rank failed to build its shard"}
            for h in handles:
                h.free()
            continue

        def token():
            for layer in range(m["L"]):
                for (hs, cnt, mout, k, ags, xb, q, l1, l2, row0, rows) in plan:
                    if rows > 0:
                        for c in range(cnt):
                            tb.peer_outputs([sv.peer_ptr(p_) + 4 * (c * mout + row0) for p_ in range(world) if p_ != rank])
                            dst = sv.local[c * mout + row0: c * mout + row0 + rows]
                            tb.gemv(hs[layer * cnt + c], 1, xb, dst)          # LUT built inside the GEMV (fp and integer path)
                    sv.barrier()                                               # the group's output vector is whole on every rank

        ok, mode = True, "one CUDA graph per token (library launches only: peer stores + one flag exchange per fused group)"
        try:
            with torch.cuda.stream(stream):
                token()
            torch.cuda.synchronize()
            tb.check(lib.tmac_b200_graph_begin(), "graph_begin")
            token()
            g = lib.tmac_b200_graph_end(); tb.check(g, "graph_end")
        except Exception as ex:
            ok, err = False, str(ex)[:160]
        if not all_ok(ok):
            res[name] = {"error": err or "another rank failed"}
            for h in handles:
                h.free()
            continue
        n = 10
        tb.check(lib.tmac_b200_graph_launch(g, 2), "warm")
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream); tb.check(lib.tmac_b200_graph_launch(g, n), "run"); e1.record(stream)
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / n * 1e-3], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sec = float(t.item())
        tot = torch.tensor([float(local_bytes)], device="cuda"); dist.all_reduce(tot)
        res[name] = {"tokens_per_s_matmul_only": 1.0 / sec, "ms_per_token": sec * 1e3, "ranks": world, "nccl_launches_per_token": 0,
                     "flag_exchanges_per_token": m["L"] * len(plan),
                     "resident_weight_GB_total": float(tot.item()) / 1e9, "weight_stream_GBps_total": float(tot.item()) / sec / 1e9, "step": mode}
        lib.tmac_b200_graph_free(g)
        for h in handles:
            h.free()
        sv.close(dist)
    return res


def tokens_per_second(tb, lib, torch, stream):
    """Matmul-only decode tokens/s (all quantised linears of every layer, preprocessors shared as in
    the model graph: q/k/v share one, gate/up share one), synthetic weights at the real shapes."""
    models = {
        "llama2_7b_w2_g128_zp": dict(L=32, bits=2, zp=True, os=False, shapes=[("qkv", 4096, 4096, 3), ("o", 4096, 4096, 1), ("gateup", 11008, 4096, 2), ("down", 4096, 11008, 1)]),
        "llama2_7b_w4_g128": dict(L=32, bits=4, zp=False, os=False, shapes=[("qkv", 4096, 4096, 3), ("o", 4096, 4096, 1), ("gateup", 11008, 4096, 2), ("down", 4096, 11008, 1)]),
        "bitnet_3b_w2": dict(L=26, bits=2, zp=False, os=True, shapes=[("qkv", 3200, 3200, 3), ("o", 3200, 3200, 1), ("gateup", 8640, 3200, 2), ("down", 3200, 8640, 1)]),
    }
    res = {}
    for name, m in models.items():
        handles, plan, total_bytes = [], [], 0
        for (tag, mout, k, cnt) in m["shapes"]:
            w, sc, z = synth(7, mout, k, m["bits"], 128, m["zp"], m["os"])
            bm = 256 if (mout * m["bits"]) % 256 == 0 else (128 if (mout * m["bits"]) % 128 == 0 else 320)
            cfg = tb.make_kcfg(mout, k, m["bits"], bm, 16, 128, k if m["os"] else 64, m["zp"], m["os"])
            base = tb.upload_plain(cfg, w, sc, z)
            hs = [base] + [tb.clone(base) for _ in range(m["L"] * cnt - 1)]
            handles += hs
            ags = k if m["os"] else 64
            with torch.cuda.stream(stream):
                xb = torch.randn((1, k), device="cuda")
                q = torch.zeros((1, k // 4, 16), dtype=torch.int8, device="cuda")
                l1 = torch.zeros((1, k // ags), device="cuda"); l2 = torch.zeros_like(l1)
                o = torch.zeros((cnt, mout), device="cuda")
            plan.append((hs, cnt, k, ags, xb, q, l1, l2, o))
            total_bytes += m["L"] * cnt * tb.load().tmac_b200_weights_nbytes(base.handle)

        def token():
            for layer in range(m["L"]):
                for (hs, cnt, k, ags, xb, q, l1, l2, o) in plan:
                    if cnt == 1:
                        tb.gemv(hs[layer], 1, xb, o[0])                      # LUT built inside the GEMV (fp and integer path)
                    elif not m["os"]:                                      # q/k/v, gate/up share their input: one grouped launch, LUT built inside
                        tb.gemv_grouped(hs[layer * cnt:(layer + 1) * cnt], 1, xb, [o[c] for c in range(cnt)])
                    else:                                                  # integer path: the row-wide scale costs a row scan per cluster; a group
                        tb.preprocessor(k, 1, ags, xb, l1, l2, q)          # shares ONE preprocessor launch instead (measured faster)
                        tb.qgemm_lut_grouped(hs[layer * cnt:(layer + 1) * cnt], 1, [q] * cnt, [l1] * cnt, [l2] * cnt, [o[c] for c in range(cnt)])
        token()
        tb.check(lib.tmac_b200_sync(), "sync")
        tb.check(lib.tmac_b200_graph_begin(), "graph_begin")
        token()
        g = lib.tmac_b200_graph_end(); tb.check(g, "graph_end")
        tb.check(lib.tmac_b200_graph_launch(g, 3), "warm"); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n = 20
        e0.record(stream); tb.check(lib.tmac_b200_graph_launch(g, n), "run"); e1.record(stream)
        torch.cuda.synchronize()
        s = e0.elapsed_time(e1) / n * 1e-3
        res[name] = {"tokens_per_s_matmul_only": 1.0 / s, "ms_per_token": s * 1e3, "resident_weight_GB": total_bytes / 1e9,
                     "weight_stream_GBps": total_bytes / s / 1e9}
        lib.tmac_b200_graph_free(g)
        for h in handles:
            h.free()
    # Full decode step (SURVEY 8 f1): the same linears inside the real per-layer op order with torch fp32 RMSNorm / RoPE / attention over
    # a 512-position KV cache / SiLU*mul / residuals, one CUDA graph per token (t-mac_b200/decode_harness.py).
    try:
        from decode_harness import DecodeModel
        for name, kw in (("llama2_7b_w2_g128_zp", dict(layers=32, hidden=4096, ffn=11008, heads=32, bits=2, zero_point=True)),):
            m = DecodeModel(ctx=512, **kw)
            m.capture(stream)
            res[name]["tokens_per_s_full_step"] = m.tokens_per_s(stream, n=10)
            res[name]["full_step"] = "quantised linears through the library + torch fp32 norm / rope / attention (ctx 512) / activation, CUDA graph"
            m.free()
    except Exception as ex:
        res["decode_harness_error"] = str(ex)[:200]
    # Prefill-shaped call (BASELINE config 4: Llama-2-7B W2, seq 256): N >= 32 takes the tcgen05 kind::i8 tile
    # (tmac_prefill.cuh): preprocessor + LUT tiling + GEMM.  Tensor-pipe utilisation = int8 MMA rate / 4500 TOP/s (dense peak).
    try:
        NB = 256
        w, sc, z = synth(9)
        cfg = tb.make_kcfg(MOUT, K, BITS, 128, 16, GS, AGS, ZP, False)
        wt = tb.upload_plain(cfg, w, sc, z)
        with torch.cuda.stream(stream):
            xb = torch.randn((NB, K), device="cuda"); ob = torch.zeros((NB, MOUT), device="cuda")
        tb.gemv(wt, NB, xb, ob); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(3):
            tb.gemv(wt, NB, xb, ob)
        e1.record(stream); torch.cuda.synchronize()
        s = e0.elapsed_time(e1) / 3 * 1e-3
        ll = tb.last_launch()
        mma = 2.0 * NB * MOUT * (2 * K) / s / 1e12            # contraction length = 8 LUT entries per K-group = 2K
        fp16_tile = ll["cluster"] == 16
        nominal = 2250.0 if fp16_tile else 4500.0             # dense fp16 / int8 tensor peak, TFLOP/s (B200_PROFILING.md)
        measured = None
        try:
            measured = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"]) * (1.0 if fp16_tile else 2.0)
        except Exception:
            pass
        res["prefill_seq256_one_tensor_11008x4096_w2"] = {
            "ms": s * 1e3, "what": "preprocessor + LUT tiling + tcgen05 GEMM, one call (tmac_b200_gemv, N = 256)",
            "tokens_per_s_this_tensor": NB / s, "dense_equivalent_TFLOPs": 2.0 * NB * MOUT * K / s / 1e12,
            "mma_TFLOPs": mma, "tensor_pipe_utilisation_vs_nominal": mma / nominal,
            "tensor_pipe_utilisation_vs_measured_cublas_peak": (mma / measured) if measured else None,
            "path": ("tcgen05.mma kind::f16 tile, scales folded into fp16 operands, fp32 accumulation in TMEM (LUT contraction, 8 entries per K-group)"
                     if fp16_tile else "tcgen05.mma kind::i8 tile (one-hot-signed LUT contraction)") if ll["batch"] < 0 else "GEMV kernel per activation row"}
        wt.free()
    except Exception as ex:
        res["prefill_seq256_one_tensor_11008x4096_w2"] = {"error": str(ex)[:160]}
    return res


if __name__ == "__main__":
    main()
