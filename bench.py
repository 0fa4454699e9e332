#!/usr/bin/env python
"""Benchmark of the rulebook -> implicit-GEMM hot path (BASELINE.json metric and configs).

    python bench.py --gpus N --steps K --warmup W              # this engine, one rank per GPU
    python bench.py --impl reference --gpus N --steps K ...    # the reference's CPU path
    python bench.py --workload second_encoder6_fp16 ...        # another BASELINE config as headline
    python bench.py --dump-outputs DIR ...                     # + the last timed step's outputs as DIR/*.npy

Headline workload = BASELINE.json configs[1] (the configuration the metric is quoted on): one
SubMConv3d 3x3x3 C = K = 64 fp16 over a ~100 k-voxel KITTI-shaped cloud per GPU.  A "step" is one
pass of the hot path over one batch: rulebook generation (hash + probe + mask sort + tile table)
-> forward -> backward (input gradient + weight gradient); at N > 1 every rank processes its own
cloud (weak scaling) and the weight gradient is all-reduced once per step over NCCL.

* ``value``  active voxels of all ranks / step time, inputs resident in HBM, CUDA events around
  every step on the launching stream, max over ranks;
* ``e2e``    the same metric through the public module API starting from pinned HOST buffers
  (H2D of coordinates + features and D2H of loss + weight gradients inside the timed region);
* ``workloads``  (default run only) the other BASELINE configs measured the same way:
  configs[2] the 6-layer SECOND encoder, configs[3] SparseConv3d stride 2 bf16 300 k voxels
  (+ its indice_key-reuse leg), configs[4] int8 SubMConv3d inference.

See DESIGN.md section "Measurement".
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time
from typing import Dict, List, Optional

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from bench_utils import (ENCODER6_LAYERS, ClockSampler, algorithmic_bytes, conv_flops,  # noqa: E402
                         load_peaks, make_encoder6, surface_cloud)

KITTI = [41, 1600, 1408]
WORKLOADS = {
    # BASELINE.json configs[1]: the configuration the metric is quoted on
    "submconv3d_k3_c64_fp16_100k_kitti": dict(kind="layer", shape=KITTI, n=100_000, c_in=64, c_out=64,
                                              dtype="fp16", subm=True, ksize=3, stride=1, padding=1),
    # BASELINE.json configs[2]: one cloud per GPU (8 clouds on 8 GPUs) / the whole batch on one GPU
    "second_encoder6_fp16": dict(kind="encoder", shape=KITTI, n=100_000, batch=1, dtype="fp16"),
    "second_encoder6_fp16_b8": dict(kind="encoder", shape=KITTI, n=100_000, batch=8, dtype="fp16"),
    # BASELINE.json configs[3]
    "sparseconv3d_k3s2_c64_128_bf16_300k": dict(kind="layer", shape=[41, 1440, 1440], n=300_000, c_in=64,
                                                c_out=128, dtype="bf16", subm=False, ksize=3, stride=2,
                                                padding=1, reuse_calls=2),
    # BASELINE.json configs[4] (inference: forward only)
    "int8_submconv3d_k3_c64_100k": dict(kind="int8", shape=KITTI, n=100_000, c_in=64, c_out=64, dtype="int8",
                                        subm=True, ksize=3, stride=1, padding=1),
}
DEFAULT_WORKLOAD = "submconv3d_k3_c64_fp16_100k_kitti"
EXTRA_WORKLOADS = ["second_encoder6_fp16", "sparseconv3d_k3s2_c64_128_bf16_300k", "int8_submconv3d_k3_c64_100k"]
METRIC = "active-voxels/sec fwd+bwd SubMConv3d 3^3 C=64"
NUM_CLOUDS = 4          # distinct clouds per rank, rotated so consecutive steps never share inputs
L2_FLUSH_BYTES = 256 << 20
CPU_THREAD_CAP = 16     # the small per-offset GEMMs get SLOWER with more BLAS threads (measured: 128 -> 3.2 s/step)
DUMP_BYTES = 60 << 20   # --dump-outputs budget (below 64 MB with the .npy headers); larger outputs are row-sampled


def metric_name(workload: str) -> str:
    """BASELINE.json's metric for the default workload; other workloads are labelled as what they are."""
    if workload == DEFAULT_WORKLOAD:
        return METRIC
    if WORKLOADS[workload]["kind"] == "int8":
        return f"active-voxels/sec fwd (inference) {workload}"
    return f"active-voxels/sec fwd+bwd {workload}"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps: of each of the three repetitions of the headline workload's timed region, and "
                         "of --impl reference; the extra workloads time max(5, min(steps, 10))")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--graph", type=int, default=1, help="replay the device-resident step from CUDA graphs")
    ap.add_argument("--pipeline", type=int, default=2,
                    help="software-pipeline the graph replay: 1 = rulebook of cloud i+1 beside the GEMMs of cloud i "
                         "(streams joined every step), 2 = rulebooks two clouds ahead on two side streams, 0 = serial; "
                         "3 = 2 + the eager encoder prefetches its whole rulebook chain from a worker thread")
    ap.add_argument("--extras", type=int, default=-1,
                    help="also measure the other BASELINE configs (default: only in the default-workload run)")
    ap.add_argument("--allreduce", default="auto", choices=["auto", "fused", "nccl", "fused-local"],
                    help="N > 1, the all-reduce of dW: nccl = from a hook right behind the weight gradient; fused = the "
                         "exchange over NVLink peer memory whose send side is the weight-gradient reduction kernel "
                         "(csrc/peer.cu); auto (default) = what was measured faster under graph replay: nccl up to 4 GPUs "
                         "(0.146 vs 0.159 ms per step at N = 2), fused from 8 (0.1661 vs 0.1686 ms; through the eager module "
                         "API fused wins everywhere: 1.4 vs 4.2 ms at N = 8); fused-local = triage (every rank exchanges "
                         "with itself)")
    ap.add_argument("--peer-triage", type=int, default=0, help="triage of the fused exchange (timing only, results are wrong): "
                    "1 skip finish, 2 plain weight gradient instead of push")
    ap.add_argument("--cpu-sample", type=int, default=100_000, help="voxels in the CPU-baseline sample")
    ap.add_argument("--debug-bits", type=int, default=0,
                    help="spx_debug_configure bits for A/B runs (64 onesweep sort, 128 round-1 conv rulebook, "
                         "512 cooperative sort); recorded in config.debug_bits")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step of the headline workload returned "
                         "(output coordinates and features, gradients, loss) as DIR/<name>.npy in float32, at most "
                         "64 MB in all (a seeded row sample of every array beyond that); rank 0 only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ============================================================================ CPU reference arm
def cpu_threads() -> int:
    return min(os.cpu_count() or 1, CPU_THREAD_CAP)


def limit_cpu_threads():
    """The reference's CPU path runs its per-offset mm on the host BLAS (torch.mm) and, in its
    CPU build, the gather/scatter loops under OpenMP; give both the thread count where the path is
    fastest on this box instead of oversubscribing every core."""
    os.environ.setdefault("OMP_NUM_THREADS", str(cpu_threads()))
    try:
        import torch
        torch.set_num_threads(cpu_threads())
    except Exception:
        pass
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=cpu_threads())
    except Exception:
        pass


def cpu_layers(wl):
    """[(subm, c_in, c_out, stride)] of the workload, as the CPU arm runs it."""
    if wl["kind"] == "encoder":
        return [(k == "subm", ci, co, 1 if k == "subm" else 2) for k, ci, co, _ in ENCODER6_LAYERS]
    return [(wl["subm"], wl["c_in"], wl["c_out"], wl["stride"])]


def cpu_reference_step(orc, inds, feats, weights, wl, impl, batch=1):
    """The reference's CPU path for one batch: rulebook (single-threaded ``std::unordered_map``
    loops, spconv/csrc/sparse/indices.py:1640-1778) + gather / torch.mm / scatter-add forward and
    backward (convops.py:1606-1633, :1831-1860) for every layer of the workload.  A rulebook shared
    through an ``indice_key`` is built once, as in the reference (conv.py:247-319)."""
    nd = 3
    t_rb = t_fwd = t_bwd = 0.0
    shape = list(wl["shape"])
    cur, x = inds, feats
    saved = []
    cache = {}
    for li, (subm, c_in, c_out, stride) in enumerate(cpu_layers(wl)):
        key = ("subm", tuple(shape), cur.shape[0]) if subm else None
        t0 = time.perf_counter()
        if key is not None and key in cache:
            out_inds, pairs, num = cache[key]
        else:
            out_inds, pairs, num = orc.get_indice_pairs(cur, batch, shape, [3] * nd, [stride] * nd, [1] * nd,
                                                        [1] * nd, [0] * nd, subm, impl=impl)
            if key is not None:
                cache[key] = (out_inds, pairs, num)
        t1 = time.perf_counter()
        y = orc.indice_conv(x, weights[li], pairs, num, out_inds.shape[0], False, subm)
        t2 = time.perf_counter()
        t_rb += t1 - t0
        t_fwd += t2 - t1
        saved.append((x, pairs, num, subm))
        if not subm:
            shape = orc.get_conv_output_size(shape, [3] * nd, [stride] * nd, [1] * nd, [1] * nd)
        cur, x = out_inds, y
    if wl["kind"] != "int8":
        dout = x * np.float32(2.0 / x.size)
        for li in range(len(saved) - 1, -1, -1):
            xi, pairs, num, subm = saved[li]
            t0 = time.perf_counter()
            dout, _ = orc.indice_conv_backward(xi, weights[li], dout, pairs, num, False, subm)
            t_bwd += time.perf_counter() - t0
    return {"rulebook_s": t_rb, "fwd_s": t_fwd, "bwd_s": t_bwd, "total_s": t_rb + t_fwd + t_bwd, "n": inds.shape[0]}


def make_cpu_sample(wl, n, seed):
    rng = np.random.default_rng(seed)
    scale = max(n / wl["n"], 1e-3) ** 0.5
    shape = [wl["shape"][0], max(64, int(wl["shape"][1] * scale)), max(64, int(wl["shape"][2] * scale))]
    inds = surface_cloud(rng, shape, n)
    layers = cpu_layers(wl)
    feats = rng.uniform(-1, 1, size=(inds.shape[0], layers[0][1])).astype(np.float32)
    weights = [rng.uniform(-1, 1, size=(co, 3, 3, 3, ci)).astype(np.float32) / np.sqrt(27 * ci) for _, ci, co, _ in layers]
    wl_s = dict(wl)
    wl_s["shape"] = shape
    return inds, feats, weights, wl_s


def cpu_arm(wl, n_sample, min_reps, max_reps, budget_s):
    """Times the CPU path on a bounded sample.  Returns (cpu_baseline dict, value)."""
    from oracle import oracle as orc
    orc.build()
    impl = "ref" if orc.have_ref() else "port"
    limit_cpu_threads()
    inds, feats, weights, wl_s = make_cpu_sample(wl, n_sample, 1234)
    cpu_reference_step(orc, inds[:2000], feats[:2000], weights, wl_s, impl)          # warm BLAS / page in
    recs, t0 = [], time.perf_counter()
    while len(recs) < min_reps or (time.perf_counter() - t0 < budget_s and len(recs) < max_reps):
        recs.append(cpu_reference_step(orc, inds, feats, weights, wl_s, impl))
    tot = sum(r["total_s"] for r in recs)
    value = inds.shape[0] * len(recs) / tot
    kind = "reference" if impl == "ref" else "port"
    what = ("the reference's own C++ (oracle/_ref: SparseConvIndicesCPU + GatherCPU compiled from /root/reference)"
            if impl == "ref" else "C restatement of the reference CPU rulebook + gather/scatter")
    sample = (f"{inds.shape[0]} voxels of the same generator in a {wl_s['shape']} grid, fp32, {len(recs)} reps "
              f"({tot:.1f} s): single-threaded hash-map rulebook + gather / torch.mm / scatter-add "
              f"{'fwd' if wl['kind'] == 'int8' else 'fwd+bwd'}; {what}")
    return ({"value": value, "unit": "voxels/s", "cores": cpu_threads(), "kind": kind, "sample": sample,
             "rulebook_ms": 1e3 * sum(r["rulebook_s"] for r in recs) / len(recs),
             "fwd_ms": 1e3 * sum(r["fwd_s"] for r in recs) / len(recs),
             "bwd_ms": 1e3 * sum(r["bwd_s"] for r in recs) / len(recs)}, value, len(recs), tot)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    cb, value, steps, tot = cpu_arm(wl, args.cpu_sample, args.steps, args.steps, 0.0)
    line = {
        "impl": "reference", "metric": metric_name(args.workload), "value": value, "unit": "voxels/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": 1, "ms_per_step": 1e3 * tot / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": {"workload": args.workload, "sample": cb["sample"], "impl_note":
                   "the reference package cannot be pip-installed here (pccm/cumm/ccimport absent); its CPU rulebook "
                   "and gather/scatter C++ are extracted and compiled by oracle/make_ref.py, mm = torch.mm as in "
                   "spconv/pytorch/cppcore.py"},
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": "voxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ============================================================================ GPU arm: workloads
class Ctx:
    """Process-wide handles (one rank = one GPU)."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        import spconv_b200.pytorch as spconv
        from spconv_b200.pytorch import ops
        self.torch, self.dist, self.spconv, self.ops, self.args = torch, dist, spconv, ops, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        assert torch.cuda.is_available(), "bench.py (impl=ours) needs a CUDA device; there is no CPU path"
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        ops._PEER_TRIAGE = int(args.peer_triage)
        if args.debug_bits:
            from spconv_b200 import _cabi
            _cabi.check(_cabi.load().spx_debug_configure(-1, 0, int(args.debug_bits), None, 0), "debug_configure")
        # N > 1: the all-reduce of dW is the tail of the weight-gradient kernel (NVLink peer stores, csrc/peer.cu);
        # --allreduce nccl keeps the library collective for A/B.  All ranks agree on which one runs.
        self.peers = None
        if args.allreduce == "fused-local":
            # triage only: every rank exchanges with itself (world-of-one group) -- the kernels of the fused path
            # without the cross-rank dependency
            from spconv_b200.pytorch.dist import PeerGroup
            self.peers = PeerGroup.local_ring(1, capacity_bytes=8 << 20, average=False)[0]
        # auto: the fused exchange serves the headline workload from 8 GPUs on (the combination measured on 8 GPUs);
        # the extra workloads keep the NCCL bucket there (their 8-GPU runs used it)
        self.allreduce_auto = args.allreduce == "auto"
        if args.allreduce == "auto":
            args.allreduce = "fused" if self.world >= 8 else "nccl"
        if self.world > 1 and args.allreduce == "fused":
            from spconv_b200.pytorch.dist import PeerGroup
            ok = torch.ones(1, device=self.dev, dtype=torch.int32)
            try:
                self.peers = PeerGroup(capacity_bytes=8 << 20, average=False)
            except Exception as e:          # no peer mapping on this box: every rank falls back together
                print(f"[bench] rank {self.rank}: fused all-reduce unavailable ({type(e).__name__}: {e}); using NCCL",
                      file=sys.stderr)
                ok.zero_()
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok.item()) == 0:
                self.peers = None
        self.flush = torch.empty(L2_FLUSH_BYTES // 4, dtype=torch.float32, device=self.dev)
        self.side = torch.cuda.Stream()
        self.side2 = torch.cuda.Stream()

    def allreduce(self, t):
        if self.world > 1 and t is not None:
            self.dist.all_reduce(t)

    def timed_loop(self, step_fn, steps):
        """K steps; CUDA events on the launching stream around every step, L2 flushed in between
        (outside the events); barrier + synchronize on both sides; returns per-step ms."""
        torch = self.torch
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()
        for i in range(steps):
            self.flush.zero_()
            evs[i][0].record()
            step_fn(i)
            evs[i][1].record()
        torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        return [a.elapsed_time(b) for a, b in evs]


TORCH_DT = {"fp16": "float16", "bf16": "bfloat16", "fp32": "float32", "int8": "int8"}


class Workload:
    """One BASELINE config.  Subclasses provide ``device_step`` (inputs resident in HBM) and
    ``e2e_body`` (public module API on freshly copied inputs)."""
    graphable = False
    inference = False
    record_outputs = False                       # --dump-outputs: steps keep references to what they returned

    def __init__(self, name: str, ctx: Ctx):
        self.name, self.ctx, self.wl = name, ctx, WORKLOADS[name]
        torch = ctx.torch
        self.tdt = getattr(torch, TORCH_DT[self.wl["dtype"]])
        self.elem = {"fp16": 2, "bf16": 2, "fp32": 4, "int8": 1}[self.wl["dtype"]]
        self.batch = int(self.wl.get("batch", 1))
        self.clouds: List[dict] = []

    # ---- inputs
    def make_clouds(self, c_in: int):
        torch, ctx = self.ctx.torch, self.ctx
        for i in range(NUM_CLOUDS):
            rng = np.random.default_rng(50051 + 1000 * ctx.rank + i)
            inds_np = surface_cloud(rng, self.wl["shape"], self.wl["n"], batch=self.batch)
            if self.wl["dtype"] == "int8":
                feats = torch.from_numpy(rng.integers(-127, 128, size=(inds_np.shape[0], c_in)).astype(np.int8))
            else:
                feats = torch.from_numpy(rng.uniform(-1, 1, size=(inds_np.shape[0], c_in)).astype(np.float32)).to(self.tdt)
            h_inds = torch.from_numpy(inds_np).pin_memory()
            h_feats = feats.pin_memory()
            self.clouds.append(dict(h_inds=h_inds, h_feats=h_feats, d_inds=h_inds.to(ctx.dev),
                                    d_feats=h_feats.to(ctx.dev), n=inds_np.shape[0]))
        self.n_per_step = sum(c["n"] for c in self.clouds) / NUM_CLOUDS

    def h2d_bytes(self):
        c = self.clouds[0]
        return int(c["h_inds"].numel() * 4 + c["h_feats"].numel() * c["h_feats"].element_size())

    # ---- hooks
    def setup(self): raise NotImplementedError
    def device_step(self, c, timer=None): raise NotImplementedError
    def grads(self): return None                 # flat tensor all-reduced / read back per step
    prefetcher = None                            # RulebookPrefetcher of the input-level SubM layers, if any
    def make_input(self, d_inds, d_feats): raise NotImplementedError
    def e2e_from_input(self, x): raise NotImplementedError
    def e2e_body(self, d_inds, d_feats): return self.e2e_from_input(self.make_input(d_inds, d_feats))
    def config(self) -> dict: return {}
    def region_kinds(self) -> Dict[str, tuple]: return {}

    def outputs(self, c) -> dict:
        """What the last step run or captured on cloud ``c`` returned to its caller, by name (recorded only
        while ``record_outputs`` is set)."""
        return c["outputs"]


class LayerWorkload(Workload):
    """One SubMConv3d / SparseConv3d layer: operator-level device step, module-level e2e."""

    def setup(self):
        ctx, wl, torch = self.ctx, self.wl, self.ctx.torch
        from spconv_b200.core import ConvAlgo
        self.algo = ConvAlgo.MaskImplicitGemm
        nd = 3
        self.ks, self.st, self.pd, self.dl = [wl["ksize"]] * nd, [wl["stride"]] * nd, [wl["padding"]] * nd, [1] * nd
        self.kv = wl["ksize"] ** nd
        self.C, self.K = wl["c_in"], wl["c_out"]
        self.graphable = bool(wl["subm"])           # a regular conv has one host sync (the output count)
        self.make_clouds(self.C)
        torch.manual_seed(48848)
        cls = ctx.spconv.SubMConv3d if wl["subm"] else ctx.spconv.SparseConv3d
        self.layer = cls(self.C, self.K, wl["ksize"], wl["stride"], wl["padding"], bias=False,
                         indice_key="bench" if wl["subm"] else None, algo=self.algo).to(ctx.dev).to(self.tdt)
        self.layer.train()
        if wl["subm"]:
            self.prefetcher = ctx.spconv.RulebookPrefetcher([self.layer], stream=ctx.side)
        self.weight = self.layer.weight.detach()
        self.weight2 = (self.weight * 0.5).contiguous()      # second layer of the indice_key-reuse leg
        self.grad_buf = torch.zeros_like(self.weight)         # what the all-reduce / D2H read
        self.hooked = False
        self.direct = False                                   # fused exchange: dW leaves backward final, no copy into grad_buf
        self.last_dw = None
        for c in self.clouds:
            res = self.rulebook(c)
            c["m"] = res[0].shape[0]
            c["pairs_total"] = int((res[2] >= 0).sum().item())
            g = torch.Generator(device=ctx.dev).manual_seed(7)
            c["dout"] = (torch.rand((c["m"], self.K), device=ctx.dev, generator=g) * 0.4 - 0.2).to(self.tdt)

    def rulebook(self, c, **kw):
        return self.ctx.ops.get_indice_pairs_implicit_gemm(c["d_inds"], self.batch, self.wl["shape"], self.algo, self.ks,
                                                           self.st, self.pd, self.dl, [0] * 3, self.wl["subm"], False,
                                                           is_train=True, **kw)

    def conv_fwd_bwd(self, c, res, weight, kw):
        ops = self.ctx.ops
        out_inds, _, pair_fwd, pair_bwd, mask_fwd, mask_bwd, sort_fwd, sort_bwd, masks = res
        out, mask_out, mw = ops.implicit_gemm(c["d_feats"], weight, pair_fwd, mask_fwd, sort_fwd, out_inds.shape[0],
                                              masks, True, self.wl["subm"], **kw)
        din, dw = ops.implicit_gemm_backward(c["d_feats"], weight, c["dout"], pair_fwd, pair_bwd, mask_fwd, mask_bwd,
                                             sort_fwd, sort_bwd, mask_out, masks, mw, self.wl["subm"], **kw)
        if self.record_outputs:
            c["outputs"] = {"out_indices": out_inds, "out_features": out, "input_grad": din, "weight_grad": dw}
        return out, din, dw

    def device_step(self, c, timer=None, calls=1):
        """rulebook -> (forward -> backward) x calls on device-resident inputs (operator layer);
        calls = 2 is the indice_key-reuse leg: one rulebook serves two layers."""
        kw = {} if timer is None else {"timer": timer}
        res = self.rulebook(c, **kw)
        dw = None
        for j in range(calls):
            _, _, dw = self.conv_fwd_bwd(c, res, self.weight if j == 0 else self.weight2, kw)
        self.keep(dw)
        return dw

    def compute(self, c, res):
        """forward + backward on an already built rulebook (the second stage of the pipelined replay)"""
        _, _, dw = self.conv_fwd_bwd(c, res, self.weight, {})
        self.keep(dw)

    def keep(self, dw):
        """what the step's all-reduce / D2H read: the gradient buffer, or (fused exchange) the reduced dW itself"""
        if self.direct:
            self.last_dw = dw
        elif not self.hooked:
            self.grad_buf.copy_(dw)

    def install_allreduce_hook(self):
        """N > 1: dW is copied into the gradient buffer and all-reduced on a forked stream right after the
        weight-gradient kernel, beside the input-gradient kernel of the same step (ops.set_wgrad_hook)."""
        dist = self.ctx.dist

        def hook(dw):
            self.grad_buf.copy_(dw)
            dist.all_reduce(self.grad_buf)
        self.ctx.ops.set_wgrad_hook(hook)
        self.hooked = True

    def grads(self):
        return self.last_dw if self.direct and self.last_dw is not None else self.grad_buf

    def make_input(self, d_inds, d_feats):
        return self.ctx.spconv.SparseConvTensor(d_feats.detach().requires_grad_(True), d_inds, self.wl["shape"],
                                                self.batch)

    def e2e_from_input(self, x):
        self.layer.weight.grad = None
        y = self.layer(x)
        loss = y.features.square().mean(dtype=self.ctx.torch.float32)
        loss.backward()
        self.keep(self.layer.weight.grad)
        return loss

    def config(self):
        c0 = self.clouds[0]
        return {"grid": self.wl["shape"], "active_voxels_per_gpu": int(self.n_per_step), "outputs": int(c0["m"]),
                "pairs_per_voxel": round(c0["pairs_total"] / c0["n"], 2), "c_in": self.C, "c_out": self.K,
                "step": ("subm" if self.wl["subm"] else "regular-conv") +
                        " rulebook (hash + probe/rank + mask sort + tile table) + fwd + dgrad + wgrad"}

    def roofline_terms(self, kind):
        c0 = self.clouds[0]
        return (algorithmic_bytes(kind, c0["n"], c0["m"], self.C, self.K, self.kv, self.elem),
                conv_flops(c0["pairs_total"], self.C, self.K))


class EncoderWorkload(Workload):
    """BASELINE configs[2]: SubM16 x2 (one indice_key) -> SparseConv 16->32 s2 -> SubM32 ->
    SparseConv 32->64 s2 -> SparseConv 64->128 s2, fp16 forward + backward through the public
    module API (the regular convs read their output count back, so the step is not graph-captured)."""

    def setup(self):
        ctx, torch = self.ctx, self.ctx.torch
        from spconv_b200.pytorch.dist import GradBucket
        self.make_clouds(16)
        torch.manual_seed(48848)
        self.layers = [m.to(ctx.dev).to(self.tdt) for m in make_encoder6(ctx.spconv)]
        for m in self.layers:
            m.train()
        self.bucket = GradBucket([m.weight for m in self.layers])
        # every layer's rulebook (the strided ones included) is built ahead of the step that uses it,
        # on the side stream, by a worker thread: the output-count read-backs of the three regular
        # convs then wait for rulebook kernels only, never for the GEMM queue of the training stream.
        # (--pipeline 3 only: measured SLOWER than the plain eager step, 2.01 vs 1.69 ms -- the worker thread's
        # Python competes with the training thread for the GIL; profiles/README.md session f)
        self.pipelined = int(ctx.args.pipeline) >= 3
        self.prefetcher = ctx.spconv.RulebookPrefetcher(self.layers if self.pipelined else [self.layers[0]], stream=ctx.side,
                                                        background=self.pipelined)
        self.staged = {}
        self.layer_stats = None

    def make_input(self, d_inds, d_feats, timer=None):
        x = self.ctx.spconv.SparseConvTensor(d_feats.detach().requires_grad_(True), d_inds, self.wl["shape"], self.batch,
                                             enable_timer=timer is not None)
        if timer is not None:
            x._timer = timer
        return x

    def e2e_from_input(self, x):
        return self.forward_backward(None, None, x=x)

    def forward_backward(self, d_inds, d_feats, timer=None, x=None):
        torch = self.ctx.torch
        if x is None:
            x = self.make_input(d_inds, d_feats, timer)
        self.bucket.zero()
        acts = [x]
        for li, m in enumerate(self.layers):
            if timer is not None:
                with timer.namespace(f"L{li}"):
                    acts.append(m(acts[-1]))
            else:
                acts.append(m(acts[-1]))
        loss = acts[-1].features.square().mean(dtype=torch.float32)
        loss.backward()
        if self.record_outputs:
            self.last_outputs = {"out_indices": acts[-1].indices, "out_features": acts[-1].features.detach(),
                                 "loss": loss.detach(), "input_grad": acts[0].features.grad, "weight_grads": self.bucket.flat}
        if self.layer_stats is None:
            self.layer_stats = [(int(a.features.shape[0]), int(b.features.shape[0])) for a, b in zip(acts[:-1], acts[1:])]
            self.pairs = []
            for (kind, ci, co, key), b in zip(ENCODER6_LAYERS, acts[1:]):
                self.pairs.append(int((b.indice_dict[key].pair_fwd >= 0).sum().item()))
        return loss

    def device_step(self, c, timer=None):
        if timer is not None or not self.pipelined:
            self.forward_backward(c["d_inds"], c["d_feats"], timer)
            return self.bucket.flat
        # rulebooks one cloud ahead: this step consumes the chain staged by the previous step (or builds
        # it now, first step of a loop) and starts the next cloud's chain before issuing its own GEMMs.
        # Each timed step = one full 5-rulebook chain + one 6-layer forward + backward.
        ci = next(j for j, cj in enumerate(self.clouds) if cj is c)
        x = self.staged.pop(ci, None)
        if x is None:
            x = self.prefetcher.prefetch(self.make_input(c["d_inds"], c["d_feats"]), wait_current=False)
        nxt = (ci + 1) % len(self.clouds)
        cn = self.clouds[nxt]
        self.staged[nxt] = self.prefetcher.prefetch(self.make_input(cn["d_inds"], cn["d_feats"]), wait_current=False)
        self.forward_backward(None, None, x=self.prefetcher.ready(x))
        return self.bucket.flat

    def grads(self):
        return self.bucket.flat

    def outputs(self, c):
        return self.last_outputs                 # eager steps only: the last forward_backward is the last step

    def config(self):
        return {"grid": self.wl["shape"], "batch_per_gpu": self.batch, "active_voxels_per_gpu": int(self.n_per_step),
                "layers": [f"{k}{ci}->{co}" for k, ci, co, _ in ENCODER6_LAYERS],
                "voxels_in_out_per_layer": self.layer_stats,
                "step": "5 rulebooks (SubM16 pair shared via indice_key) + 6 x (fwd + dgrad + wgrad) through "
                        "SparseConvTensor / SubMConv3d / SparseConv3d + autograd"}

    def roofline_terms_layer(self, li, kind):
        _, ci, co, _ = ENCODER6_LAYERS[li]
        n_in, n_out = self.layer_stats[li]
        return algorithmic_bytes(kind, n_in, n_out, ci, co, 27, self.elem), conv_flops(self.pairs[li], ci, co)


class Int8Workload(Workload):
    """BASELINE configs[4]: int8 SubMConv3d inference (rulebook + int8 implicit GEMM with the
    per-channel scale / bias / clip epilogue, test/test_all_algo.py:272-287)."""
    inference = True
    graphable = True

    def setup(self):
        ctx, wl, torch = self.ctx, self.wl, self.ctx.torch
        from spconv_b200.core import ConvAlgo
        self.algo = ConvAlgo.MaskImplicitGemm
        self.C, self.K, self.kv = wl["c_in"], wl["c_out"], 27
        self.make_clouds(self.C)
        g = torch.Generator().manual_seed(5)
        self.weight = torch.randint(-127, 128, (self.K, 3, 3, 3, self.C), generator=g, dtype=torch.int8).to(ctx.dev)
        self.scale = (torch.rand(self.K, generator=g) * 2e-3 + 1e-4).to(ctx.dev)      # per-channel quant scale
        self.bias = (torch.rand(self.K, generator=g) - 0.5).to(ctx.dev)
        for c in self.clouds:
            res = self.rulebook(c)
            c["m"] = res[0].shape[0]
            c["pairs_total"] = int((res[2] >= 0).sum().item())
        self.h_out = torch.empty((max(c["n"] for c in self.clouds), self.K), dtype=torch.int8).pin_memory()

    def rulebook(self, c, **kw):
        return self.ctx.ops.get_indice_pairs_implicit_gemm(c["d_inds"], 1, self.wl["shape"], self.algo, [3] * 3, [1] * 3,
                                                           [1] * 3, [1] * 3, [0] * 3, True, False, is_train=False, **kw)

    def compute(self, c, res):
        return self.conv(c["d_feats"], res, {}, c)

    def run(self, d_inds, d_feats, c, kw):
        res = self.ctx.ops.get_indice_pairs_implicit_gemm(d_inds, 1, self.wl["shape"], self.algo, [3] * 3, [1] * 3,
                                                          [1] * 3, [1] * 3, [0] * 3, True, False, is_train=False, **kw)
        return self.conv(d_feats, res, kw, c)

    def conv(self, d_feats, res, kw, c=None):
        from spconv_b200.core import Activation
        out_inds, _, pair_fwd, _, mask_fwd, _, sort_fwd, _, masks = res
        out, _, _ = self.ctx.ops.implicit_gemm(d_feats, self.weight, pair_fwd, mask_fwd, sort_fwd, out_inds.shape[0], masks,
                                               False, True, bias=self.bias, act_type=Activation.ReLU, scale=self.scale,
                                               output_dtype=self.ctx.torch.int8, **kw)
        if c is not None and self.record_outputs:
            c["outputs"] = {"out_indices": out_inds, "out_features": out}
        return out

    def device_step(self, c, timer=None):
        return self.run(c["d_inds"], c["d_feats"], c, {} if timer is None else {"timer": timer})

    def make_input(self, d_inds, d_feats):
        return (d_inds, d_feats)

    def e2e_from_input(self, x):
        return self.run(x[0], x[1], None, {})

    def config(self):
        c0 = self.clouds[0]
        return {"grid": self.wl["shape"], "active_voxels_per_gpu": int(self.n_per_step),
                "pairs_per_voxel": round(c0["pairs_total"] / c0["n"], 2), "c_in": self.C, "c_out": self.K,
                "step": "subm rulebook + int8 tcgen05 (kind::i8) forward, per-channel scale + bias + ReLU + clip to int8"}

    def roofline_terms(self, kind):
        c0 = self.clouds[0]
        return (algorithmic_bytes("fwd", c0["n"], c0["m"], self.C, self.K, self.kv, 1),
                conv_flops(c0["pairs_total"], self.C, self.K))


def make_workload(name, ctx) -> Workload:
    kind = WORKLOADS[name]["kind"]
    return {"layer": LayerWorkload, "encoder": EncoderWorkload, "int8": Int8Workload}[kind](name, ctx)


# ============================================================================ GPU arm: measurement
def measure(w: Workload, ctx: Ctx, steps: int, warmup: int, headline: bool, dump_dir: Optional[str] = None) -> dict:
    """Times one workload: value (device-resident), e2e (graph when possible + eager), per-region
    kernel times and the roofline of the dominant GEMM region.  Returns a dict of results reduced
    over ranks (max time, sum voxels).  ``dump_dir``: where rank 0 writes the outputs of the last timed
    step of ``value`` (see write_outputs)."""
    torch, dist, ops = ctx.torch, ctx.dist, ctx.ops
    from spconv_b200.pytorch.core import CUDAKernelTimer
    w.setup()
    w.record_outputs = dump_dir is not None and ctx.rank == 0
    world = ctx.world
    clouds = w.clouds
    train = not w.inference
    fused_ar = train and ctx.peers is not None and (headline or not ctx.allreduce_auto)
    if fused_ar:
        ops.set_peer_group(ctx.peers)            # every dW leaves its kernel already summed over the ranks

    elif world > 1 and train and hasattr(w, "install_allreduce_hook"):
        w.install_allreduce_hook()               # all-reduce(dW) beside the input gradient of the same step
    explicit_ar = world > 1 and train and not fused_ar and not getattr(w, "hooked", False)
    if hasattr(w, "direct"):
        # nothing reads a separate gradient buffer unless NCCL reduces it: the step's dW itself is what the D2H of the
        # e2e legs reads (autograd does the same: the first accumulation takes the tensor, it does not copy it)
        w.direct = train and not explicit_ar and not getattr(w, "hooked", False)

    # ---------------- warm-up (also configures kernels / NCCL before any graph capture)
    for i in range(max(warmup, 3)):
        w.device_step(clouds[i % NUM_CLOUDS])
        if explicit_ar:
            ctx.allreduce(w.grads())
    torch.cuda.synchronize()

    # ---------------- CUDA graphs of the device-resident step (one per cloud).  At N > 1 the
    # all-reduce of the PREVIOUS step's gradient buffer is a parallel branch of the graph: it
    # overlaps the rulebook generation of this step (which does not depend on weights) and is
    # joined before the forward pass -- exactly where an optimizer update would consume it.
    graphs = None
    graph_outs = pipe_outs = None                # per cloud: the output tensors of its captured graph
    use_graph = bool(ctx.args.graph) and w.graphable
    if use_graph:
        try:
            graphs = []
            for c in clouds:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    if explicit_ar:
                        main = torch.cuda.current_stream()
                        ctx.side.wait_stream(main)
                        with torch.cuda.stream(ctx.side):
                            dist.all_reduce(w.grads())
                        res = w.rulebook(c)
                        main.wait_stream(ctx.side)
                        _, _, dw = w.conv_fwd_bwd(c, res, w.weight, {})
                        w.grad_buf.copy_(dw)
                    else:
                        w.device_step(c)
                graphs.append(g)
            torch.cuda.synchronize()
            graph_outs = [c.get("outputs") for c in clouds]
        except Exception as e:                       # capture is an optimisation, never a requirement
            print(f"[bench] CUDA-graph capture failed ({type(e).__name__}: {e}); running eagerly", file=sys.stderr)
            graphs, use_graph = None, False
            torch.cuda.synchronize()

    # ---------------- software-pipelined replay (the default `value`): the rulebook depends only on the
    # coordinates, never on weights or features, so -- like a data loader prefetching the next batch --
    # the rulebook of cloud i+1 is generated on a side stream WHILE cloud i runs forward + backward.
    # Every timed step still contains exactly one rulebook generation and one fwd + dgrad + wgrad
    # (+ the all-reduce of the previous step's dW at N > 1, placed before the forward pass where an
    # optimizer would consume it); both streams are joined before the step's end event.
    pipe = None
    if use_graph and bool(ctx.args.pipeline) and hasattr(w, "compute"):
        try:
            rb_graphs, ge_graphs, rb_out = [], [], []
            for c in clouds:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    rb_out.append(w.rulebook(c))
                rb_graphs.append(g)
            for c, res in zip(clouds, rb_out):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    if explicit_ar:
                        dist.all_reduce(w.grads())
                    w.compute(c, res)
                ge_graphs.append(g)
            for g in rb_graphs:                      # every rulebook resident once before the first timed step
                g.replay()
            torch.cuda.synchronize()
            pipe = (rb_graphs, ge_graphs)
            pipe_outs = [c.get("outputs") for c in clouds]
        except Exception as e:
            print(f"[bench] pipelined capture failed ({type(e).__name__}: {e}); serial graph replay", file=sys.stderr)
            pipe = None
            torch.cuda.synchronize()

    def serial_step(i):
        graphs[i % NUM_CLOUDS].replay()

    depth2 = pipe is not None and int(ctx.args.pipeline) >= 2
    sides = [ctx.side, ctx.side2]
    ge_done = [torch.cuda.Event() for _ in range(NUM_CLOUDS)]

    def value_step(i):
        j = i % NUM_CLOUDS
        if depth2:
            # rulebooks run TWO clouds ahead, alternating between two side streams: the rulebook of
            # cloud i was replayed on sides[i % 2] at step i-2; this step waits for it, then queues the
            # rulebook of cloud i+2 behind it.  No join at the end of the step -- a rulebook that is the
            # bottleneck shows up as the wait at the head of the step that needs it.
            main = torch.cuda.current_stream()
            sd = sides[i % 2]
            main.wait_stream(sd)
            jn = (i + 2) % NUM_CLOUDS
            sd.wait_event(ge_done[jn])                          # the last reader of that cloud's rulebook buffers
            with torch.cuda.stream(sd):
                pipe[0][jn].replay()
            pipe[1][j].replay()
            ge_done[j].record(main)
        elif pipe is not None:
            main = torch.cuda.current_stream()
            ctx.side.wait_stream(main)
            with torch.cuda.stream(ctx.side):
                pipe[0][(i + 1) % NUM_CLOUDS].replay()          # rulebook of the NEXT cloud
            pipe[1][j].replay()                                 # fwd + bwd of this cloud
            main.wait_stream(ctx.side)
        elif use_graph:
            graphs[j].replay()
        else:
            w.device_step(clouds[j])
            if explicit_ar:
                ctx.allreduce(w.grads())

    # ---------------- e2e: public module API from pinned host buffers
    # Every step copies this step's coordinates + features H2D, runs the module(s) + loss + backward
    # and reads the loss and the weight gradients (inference: the int8 output) back to the host.
    h_loss = torch.zeros((), dtype=torch.float32).pin_memory()
    h_grads = torch.zeros_like(w.grads(), device="cpu").pin_memory() if train else None

    def d2h(result):
        if train:
            h_loss.copy_(result.detach(), non_blocking=True)
            h_grads.copy_(w.grads(), non_blocking=True)
        else:
            w.h_out[:result.shape[0]].copy_(result, non_blocking=True)

    def e2e_step_eager(i):
        c = clouds[i % NUM_CLOUDS]
        d_inds = c["h_inds"].to(ctx.dev, non_blocking=True)
        d_feats = c["h_feats"].to(ctx.dev, non_blocking=True)
        result = w.e2e_body(d_inds, d_feats)
        if explicit_ar:
            ctx.allreduce(w.grads())
        d2h(result)

    # The same loop as a user would pipeline it WITHOUT graphs: while cloud i runs forward + backward on
    # the current stream, the side stream copies cloud i+1 H2D into the other device buffer and
    # prefetches its input-level SubM rulebook (spconv.RulebookPrefetcher).  Every timed step still
    # holds one full H2D, one rulebook generation, one fwd + bwd and the D2H of its results.
    n_max = max(c["n"] for c in clouds)
    ebufs = [dict(inds=torch.empty((n_max, 4), dtype=torch.int32, device=ctx.dev),
                  feats=torch.empty((n_max, clouds[0]["h_feats"].shape[1]), dtype=clouds[0]["h_feats"].dtype,
                                    device=ctx.dev)) for _ in range(2)]
    ev_ready = [torch.cuda.Event(), torch.cuda.Event()]
    ev_done = [torch.cuda.Event(), torch.cuda.Event()]
    staged = [dict(cloud=-1, x=None), dict(cloud=-1, x=None)]

    def stage(k, ci):
        c = clouds[ci]
        ctx.side.wait_event(ev_done[k])              # the step that last used buffer k has been issued before
        with torch.cuda.stream(ctx.side):
            ebufs[k]["inds"][:c["n"]].copy_(c["h_inds"], non_blocking=True)
            ebufs[k]["feats"][:c["n"]].copy_(c["h_feats"], non_blocking=True)
            x = w.make_input(ebufs[k]["inds"][:c["n"]], ebufs[k]["feats"][:c["n"]])
            if w.prefetcher is not None:
                w.prefetcher.prefetch(x)
            ev_ready[k].record(ctx.side)
        staged[k] = dict(cloud=ci, x=x)

    def e2e_step_eager_pipe(i):
        k, ci = i % 2, i % NUM_CLOUDS
        if staged[k]["cloud"] != ci:                 # first step of a loop: nothing was prefetched for it
            stage(k, ci)
        stage((i + 1) % 2, (i + 1) % NUM_CLOUDS)
        main = torch.cuda.current_stream()
        main.wait_event(ev_ready[k])
        x = staged[k]["x"]
        if w.prefetcher is not None:
            w.prefetcher.ready(x)
        result = w.e2e_from_input(x)
        if explicit_ar:
            ctx.allreduce(w.grads())
        d2h(result)
        ev_done[k].record(main)

    for i in range(3):
        e2e_step_eager(i)
    for i in range(4):
        e2e_step_eager_pipe(i)
    torch.cuda.synchronize()

    # Graph-captured e2e step with double buffering: the replay of step i computes on device buffer
    # i%2 and, on a forked stream inside the same graph, copies the NEXT cloud H2D into buffer
    # (i+1)%2 -- every timed step still contains one full H2D of a step's inputs and the D2H of its
    # results, but the copy overlaps the kernels.
    e2e_graphs = None
    if use_graph:
        try:
            n_max = max(c["n"] for c in clouds)
            c_in = clouds[0]["h_feats"].shape[1]
            bufs = [dict(inds=torch.empty((n_max, 4), dtype=torch.int32, device=ctx.dev),
                         feats=torch.empty((n_max, c_in), dtype=clouds[0]["h_feats"].dtype, device=ctx.dev))
                    for _ in range(2)]
            e2e_graphs = []
            for j, c in enumerate(clouds):
                cur, nxt = bufs[j % 2], bufs[(j + 1) % 2]
                cn = clouds[(j + 1) % NUM_CLOUDS]
                cur["inds"][:c["n"]].copy_(c["h_inds"])
                cur["feats"][:c["n"]].copy_(c["h_feats"])
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    main = torch.cuda.current_stream()
                    ctx.side.wait_stream(main)
                    with torch.cuda.stream(ctx.side):
                        nxt["inds"][:cn["n"]].copy_(cn["h_inds"], non_blocking=True)
                        nxt["feats"][:cn["n"]].copy_(cn["h_feats"], non_blocking=True)
                    result = w.e2e_body(cur["inds"][:c["n"]], cur["feats"][:c["n"]])
                    if explicit_ar:
                        dist.all_reduce(w.grads())
                    d2h(result)
                    main.wait_stream(ctx.side)
                e2e_graphs.append(g)
            torch.cuda.synchronize()
            # prologue: cloud 0 must be resident in buffer 0 before the first replay
            bufs[0]["inds"][:clouds[0]["n"]].copy_(clouds[0]["h_inds"])
            bufs[0]["feats"][:clouds[0]["n"]].copy_(clouds[0]["h_feats"])
            torch.cuda.synchronize()
        except Exception as e:
            print(f"[bench] e2e CUDA-graph capture failed ({type(e).__name__}: {e}); e2e runs eagerly", file=sys.stderr)
            e2e_graphs = None
            torch.cuda.synchronize()

    def e2e_step(i):
        if e2e_graphs is None:                      # not capturable: the pipelined eager loop IS the e2e path
            return e2e_step_eager_pipe(i)
        e2e_graphs[i % NUM_CLOUDS].replay()

    # kernels of THIS library per step (graph replays re-issue exactly the captured launches)
    ops.launch_count(reset=True)
    w.device_step(clouds[0])
    launches_per_step = ops.launch_count(reset=True)
    torch.cuda.synchronize()

    sampler = ClockSampler(ctx.local_rank)
    if ctx.rank == 0 and headline:
        sampler.start()
    # three repetitions of the K-step timed region; the median repetition is reported (one region of
    # 20 x 0.15 ms is a thin sample)
    if pipe is not None:
        for i in range(2 * NUM_CLOUDS):
            value_step(i)
    runs = [float(np.mean(ctx.timed_loop(value_step, steps))) for _ in range(3)]
    ms_value = sorted(runs)[1]
    dumped = None
    if w.record_outputs:
        # the last timed step ran cloud j.  A graph replay rewrites the tensors captured with the graph that
        # value_step replays (eager steps outside the timed loop record other tensors); an eager timed step
        # recorded its own.  Host copy now: the legs below run the same clouds again.
        j = (steps - 1) % NUM_CLOUDS
        outs = pipe_outs[j] if pipe is not None else graph_outs[j] if use_graph else w.outputs(clouds[j])
        dumped = {k: t.detach().cpu() for k, t in outs.items()}
        w.record_outputs = False
    ms_serial = float(np.mean(ctx.timed_loop(serial_step, steps))) if pipe is not None else None
    ms_e2e = float(np.mean(ctx.timed_loop(e2e_step, steps)))
    clocks = sampler.stop() if (ctx.rank == 0 and headline) else {}
    # The eager legs are host-bound: 20 steps are ~12 ms of wall clock, one scheduling hiccup (or the clock sampler
    # forking nvidia-smi, hence stopped above: it covers the device-timed legs) doubles the mean.  Median of three
    # repetitions, as for `value`.
    ms_e2e_naive = sorted(float(np.mean(ctx.timed_loop(e2e_step_eager, steps))) for _ in range(3))[1]
    ms_e2e_eager = sorted(float(np.mean(ctx.timed_loop(e2e_step_eager_pipe, steps))) for _ in range(3))[1]

    # indice_key-reuse leg (configs[3]): one rulebook, two layers
    ms_reuse = None
    if isinstance(w, LayerWorkload) and w.wl.get("reuse_calls"):
        calls = int(w.wl["reuse_calls"])
        for i in range(3):
            w.device_step(clouds[i % NUM_CLOUDS], calls=calls)
        ms_reuse = float(np.mean(ctx.timed_loop(lambda i: w.device_step(clouds[i % NUM_CLOUDS], calls=calls), steps)))

    # ---------------- per-kernel timing for the roofline (events around every C-ABI region)
    reps = max(5, min(steps, 12))
    samples: Dict[str, List[float]] = {}
    for i in range(reps):
        timer = CUDAKernelTimer(True)
        ctx.flush.zero_()
        # a ~0.5 ms device-side spin lets the host queue work ahead of the GPU, so the events bracket
        # back-to-back kernels and not the host's launch latency
        torch.cuda._sleep(1_000_000)
        w.device_step(clouds[i % NUM_CLOUDS], timer)
        for k, v in timer.get_all_pair_time().items():
            samples.setdefault(k, []).append(v)
    regions = {k: float(np.median(v)) for k, v in samples.items()}

    # ---------------- reduce over ranks (max time, sum voxels)
    t = torch.tensor([ms_value, ms_e2e, ms_e2e_eager, ms_reuse or 0.0, ms_serial or 0.0, ms_e2e_naive], device=ctx.dev,
                     dtype=torch.float64)
    n_total = torch.tensor([w.n_per_step], device=ctx.dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(n_total, op=dist.ReduceOp.SUM)
    ms_value, ms_e2e, ms_e2e_eager, ms_reuse_r, ms_serial_r, ms_e2e_naive = (float(v) for v in t)
    voxels = float(n_total[0])

    res = {
        "value": voxels / (ms_value * 1e-3), "ms_per_step": ms_value, "ms_per_step_runs": [round(r, 5) for r in runs],
        "voxels_per_step": voxels, "cuda_graph": use_graph, "launches_per_step": int(launches_per_step),
        "pipelined": (2 if depth2 else 1) if pipe is not None else 0,
        "serial_ms_per_step": ms_serial_r if pipe is not None else None,
        "e2e": {"value": voxels / (ms_e2e * 1e-3), "unit": "voxels/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": w.h2d_bytes(),
                "d2h_bytes_per_step": int(h_grads.numel() * h_grads.element_size() + 4) if train
                else int(clouds[0]["n"] * w.K),
                "api": "SparseConvTensor -> module forward -> loss.backward (pinned host in, loss + dW out)" if train
                else "ops.get_indice_pairs_implicit_gemm + ops.implicit_gemm int8 (pinned host in, int8 features out)",
                "cuda_graph": e2e_graphs is not None,
                "overlap": "H2D of the next cloud on a forked stream inside the step's graph"
                if e2e_graphs is not None else "none",
                # no graphs, public API only.  Two loops are timed: "naive" (copy, compute, read back, one stream)
                # and "prefetch" (H2D of the next cloud + RulebookPrefetcher on a side stream beside this cloud's
                # fwd + bwd).  Both are host-bound at this size, so which one wins depends on the box's CPU.
                "eager_value": voxels / (min(ms_e2e_eager, ms_e2e_naive) * 1e-3),
                "eager_ms_per_step": min(ms_e2e_eager, ms_e2e_naive),
                "eager_variant": "prefetch" if ms_e2e_eager <= ms_e2e_naive else "naive",
                "eager_prefetch_ms_per_step": ms_e2e_eager, "eager_naive_ms_per_step": ms_e2e_naive},
        "clocks": clocks,
        "kernel_ms": {k: round(v, 4) for k, v in sorted(regions.items())},
        # rulebook generation (hash / rank / mask sort / tile tables) vs the GEMM kernels, summed over the layers;
        # a rulebook shared through an indice_key is built once and so counted once
        "kernel_ms_summary": {
            "rulebook": round(sum(v for k, v in regions.items() if "gen_" in k or "tile_table" in k), 4),
            "gemm_fwd": round(sum(v for k, v in regions.items() if k.split(".")[-1] in ("implicit_gemm", "implicit_gemm_int8")), 4),
            "gemm_bwd": round(sum(v for k, v in regions.items() if k.split(".")[-1] in ("implicit_gemm_dgrad", "implicit_gemm_wgrad")), 4)},
        "config": w.config(),
    }
    if ms_reuse is not None:
        calls = int(w.wl["reuse_calls"])
        res["indice_key_reuse"] = {"calls": calls, "ms_per_step": ms_reuse_r,
                                   "value_per_call": voxels * calls / (ms_reuse_r * 1e-3),
                                   "note": "one rulebook + tile tables, then fwd+bwd of two layers that share it"}
    res["roofline"] = roofline_of(w, regions)
    res["allreduce"] = ("fused: tail of the weight-gradient reduction kernel (fp32 slices pushed to every rank's exchange "
                        "buffer over NVLink peer memory, summed locally in rank order; csrc/peer.cu)" if fused_ar else
                        "NCCL hook: right after the weight-gradient kernel, beside the input gradient (ops.set_wgrad_hook)"
                        if getattr(w, "hooked", False) else ("NCCL: one flat bucket after backward" if explicit_ar else "none"))
    ops.set_wgrad_hook(None)
    ops.set_peer_group(None)
    if dumped is not None:
        write_outputs(dump_dir, dumped)
    return res


def write_outputs(path: str, outputs: dict) -> None:
    """``path/<name>.npy`` in float32 (float64 stays float64).  When the arrays exceed DUMP_BYTES, every array
    keeps the same fraction of its rows, chosen by a fixed seed (identical rows from run to run)."""
    arrays = {name: (t if str(t.dtype) == "torch.float64" else t.float()).numpy() for name, t in outputs.items()}
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_BYTES and a.ndim > 0 and a.shape[0] > 1:
            keep = max(1, a.shape[0] * DUMP_BYTES // total)
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(path, f"{name}.npy"), a)


def roofline_of(w: Workload, regions: Dict[str, float]) -> Optional[dict]:
    """Algorithmic bytes of the slowest GEMM region / its event time / measured HBM peak."""
    peaks = load_peaks()
    name_map = {"implicit_gemm": "fwd", "implicit_gemm_dgrad": "dgrad", "implicit_gemm_wgrad": "wgrad",
                "implicit_gemm_int8": "fwd"}
    cand = {}
    for k, ms in regions.items():
        leaf = k.split(".")[-1]
        if leaf not in name_map:
            continue
        kind = name_map[leaf]
        if isinstance(w, EncoderWorkload):
            li = int(k.split(".")[0][1:])
            b, f = w.roofline_terms_layer(li, kind)
        else:
            b, f = w.roofline_terms(kind)
        agg = cand.setdefault(kind, {"bytes": 0, "flops": 0, "ms": 0.0})
        agg["bytes"] += b
        agg["flops"] += f
        agg["ms"] += ms
    if not cand:
        return None
    kind = max(cand, key=lambda k: cand[k]["ms"])
    a = cand[kind]
    achieved = a["bytes"] / (a["ms"] * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(w.name, {}).get(kind)
        except Exception:
            traffic = None
    fwd = cand.get("fwd")
    out = {"bound": "hbm", "kernel": "tc_wgrad (+ wgrad_reduce)" if kind == "wgrad" else f"tc_gather_gemm/{kind}",
           "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
           "traffic": traffic,
           "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks["source"] == "measured"
           else "fallback (B200_PROFILING.md)",
           "algorithmic_bytes": int(a["bytes"]), "launch_ms": a["ms"],
           "per_kind": {k: {"ms": round(v["ms"], 4), "GBps": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1),
                            "frac": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9 / peaks["hbm_gbs"], 4)}
                        for k, v in cand.items()}}
    if fwd:
        out["tensor_tflops_fwd"] = fwd["flops"] / (fwd["ms"] * 1e-3) / 1e12
        out["tensor_frac_fwd"] = out["tensor_tflops_fwd"] / peaks["bf16_tflops"]
    return out


def run_ours(args):
    ctx = Ctx(args)
    world, rank = ctx.world, ctx.rank
    extras = args.extras if args.extras >= 0 else int(args.workload == DEFAULT_WORKLOAD)
    head = measure(make_workload(args.workload, ctx), ctx, args.steps, args.warmup, True, args.dump_outputs)
    others = {}
    if extras:
        # at N > 1 only the encoder (BASELINE configs[2] is the multi-GPU config) rides along: every
        # extra workload is another chance for one rank to fail inside a collective
        for name in (EXTRA_WORKLOADS if world == 1 else EXTRA_WORKLOADS[:1]):
            if name == args.workload:
                continue
            ctx.torch.cuda.empty_cache()
            try:
                r = measure(make_workload(name, ctx), ctx, max(5, min(args.steps, 10)), 3, False)
                others[name] = {"metric": metric_name(name), "unit": "voxels/s", "dtype": WORKLOADS[name]["dtype"], **r}
                others[name].pop("clocks", None)
            except Exception as e:                   # an extra workload must never take the headline down
                others[name] = {"error": f"{type(e).__name__}: {e}"}
                ctx.torch.cuda.synchronize()
    if rank == 0:
        wl = WORKLOADS[args.workload]
        line = {
            "metric": metric_name(args.workload), "value": head["value"], "unit": "voxels/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": head["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": wl["dtype"],
            "data": "synthetic",
            "config": {"workload": args.workload, **head["config"],
                       "parallelism": f"dp{world} (one batch per GPU)" + (
                           "; NCCL all-reduce(dW) captured inside the step: launched right after the weight-gradient "
                           "kernel on a forked stream, beside the input-gradient kernel"
                           if world > 1 and head["cuda_graph"] else ("; NCCL all-reduce(dW) per step" if world > 1 else "")),
                       "cuda_graph": head["cuda_graph"], "debug_bits": int(args.debug_bits),
                       "pipeline": (("rulebooks two clouds ahead on two alternating side streams (one rulebook + one "
                                     "fwd/dgrad/wgrad per timed step; a step waits for its own rulebook); "
                                     if head.get("pipelined") == 2 else
                                     "rulebook of cloud i+1 on a side stream beside fwd + bwd of cloud i (one rulebook + one "
                                     "fwd/dgrad/wgrad per timed step, streams joined before the end event); ") +
                                    f"serial replay of the same step: {head['serial_ms_per_step']:.4f} ms")
                       if head.get("pipelined") else "none",
                       "l2": f"{L2_FLUSH_BYTES >> 20} MiB buffer written between timed steps; {NUM_CLOUDS} rotating clouds",
                       "timing": "median of 3 repetitions of the K-step timed region (ms_per_step_runs)"},
            "ms_per_step_runs": head["ms_per_step_runs"],
            "serial_ms_per_step": head.get("serial_ms_per_step"),
            "e2e": head["e2e"],
            "gpu_launches": int(head["launches_per_step"] * args.steps),
            "clocks": head["clocks"],
            "kernel_ms": head["kernel_ms"],
            "kernel_ms_summary": head["kernel_ms_summary"],
            "allreduce": head["allreduce"],
            "roofline": head["roofline"],
        }
        if "indice_key_reuse" in head:
            line["indice_key_reuse"] = head["indice_key_reuse"]
        if others:
            line["workloads"] = others
        if world == 1:                               # bounded CPU-baseline sample, rank 0 at N = 1 only
            cb, _, _, _ = cpu_arm(wl, args.cpu_sample, 2, 12, 10.0)
            line["cpu_baseline"] = cb
        else:
            line["cpu_baseline"] = {"value": None, "unit": "voxels/s", "cores": 0, "kind": "reference",
                                    "sample": "timed at N = 1 only (see the N = 1 line / --impl reference)"}
        print(json.dumps(line), flush=True)
    if world > 1:
        ctx.dist.barrier()
        ctx.dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
