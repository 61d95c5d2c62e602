#!/usr/bin/env python
"""bench.py -- surfel-rasterizer forward+backward frames/s at 512x512 / 300 K surfels (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A STEP = one pass of the hot path over one batch: every rank rasterizes `--frames-per-step` frames (forward +
backward, each frame a different camera), accumulates the surfel gradients, and -- for N > 1 -- joins ONE NCCL
all-reduce of the flat gradient buffer (frames are the shard axis; weak scaling: per-GPU work is fixed).
Ours: the F frames of a step are ONE batched launch set (sr_forward_batch / sr_backward_batch: every kernel has a frame
dimension), captured in a CUDA graph; `--mode streams` keeps round 1's harness (F single-frame calls over S streams).
Both arms of ours alternate between two captures of the step, so that the host checks step k-1 (overflow words; in the e2e
arm also the loss read-back) only after it has queued step k.  In the value arm, for N > 1, step k's all-reduce runs on a
communication stream under step k+1's compute (each capture owns its flat gradient buffer) and a step's timed interval
ends only once the previous step's all-reduce is complete; in the e2e arm the all-reduce feeds the optimizer and is serial.

One JSON line (rank 0):
  value       frames/s over all ranks, inputs resident in HBM, C-ABI calls, device-event timed (max over ranks)
  e2e         frames/s through the public API render() -> loss -> backward -> (all-reduce) -> Adam step, with each
              step's camera block + target images copied from pinned host memory and the loss read back
  roofline    the dominant kernel: algorithmic bytes / its CUDA-event time (sr_set_profiling) vs MEASURED_PEAKS.json
  cpu_baseline  the oracle (C restatement, OpenMP) fwd+bwd on host cores on a bounded sample of the same frames
  reference_cuda  (ours arm, N=1) the unmodified reference extension timed in the same run, same frames

--impl reference runs the UNMODIFIED reference extension (oracle/_ref/_C.so, its own CUDA path) through the same
harness; if the .so is missing it falls back to the CPU oracle port and says so.

--dump-outputs DIR writes what the last timed step of the value arm computed (rank 0), as float32 .npy files a caller
of that path would receive: color (F,3,n) and allmap (F,8,n) at n pixels, radii (F,m), and the frame-summed surfel
gradients dL_dmeans3D / dL_dsh / dL_dopacity / dL_dscales / dL_drotations (m,...) of m surfels.  n and m are every
pixel and surfel when the files fit in 64 MB, otherwise a fixed sample of them: sorted indices drawn by
np.random.default_rng(0) (pixels) and np.random.default_rng(1) (surfels).  The inputs are seeded, so two builds run
with the same arguments can be compared file by file.
"""
from __future__ import annotations

import argparse
import atexit
import contextlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from vidu4d_b200 import distributed as D  # noqa: E402
from vidu4d_b200.synthetic import SurfelCloud, object_scene, orbit_view, projection_matrix  # noqa: E402

NVIEWS = 64
TAN = 0.5
L2_MB = 126
GRAD_KEYS = ("dL_dmeans3D", "dL_dsh", "dL_dopacity", "dL_dscales", "dL_drotations")      # the flat gradient buffer, in order
DUMP_BYTES = 63 * 10**6     # --dump-outputs: array bytes, leaving room for the .npy headers under 64 MB


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--surfels", type=int, default=300_000)
    ap.add_argument("--res", type=int, default=512)
    ap.add_argument("--frames-per-step", type=int, default=8)
    ap.add_argument("--opacity", default="trained", choices=["trained", "init"])
    ap.add_argument("--cpu-frames", type=int, default=8, help="frames of the cpu_baseline sample after one warm-up frame (0 = skip)")
    ap.add_argument("--mode", default="batch", choices=["batch", "streams"], help="ours: one batched launch set per step, or F single-frame calls over --streams CUDA streams")
    ap.add_argument("--no-value-graph", action="store_true", help="keep the value-arm step eager (no CUDA-graph capture)")
    ap.add_argument("--split-features", action="store_true", help="e2e model keeps the reference's _features_dc / _features_rest "
                    "pair (one torch.cat per step + the split of its gradient) instead of one (P,16,3) SH parameter")
    ap.add_argument("--no-variants", action="store_true", help="skip the 1- and 2-frame-per-call variants of the value arm")
    ap.add_argument("--split", type=int, default=1, help="batch mode: render the step's frames as this many sub-batches on parallel "
                    "streams inside the captured step (bandwidth-bound kernels of one overlap the composites of another)")
    ap.add_argument("--no-ref-cuda", action="store_true", help="skip timing the reference extension in the ours arm")
    ap.add_argument("--ref-device", default="cuda", choices=["cuda", "cpu"])
    ap.add_argument("--no-graph", action="store_true", help="keep the e2e step eager (no CUDA-graph capture)")
    ap.add_argument("--no-fused", action="store_true", help="e2e through render() instead of render_fused()")
    ap.add_argument("--e2e-streams", type=int, default=1, help="(debug) streams of the eager e2e step when --no-graph")
    ap.add_argument("--streams", type=int, default=8, help="CUDA streams the frames of a step alternate over (value arm)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed value-arm step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)         # never outlive the benchmark, even when it fails before stop()
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_views(device):
    vms, cps, pms = [], [], []
    P = projection_matrix(TAN, TAN).astype(np.float64)
    for f in range(NVIEWS):
        R, t = orbit_view(f, NVIEWS)
        W2C = np.eye(4); W2C[:3, :3] = R; W2C[:3, 3] = t
        vm = W2C.T
        vms.append(vm.astype(np.float32)); pms.append((vm @ P).astype(np.float32)); cps.append((-R.T @ t).astype(np.float32))
    return np.stack(vms), np.stack(pms), np.stack(cps)


def sync_all(world):
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()


def max_over_ranks(ms: float, world: int, device) -> float:
    if world == 1:
        return ms
    t = torch.tensor([ms], dtype=torch.float64, device=device)
    torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    return float(t.item())


# ------------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def emit(line: dict):
    """The ONE JSON line goes to the process's real stdout; everything else (NCCL banners, library chatter) was
    rerouted to stderr at the file-descriptor level in main()."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)                     # C libraries (NCCL prints its version banner on stdout) now write to stderr
    args = parse()
    rank, world, local_rank = D.env_rank_world()
    if args.impl == "reference" and (args.ref_device == "cpu" or not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "_C.so"))):
        if args.dump_outputs:
            sys.exit("--dump-outputs: the CPU oracle arm has no GPU outputs to write")
        return reference_cpu_arm(args, rank, world)
    assert torch.cuda.is_available(), "bench.py needs a GPU (the CPU oracle is only the baseline leg)"
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    D.init_distributed("nccl", device)
    F, K, Wm, RES, P = args.frames_per_step, args.steps, max(args.warmup, 3), args.res, args.surfels

    try:
        torch.autograd.graph.set_warn_on_accumulate_grad_stream_mismatch(False)   # frames deliberately run on several streams
    except Exception:
        pass
    from vidu4d_b200 import _capi, rasterizer as RZ, renderer as RN
    if args.impl == "reference":
        from oracle import ref_ext
        ref_ext.load()
        RN.GaussianRasterizer = ref_ext.RefGaussianRasterizer        # same render() glue, reference rasterizer under it
    else:
        _capi.load()   # fail loudly if the CUDA library is missing

    scene = object_scene(P, seed=0, opacity=args.opacity, center=(0.0, 0.0, 0.0))
    # SH rows stored as one (P,16,3) parameter (both arms): no per-step concatenation of _features_dc / _features_rest
    cloud = SurfelCloud(scene, device, fused_features=not args.split_features)
    vms_h, pms_h, cps_h = build_views(device)
    vms = torch.from_numpy(vms_h).to(device); pms = torch.from_numpy(pms_h).to(device); cps = torch.from_numpy(cps_h).to(device)
    bg = torch.zeros(3, device=device)
    g = torch.Generator(device=device).manual_seed(1234)
    dLc = torch.randn((3, RES, RES), device=device, generator=g)
    dLo = torch.randn((8, RES, RES), device=device, generator=g) * 0.1
    flush = torch.empty((256 << 20,), dtype=torch.uint8, device=device)     # > L2 (126 MB)
    e = torch.empty((0,), device=device)

    with torch.no_grad():
        t_in = dict(means3D=cloud.get_xyz.detach().contiguous(), opac=cloud.get_opacity.detach().contiguous(),
                    scales=cloud.get_scaling.detach().contiguous(), rots=cloud.get_rotation.detach().contiguous(),
                    shs=cloud.get_features.detach().contiguous())
    acc = [torch.zeros_like(t_in[k]) for k in ("means3D", "shs", "opac", "scales", "rots")]
    acc_flat_bytes = sum(a.numel() for a in acc) * 4

    def view_of(step, f):
        return (step * world * F + rank * F + f) % NVIEWS

    # ---------------- device-resident arm: C-ABI level (or the reference's pybind _C) ----------------
    if args.impl == "ours":
        C = RZ._C
        RZ.set_sync_mode(False)

        def frame_dev(v):
            o = C.rasterize_gaussians(bg, t_in["means3D"], e, t_in["opac"], t_in["scales"], t_in["rots"], 1.0, e, vms[v],
                                      pms[v], TAN, TAN, RES, RES, t_in["shs"], 3, cps[v], False, False)
            return o, C.rasterize_gaussians_backward(bg, t_in["means3D"], o[3], e, t_in["scales"], t_in["rots"], 1.0, e,
                                                     vms[v], pms[v], TAN, TAN, dLc, dLo, t_in["shs"], 3, cps[v], o[4],
                                                     o[0], o[5], o[6], False)
    else:
        from oracle import ref_ext
        Cr = ref_ext.load()

        def frame_dev(v):
            o = Cr.rasterize_gaussians(bg, t_in["means3D"], e, t_in["opac"], t_in["scales"], t_in["rots"], 1.0, e, vms[v],
                                       pms[v], TAN, TAN, RES, RES, t_in["shs"], 3, cps[v], False, False)
            return o, Cr.rasterize_gaussians_backward(bg, t_in["means3D"], o[3], e, t_in["scales"], t_in["rots"], 1.0, e,
                                                      vms[v], pms[v], TAN, TAN, dLc, dLo, t_in["shs"], 3, cps[v], o[4],
                                                      o[0], o[5], o[6], False)

    # ---- ours, default: the F frames of a step are ONE batched launch set; the step (camera gather -> forward -> backward ->
    # sum over frames into the flat gradient) is captured in a CUDA graph, then one NCCL all-reduce and the step's only
    # host<->device synchronisation (check_overflow).  `--mode streams` keeps round 1's harness: F single-frame calls
    # alternating over `--streams` CUDA streams, per-stream gradient rows reduced once per step.
    BATCH = args.impl == "ours" and args.mode == "batch"
    NS = 1 if (args.impl != "ours" or BATCH) else max(1, args.streams)
    side = [torch.cuda.Stream(device=device) for _ in range(max(NS, 2, args.split))]
    nflt = acc_flat_bytes // 4
    stack = torch.zeros((NS, nflt), device=device)
    flat_acc = torch.zeros((nflt,), device=device) if (NS > 1 or BATCH) else stack[0]

    def views(row):
        out, o_ = [], 0
        for a in acc:
            out.append(row[o_:o_ + a.numel()].view(a.shape)); o_ += a.numel()
        return out
    accs = [views(stack[k]) for k in range(NS)]
    flat_views = views(flat_acc)
    flat_outs = dict(zip(GRAD_KEYS, flat_views))
    # second flat gradient buffer: the two captured value-arm steps each write their own, so that step k's all-reduce can
    # run on the communication stream while step k+1 computes (multi-GPU only; see step_dev)
    flat_acc2 = torch.zeros((nflt,), device=device) if (BATCH and world > 1) else flat_acc
    flat_outs2 = dict(zip(GRAD_KEYS, views(flat_acc2)))
    flat_accs, flat_outss = [flat_acc, flat_acc2], [flat_outs, flat_outs2]
    GIDX = (3, 5, 2, 6, 7)      # gr = (dmeans2D, dcolors, dopacity, dmeans3D, dtransMat, dsh, dscales, drots)
    step_ctr = torch.zeros((), dtype=torch.int64, device=device)      # lives on the device: the captured step advances it
    ar = torch.arange(F, device=device)
    dLc_b = dLc.expand(F, -1, -1, -1).contiguous() if BATCH else None
    dLo_b = dLo.expand(F, -1, -1, -1).contiguous() if BATCH else None
    value_graph = [None]
    R_last_box = [0]

    SPLIT = max(1, args.split) if BATCH else 1
    split_rows = torch.zeros((SPLIT, nflt), device=device) if SPLIT > 1 else None
    split_outs = [dict(zip(GRAD_KEYS, views(split_rows[k])))
                  for k in range(SPLIT)] if SPLIT > 1 else None

    def batch_body(fpc=None, slot=0):
        """One batched forward+backward of `fpc` frames (default F) + the sum over frames into the flat gradient
        (buffer `slot`).  Returns the forward outputs of each launch and the flat gradient buffer written."""
        n = F if fpc is None else fpc
        idx = (step_ctr * (world * F) + rank * F + ar[:n]) % NVIEWS
        step_ctr.add_(1)
        vm_b, pm_b, cp_b = vms.index_select(0, idx), pms.index_select(0, idx), cps.index_select(0, idx)
        if SPLIT > 1 and n == F:
            main = torch.cuda.current_stream()
            sub = F // SPLIT
            fwd = []
            for k in range(SPLIT):
                side[k].wait_stream(main)
                with torch.cuda.stream(side[k]):
                    sl = slice(k * sub, (k + 1) * sub)
                    o = C.rasterize_gaussians_batch(bg, t_in["means3D"], e, t_in["opac"], t_in["scales"], t_in["rots"], 1.0, vm_b[sl],
                                                    pm_b[sl], TAN, TAN, RES, RES, t_in["shs"], 3, cp_b[sl])
                    fwd.append(o)
                    C.rasterize_gaussians_backward_batch(bg, t_in["means3D"], o[3], e, t_in["scales"], t_in["rots"], 1.0, vm_b[sl],
                                                         pm_b[sl], TAN, TAN, dLc_b[sl], dLo_b[sl], t_in["shs"], 3, cp_b[sl], o[4], o[5],
                                                         o[6], sum_shared=True, want_transmat=False, outs=split_outs[k])
            for k in range(SPLIT):
                main.wait_stream(side[k])
            torch.sum(split_rows, dim=0, out=flat_acc)
            return fwd, flat_acc
        o = C.rasterize_gaussians_batch(bg, t_in["means3D"], e, t_in["opac"], t_in["scales"], t_in["rots"], 1.0, vm_b, pm_b,
                                        TAN, TAN, RES, RES, t_in["shs"], 3, cp_b)
        # gradients of the (shared) surfel parameters are summed over the frames inside the per-surfel kernel and land
        # directly in the flat buffer the all-reduce runs over
        gr = C.rasterize_gaussians_backward_batch(bg, t_in["means3D"], o[3], e, t_in["scales"], t_in["rots"], 1.0, vm_b, pm_b,
                                                  TAN, TAN, dLc_b[:n], dLo_b[:n], t_in["shs"], 3, cp_b, o[4], o[5], o[6],
                                                  sum_shared=True, want_transmat=False, outs=flat_outss[slot] if n == F else None)
        if n != F:      # the 1- and 2-frames-per-call variants: several calls per step accumulate into the flat buffer
            for a_, gi in zip(flat_views, GIDX):
                a_.add_(gr[gi].reshape(a_.shape))
            return [o], flat_acc
        return [o], flat_accs[slot]

    # Two captures of the same step, used alternately, each with its own pinned status words and a "done" event: the host
    # checks step k-1's overflow words only AFTER it has queued step k, so the GPU never waits for the host between steps
    # (and the ranks of a multi-GPU run do not drift apart at the collective).  The check is still once per step.
    done_ev = [torch.cuda.Event(), torch.cuda.Event()]
    inflight = [None]

    def drain():
        """Wait for the step still in flight (if any) and check its overflow words."""
        if inflight[0] is not None:
            k = inflight[0]
            done_ev[k].synchronize()
            arm(value_graphs[k])
            RZ.check_overflow(keep=True, sync=False)
            inflight[0] = None

    comm_stream = torch.cuda.Stream(device=device)
    ar_done = [torch.cuda.Event(), torch.cuda.Event()]
    ar_pending = [False, False]

    def flush_allreduce():
        """Make the current stream wait for any all-reduce still running on the communication stream."""
        for k in range(2):
            if ar_pending[k]:
                torch.cuda.current_stream().wait_event(ar_done[k]); ar_pending[k] = False

    last_out = [None]       # (forward outputs, flat gradient buffer) of the latest step, for --dump-outputs

    def step_dev(step):
        R_last = 0
        if BATCH:
            if value_graph[0] is not None:
                k = step & 1
                value_graphs[k].replay()
                last_out[0] = value_graphs[k].result
                if world > 1:
                    # step k's all-reduce (its own flat buffer) goes to the communication stream and overlaps step k+1's
                    # compute; this step's timed interval ends only after the PREVIOUS step's all-reduce has finished, so
                    # every exchange lies inside a timed interval (the last one is flushed by step_dev.flush)
                    main = torch.cuda.current_stream()
                    comm_stream.wait_stream(main)
                    with torch.cuda.stream(comm_stream):
                        torch.distributed.all_reduce(flat_accs[k])
                        ar_done[k].record()
                    if ar_pending[1 - k]:
                        main.wait_event(ar_done[1 - k]); ar_pending[1 - k] = False
                    ar_pending[k] = True
                done_ev[k].record()
                drain()                     # step k-1 (the other graph): its words landed long ago
                inflight[0] = k
                return R_last
            last_out[0] = batch_body()
            if world > 1:
                torch.distributed.all_reduce(flat_acc)
            RZ.check_overflow()             # eager fallback: the step's only host<->device synchronisation
            return R_last
        main = torch.cuda.current_stream()
        if NS > 1:
            for st_ in side:
                st_.wait_stream(main)
        fwd = []
        for f in range(F):
            k = f % NS
            ctx = torch.cuda.stream(side[k]) if NS > 1 else contextlib.nullcontext()
            with ctx:
                o, gr = frame_dev(view_of(step, f))
                for a_, gi in zip(accs[k], GIDX):
                    if f < NS:
                        a_.copy_(gr[gi].view(a_.shape))
                    else:
                        a_.add_(gr[gi].view(a_.shape))
                R_last = o[0]
                if args.dump_outputs:
                    fwd.append(o[:4])
        last_out[0] = (fwd, flat_acc)
        if NS > 1:
            for st_ in side:
                main.wait_stream(st_)
            if F >= NS:
                torch.sum(stack, dim=0, out=flat_acc)
            else:
                torch.sum(stack[:F], dim=0, out=flat_acc)
        if world > 1:
            torch.distributed.all_reduce(flat_acc)
        if args.impl == "ours":
            RZ.check_overflow()     # the step's only host<->device synchronisation
        return R_last

    def capture(body_fn, what):
        """Warm up eagerly (allocator pools, capacity hints), then capture body_fn into a CUDA graph; None on failure."""
        try:
            RZ.set_sync_mode(True); body_fn(); RZ.set_sync_mode(False)      # learn the instance capacity
            for _ in range(2):
                body_fn()
            RZ.check_overflow()
            RZ.reserve_host_slots(8)
            warm = torch.cuda.Stream(device=device)
            warm.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(warm):
                body_fn(); RZ.check_overflow()
            torch.cuda.current_stream().wait_stream(warm)
            torch.cuda.synchronize()
            RZ.reserve_host_slots(8)
            gph = torch.cuda.CUDAGraph()
            lc0 = _capi.launch_count()
            with torch.cuda.graph(gph):
                gph.result = body_fn()          # the graph's outputs: every replay rewrites these tensors
            gph.launches = _capi.launch_count() - lc0      # kernels of OUR library one replay launches
            gph.watch = list(RZ._pending)      # the pinned status words this graph rewrites on every replay
            return gph
        except Exception as ex:   # pragma: no cover
            sys.stderr.write(f"[bench] CUDA-graph capture of {what} failed: {ex!r}\n")
            RZ._pending.clear()
            torch.cuda.synchronize()
            return None

    def arm(gph):
        """Make check_overflow(keep=True) watch the status words of the graph that is about to be replayed."""
        RZ._pending[:] = gph.watch if gph is not None else []

    value_mode = "eager"
    value_graphs = [None, None]
    if BATCH and not args.no_value_graph:
        value_graphs = [capture(lambda: batch_body(slot=0), "the value-arm step"),
                        capture(lambda: batch_body(slot=1), "the value-arm step (second copy)")]
        value_graph[0] = value_graphs[0] if all(g is not None for g in value_graphs) else None
        value_mode = ("2 x cuda_graph(batched forward+backward+frame-sum), overflow check of step k-1 after step k is queued"
                      + ("; step k's all-reduce (own flat buffer, communication stream) overlaps step k+1's compute" if world > 1 else "")
                      if value_graph[0] is not None else "eager (capture failed)")

    def timed(step_fn, nsteps, nwarm):
        for s in range(nwarm):
            step_fn(s)
        if step_fn is step_dev and BATCH:
            flush_allreduce()
            drain()
        if getattr(step_fn, "drain", None) is not None:
            step_fn.drain()
        sync_all(world)
        starts = [torch.cuda.Event(enable_timing=True) for _ in range(nsteps)]
        ends = [torch.cuda.Event(enable_timing=True) for _ in range(nsteps)]
        t0 = time.perf_counter()
        for s in range(nsteps):
            flush.fill_(s & 255)                      # L2 flush between timed iterations (not timed)
            starts[s].record()
            step_fn(nwarm + s)
            if s == nsteps - 1 and step_fn is step_dev and BATCH:
                flush_allreduce()                     # the last step's exchange ends inside its own timed interval
            ends[s].record()
        if step_fn is step_dev and BATCH:
            drain()                                   # the last step's overflow check (inside the wall-clock, after its event)
        if getattr(step_fn, "drain", None) is not None:
            step_fn.drain()                           # e2e: the last step's loss readback + overflow check
        sync_all(world)
        wall = (time.perf_counter() - t0) * 1e3
        per = [a.elapsed_time(b) for a, b in zip(starts, ends)]
        return sum(per), per, wall

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = _capi.launch_count() if args.impl == "ours" else 0
    if BATCH:
        arm(value_graph[0])
    total_ms, per_ms, wall_ms = timed(step_dev, K, Wm)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last_out[0], views)
    launches = (_capi.launch_count() - launches0) if args.impl == "ours" else None
    if BATCH and value_graph[0] is not None:
        launches = value_graph[0].launches * K          # graph replays do not pass through the library's host-side counter
    total_ms = max_over_ranks(total_ms, world, device)
    frames = K * F * world
    value = frames / (total_ms * 1e-3)

    # the same F frames per step with 1 and 2 frames per call (Stage 3 renders M = 2 frames per step,
    # lab4d/engine/trainer.py:453-468): what the path delivers when the caller cannot batch 8 frames
    variants = None
    if BATCH and world == 1 and not args.no_variants:
        variants = {}
        for n in (1, 2):
            gph = capture(lambda: batch_body(n), f"the {n}-frame variant")

            def vstep(step, gph=gph, n=n):
                for _ in range(F // n):
                    if gph is not None:
                        gph.replay()
                    else:
                        batch_body(n)
                RZ.check_overflow(keep=gph is not None)
            arm(gph)
            vt, _, _ = timed(vstep, max(3, K // 2), 3)
            variants[f"frames_per_call_{n}"] = round(max(3, K // 2) * F / (vt * 1e-3), 2)
            del gph
        arm(value_graph[0])

    # R (instances) of a representative frame, for the algorithmic-byte figures
    if args.impl == "ours":
        RZ.set_sync_mode(True)
        o_probe = RZ._C.rasterize_gaussians(bg, t_in["means3D"], e, t_in["opac"], t_in["scales"], t_in["rots"], 1.0, e, vms[0],
                                            pms[0], TAN, TAN, RES, RES, t_in["shs"], 3, cps[0], False, False)
        R_inst = int(o_probe[0])
        # secondary, explanatory figure (SURVEY 8d): (pixel, instance) pair evaluations of the probe frame, as the
        # upper bound 256 x tile-list length summed over tiles (what a tile-wide walk would evaluate)
        from vidu4d_b200 import debug as _dbg
        _dec = _dbg.decode(o_probe[4], o_probe[5], o_probe[6], P, RES, RES, R_inst)
        _rg = _dec["ranges"].to(torch.int64)
        pair_upper = int(((_rg[:, 1] - _rg[:, 0]) * 256).sum().item())
        pairs_contrib = _dbg.contributing_pairs(_dec)          # (pixel, instance) pairs that passed every test
        V_vis = int((o_probe[3] > 0).sum().item())             # visible surfels of the probe frame
        del _dec, _rg
        RZ.set_sync_mode(False)
    else:
        R_inst = int(frame_dev(0)[0][0])

    # ---------------- e2e arm: public API with host buffers ----------------
    from vidu4d_b200.renderer import MiniCam, PipelineParams, render as render_unfused, render_fused
    # ours: the fused post-processing path of the public API; reference arm: the reference's own torch glue
    render = render_fused if (args.impl == "ours" and not args.no_fused) else render_unfused
    pipe = PipelineParams()
    params = cloud.flat_params()
    fg = D.FlatGrads(params)
    opt = torch.optim.Adam(params, lr=1e-7, fused=True)
    targets_h = torch.rand((F, 3, RES, RES), generator=torch.Generator().manual_seed(5)).pin_memory()
    # host side of a step's inputs: per-view camera blocks live in pinned tables; every step gathers ITS F views into a
    # pinned staging block (two of them, so that the host can stage step k+1 while the copy engine still reads step k's)
    cam_tab_h = torch.from_numpy(np.stack([np.stack([vms_h[v], pms_h[v]]) for v in range(NVIEWS)]).astype(np.float32)).pin_memory()
    cps_tab_h = torch.from_numpy(np.ascontiguousarray(cps_h, dtype=np.float32).reshape(NVIEWS, 3)).pin_memory()
    cam_hs = [torch.empty((F, 2, 4, 4)).pin_memory() for _ in range(2)]      # viewmatrix, full_proj per frame
    cps_hs = [torch.empty((F, 3)).pin_memory() for _ in range(2)]
    loss_hs = [torch.empty((1,)).pin_memory() for _ in range(2)]
    cam_h, cps_hh, loss_h = cam_hs[0], cps_hs[0], loss_hs[0]
    h2d = targets_h.numel() * 4 + cam_h.numel() * 4 + cps_hh.numel() * 4
    fov = 2.0 * float(np.arctan(TAN))

    tg = torch.empty((F, 3, RES, RES), device=device); cam = torch.empty((F, 2, 4, 4), device=device); cp = torch.empty((F, 3), device=device)
    tot = torch.zeros((), device=device)

    view_idx = {}

    def fill_host(step, slot=0):
        idx = view_idx.get(step)
        if idx is None:
            idx = view_idx[step] = torch.tensor([view_of(step, f) for f in range(F)], dtype=torch.int64)
        torch.index_select(cam_tab_h, 0, idx, out=cam_hs[slot])
        torch.index_select(cps_tab_h, 0, idx, out=cps_hs[slot])

    e2e_streams = [1]
    tots = [torch.zeros((), device=device) for _ in range(8)]

    def body_frames():
        """H2D of this step's inputs -> render x F -> loss -> backward (everything a CUDA graph can hold).  Frames
        alternate over e2e_streams[0] streams; autograd runs each frame's backward on its forward stream and
        serialises the accumulation into the (flat) .grad buffers itself."""
        ns = e2e_streams[0]
        main = torch.cuda.current_stream()
        # cameras up front (small); each frame's target image is uploaded on the stream that renders the frame, so the
        # copy engine works while the other streams' frames compute (same bytes per step, nothing cached across steps)
        cam.copy_(cam_h, non_blocking=True); cp.copy_(cps_hh, non_blocking=True)
        fg.zero_()
        for t_ in tots:
            t_.zero_()
        if ns > 1:
            for k in range(ns):
                side[k].wait_stream(main)
        for f in range(F):
            k = f % ns
            with (torch.cuda.stream(side[k]) if ns > 1 else contextlib.nullcontext()):
                tg[f].copy_(targets_h[f], non_blocking=True)
                view = MiniCam(RES, RES, fov, fov, 0.01, 100.0, cam[f, 0], cam[f, 1], cp[f])
                out = render(view, cloud, pipe, bg)
                loss = (out["render"] - tg[f]).abs().mean() + 0.05 * (1.0 - (out["rend_normal"] * out["surf_normal"]).sum(0)).mean() \
                    + 0.01 * out["rend_dist"].mean()
                loss.backward()
                tots[k].add_(loss.detach())
        if ns > 1:
            for k in range(ns):
                main.wait_stream(side[k])
        tot.copy_(torch.stack(tots).sum())

    if BATCH:
        from vidu4d_b200.renderer import BatchCameras, render_loss_batch

        def body_batch(slot=0):
            """H2D of this step's inputs -> ONE batched rasterize + fused post-processing + losses -> ONE batched backward."""
            main = torch.cuda.current_stream()
            cam.copy_(cam_hs[slot], non_blocking=True); cp.copy_(cps_hs[slot], non_blocking=True)
            side[0].wait_stream(main)
            with torch.cuda.stream(side[0]):           # the step's target images upload beside the rasterizer forward
                tg.copy_(targets_h, non_blocking=True)
            fg.zero_()
            bc = BatchCameras(RES, RES, fov, fov, cam[:, 0], cam[:, 1], cp)
            out = render_loss_batch(bc, cloud, pipe, bg, tg, w_rgb=1.0, lambda_normal=0.05, lambda_dist=0.01,
                                    target_stream=side[0])
            out["loss"].backward()
            tot.copy_(out["loss"].detach())

    body_sel = [body_batch if BATCH else body_frames]

    def body():
        body_sel[0]()

    freeze = [False]

    def tail():
        fg.allreduce_(average_over=F * world)
        if not freeze[0]:
            opt.step()
        loss_h.copy_(tot.reshape(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        if args.impl == "ours":
            RZ.check_overflow(keep=graph is not None)
        return float(loss_h[0])

    graph, e2e_mode = None, "eager"
    # Pipelined e2e loop (ours, batch mode): two captures of the step, each bound to its own pinned staging block, loss
    # word and status words.  The host stages + queues step k (H2D, render, losses, backward, all-reduce, Adam, D2H of the
    # loss), THEN waits for step k-1's event, reads its loss and checks its overflow words -- every step still uploads its
    # inputs and has its result read on the host, but the GPU never idles while the host prepares the next step.
    e2e_graphs = [None, None]
    e2e_done = [torch.cuda.Event(), torch.cuda.Event()]
    e2e_inflight = [None]
    pipelined = [False]

    def drain_e2e():
        """Host side of the step still in flight: wait for it, check its overflow words, return its loss."""
        k = e2e_inflight[0]
        if k is None:
            return None
        e2e_done[k].synchronize()
        RZ._pending[:] = e2e_graphs[k].watch
        RZ.check_overflow(keep=True, sync=False)
        e2e_inflight[0] = None
        return float(loss_hs[k][0])

    def step_e2e(step):
        if pipelined[0]:
            k = step & 1
            fill_host(step, k)
            e2e_graphs[k].replay()
            fg.allreduce_(average_over=F * world)
            if not freeze[0]:
                opt.step()
            loss_hs[k].copy_(tot.reshape(1), non_blocking=True)
            e2e_done[k].record()
            last = drain_e2e()              # step k-1: finished long ago
            e2e_inflight[0] = k
            return last
        fill_host(step)
        if graph is not None:
            graph.replay()
        else:
            body()
        return tail()
    step_e2e.drain = drain_e2e

    def step_e2e_sync(step):
        """One step, its loss returned (the check below compares single steps)."""
        r = step_e2e(step)
        return drain_e2e() if pipelined[0] else r

    if args.impl == "ours" and not args.no_graph:
        # The sync-free forward makes the whole step capturable: one cudaGraphLaunch replaces ~150 small launches.
        # (The reference cannot be captured: its forward blocks on a D2H copy, rasterizer_impl.cu:282.)
        for ns_try in (sorted({min(NS, 8, F), min(NS, 4), min(NS, 2), 1}, reverse=True) if (NS > 1 and not BATCH) else [1]):
            try:
                e2e_streams[0] = ns_try
                for s_ in range(2):
                    step_e2e(s_)                               # eager warm-up: allocator pools, caches, capacity hints
                RZ.check_overflow()
                RZ._pending.clear()
                RZ.reserve_host_slots(F + 4)
                gph = torch.cuda.CUDAGraph()
                warm = torch.cuda.Stream(device=device)
                warm.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(warm):
                    fill_host(0); body(); RZ.check_overflow()   # once on a side stream, as torch recommends
                torch.cuda.current_stream().wait_stream(warm)
                torch.cuda.synchronize()
                RZ.reserve_host_slots(F + 4)
                with torch.cuda.graph(gph):
                    body()
                graph = gph
                graph.watch = list(RZ._pending)
                e2e_mode = (f"cuda_graph(H2D + batched render_loss_batch + backward, 1 stream) + eager all-reduce/Adam/readback" if BATCH else
                            f"cuda_graph(H2D+render+loss+backward, {ns_try} stream(s)) + eager all-reduce/Adam/readback")
                if BATCH:       # second copy, bound to staging slot 1; if it cannot be captured the single graph above stays
                    try:
                        RZ._pending.clear()
                        RZ.reserve_host_slots(F + 4)
                        with torch.cuda.stream(warm):
                            fill_host(1, 1); body_batch(1); RZ.check_overflow()
                        torch.cuda.current_stream().wait_stream(warm)
                        torch.cuda.synchronize()
                        RZ.reserve_host_slots(F + 4)
                        gph2 = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(gph2):
                            body_batch(1)
                        gph2.watch = list(RZ._pending)
                        e2e_graphs[0], e2e_graphs[1] = gph, gph2
                        pipelined[0] = True
                        e2e_mode = ("2 x cuda_graph(H2D + batched render_loss_batch + backward) used alternately + all-reduce/Adam/loss D2H; "
                                    "step k-1's loss is read and its overflow words checked after step k is queued")
                    except Exception as ex2:   # pragma: no cover
                        sys.stderr.write(f"[bench] second capture of the e2e step failed ({ex2!r}); single-graph synchronous loop\n")
                        pipelined[0] = False
                        torch.cuda.synchronize()
                    RZ._pending[:] = graph.watch
                break
            except Exception as ex:   # pragma: no cover
                sys.stderr.write(f"[bench] CUDA-graph capture of the e2e step ({ns_try} streams) failed: {ex!r}\n")
                graph = None
                e2e_streams[0] = 1
                RZ._pending.clear()
                torch.cuda.synchronize()

    # sanity of the captured multi-stream step against a plain eager single-stream step on the same inputs
    e2e_check = None
    if args.impl == "ours":
        if graph is None and NS > 1 and not args.no_graph is False:
            pass
        if graph is None and args.e2e_streams > 1:
            e2e_streams[0] = args.e2e_streams          # eager multi-stream (only for debugging the check)
        freeze[0] = True                                # same parameters for every evaluation of the check
        l_mode = step_e2e_sync(1000)
        torch.cuda.synchronize()
        g_mode = fg.flat.clone()
        keep_graph, keep_ns, keep_pipe = graph, e2e_streams[0], pipelined[0]
        graph, e2e_streams[0], pipelined[0] = None, 1, False
        RZ._pending.clear()
        # the eager leg is round 1's per-frame path: render_fused() + the torch loss expressions + autograd -- an
        # independent evaluation of what the batched fused-loss step computes
        body_sel[0] = body_frames
        l_eager = step_e2e(1000)
        torch.cuda.synchronize()
        g_eager = fg.flat.clone()
        l_eager2 = step_e2e(1000)
        torch.cuda.synchronize()
        g_eager2 = fg.flat.clone()
        graph, e2e_streams[0], pipelined[0] = keep_graph, keep_ns, keep_pipe
        body_sel[0] = body_batch if BATCH else body_frames
        RZ._pending[:] = graph.watch if graph is not None else []
        freeze[0] = False
        nrm = float(g_eager.double().norm() + 1e-30)
        e2e_check = {"loss_mode": l_mode, "loss_eager": l_eager,
                     "grad_rel_l2_diff": float((g_mode - g_eager).double().norm()) / nrm,
                     "eager_self_rel_l2_diff": float((g_eager2 - g_eager).double().norm()) / nrm,
                     "eager_path": "per-frame render_fused() + torch losses + autograd"}

    e2e_total, _, _ = timed(step_e2e, K, Wm)
    e2e_total = max_over_ranks(e2e_total, world, device)
    e2e_value = frames / (e2e_total * 1e-3)
    clocks = sampler.stop() if rank == 0 else None
    if os.environ.get("BENCH_PROFILE_E2E") and args.impl == "ours":
        # launch list of the e2e step for `ncu --profile-from-start off --metrics gpu__time_duration.sum`: two EAGER steps
        # (graph replays hide the kernels from the profiler's range) between cudaProfilerStart / Stop
        keep = (graph, pipelined[0])
        graph, pipelined[0] = None, False
        RZ._pending.clear()
        step_e2e(2000); torch.cuda.synchronize()
        torch.cuda.profiler.start()
        step_e2e(2001); step_e2e(2002); torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        graph, pipelined[0] = keep
        RZ._pending[:] = graph.watch if graph is not None else []

    # ---------------- per-kernel profile + roofline (ours only) ----------------
    roofline, kernels = None, None
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json (measured)" if peaks else "B200_PROFILING.md fallback 6650 GB/s"
    N = RES * RES
    if args.impl == "ours" and rank == 0:
        # The same step as the timed region, eager, with the library's per-kernel CUDA events switched on
        # (sr_set_profiling: events on the launching stream around every kernel; nothing else is in flight).
        RZ._pending.clear()
        prof_step = (lambda: batch_body()) if BATCH else (lambda: [frame_dev(f % NVIEWS) for f in range(F)])
        prof_step()
        torch.cuda.synchronize()
        _capi.get_profile()
        _capi.set_profiling(True)
        nprof = 3
        for _ in range(nprof):
            prof_step()
        prof = _capi.get_profile()
        _capi.set_profiling(False)
        RZ.check_overflow()
        Fl = F if BATCH else 1                       # frames one launch processes
        Vv = V_vis
        # ALGORITHMIC bytes per frame of each kernel (SURVEY.md 8(d), split per kernel in DESIGN.md section 3);
        # implementation-only traffic (contribution masks, instance-record stream written by the gather) is listed apart
        alg = {
            "preprocess_fwd": P * (40 + 12 * 16) + Vv * 87, "scan_block_sums": (P // 256) * 8,
            "emit_keys": P * 20 + R_inst * 12, "sort_histogram": R_inst * 8, "sort_plan": 6 * 256 * 8,
            "onesweep_passes": R_inst * 24 * 6, "ranges_gather": R_inst * 8 + 8 * (RES // 16) ** 2,
            "composite_fwd": R_inst * 76 + N * 64, "composite_bwd": R_inst * 76 + N * 64 + Vv * 72,
            "surfel_bwd": Vv * (343 + 240), "tile_order": 12 * (RES // 16) ** 2,
        }
        impl = {"ranges_gather": R_inst * (12 + 80 + 80), "composite_fwd": R_inst * (80 + 32) + N * 64,
                "composite_bwd": R_inst * (80 + 32) + N * 64 + Vv * 80}
        kernels = {}
        for k, v in prof.items():
            ms = v["ms"] / max(v["count"], 1)                       # per launch
            ab = alg.get(k, 0) * Fl
            kernels[k] = {"ms_per_launch": round(ms, 5), "ms_per_frame": round(ms / Fl, 5), "frames_per_launch": Fl,
                          "alg_MB_per_launch": round(ab / 1e6, 2), "GBps": round(ab / 1e9 / (ms * 1e-3), 1) if ms > 0 else None}
            if k in impl:
                kernels[k]["impl_MB_per_launch"] = round(impl[k] * Fl / 1e6, 2)
        dom = max(kernels, key=lambda k: kernels[k]["ms_per_launch"])
        ach = kernels[dom]["GBps"]
        ncu = {}
        try:   # counters of that kernel from the committed `ncu --set full` capture (per launch of ONE frame)
            ncu = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(dom, {})
        except Exception:
            pass
        # the capture is of a batch of `frames_per_launch` frames per launch: rescale to this run's launch
        nfl = float(ncu.get("frames_per_launch", 1) or 1)
        traffic = ncu.get("dram_bytes_per_launch")
        if traffic is not None:
            traffic = int(traffic * Fl / nfl)
        frame_alg = 1002 * P + 324 * R_inst + 128 * N
        roofline = {"kernel": dom, "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                    "frac": round(ach / hbm_peak, 5), "traffic": traffic, "peak_source": peak_src,
                    "alg_bytes_per_launch": alg.get(dom, 0) * Fl, "impl_bytes_per_launch": impl.get(dom, alg.get(dom, 0)) * Fl,
                    "launch_ms": kernels[dom]["ms_per_launch"], "frames_per_launch": Fl,
                    "traffic_note": "dram__bytes_read+write of this kernel's launch from the committed ncu --set full capture "
                                    "(profiles/ncu_traffic.json), rescaled to this run's frames per launch",
                    "l2_red_sectors": (None if ncu.get("l2_red_sectors") is None else int(ncu["l2_red_sectors"] * Fl / nfl)),
                    "lanes_active": ncu.get("lanes_active"),
                    "contributing_pairs": pairs_contrib, "visible_surfels": Vv,
                    "note": "the composite kernels are FP32-issue / latency bound by construction (SURVEY 8d): each instance record "
                            "is read once per tile but evaluated against ~10 pixels; algorithmic HBM bytes are small. "
                            "pairs/s is the explanatory figure, profiles/ holds the ncu pipe utilisation",
                    "contributing_pairs_per_s": round(pairs_contrib * (K * F * world) / (total_ms * 1e-3), 0),
                    "pair_evals_upper_per_frame": pair_upper,
                    "frame_alg_MB": round(frame_alg / 1e6, 1),
                    "frame_GBps": round(frame_alg / 1e9 / (total_ms * 1e-3 / (K * F)), 1),
                    "frame_frac": round(frame_alg / 1e9 / (total_ms * 1e-3 / (K * F)) / hbm_peak, 4)}

    # ---------------- reference CUDA extension in the same run (ours arm, rank 0, N=1) ----------------
    reference_cuda = None
    if args.impl == "ours" and world == 1 and not args.no_ref_cuda and os.path.exists(os.path.join(ROOT, "oracle", "_ref", "_C.so")):
        try:
            from oracle import ref_ext
            Cr = ref_ext.load()

            def ref_step(step):
                for f in range(F):
                    v = view_of(step, f)
                    o = Cr.rasterize_gaussians(bg, t_in["means3D"], e, t_in["opac"], t_in["scales"], t_in["rots"], 1.0, e, vms[v],
                                               pms[v], TAN, TAN, RES, RES, t_in["shs"], 3, cps[v], False, False)
                    gr = Cr.rasterize_gaussians_backward(bg, t_in["means3D"], o[3], e, t_in["scales"], t_in["rots"], 1.0, e,
                                                         vms[v], pms[v], TAN, TAN, dLc, dLo, t_in["shs"], 3, cps[v], o[4],
                                                         o[0], o[5], o[6], False)
                    acc[0].add_(gr[3]); acc[1].add_(gr[5]); acc[2].add_(gr[2]); acc[3].add_(gr[6]); acc[4].add_(gr[7])
            rt, _, _ = timed(ref_step, max(3, K // 2), 3)
            reference_cuda = {"value": round(max(3, K // 2) * F / (rt * 1e-3), 2), "unit": "frames/s",
                              "what": "unmodified reference extension (oracle/_ref/_C.so, sm_100a), same frames, device-resident"}
        except Exception as ex:  # pragma: no cover
            reference_cuda = {"unavailable": repr(ex)}

    # ---------------- CPU baseline (oracle port) ----------------
    cpu_baseline = None
    if rank == 0 and world == 1 and args.cpu_frames > 0:
        cpu_baseline = cpu_oracle_fps(scene, vms_h, pms_h, cps_h, RES, args.cpu_frames, dLc.cpu().numpy(), dLo.cpu().numpy())

    if rank == 0:
        line = {
            "metric": "raster fwd+bwd frames/sec @512^2, 300K surfels", "value": round(value, 2), "unit": "frames/s",
            "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": round(total_ms / K, 4), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": args.impl,
            "config": {"workload": f"HL: {P} surfels (seeded noisy sphere, SH deg 3, opacity={args.opacity}), {RES}x{RES}, "
                                   f"{F} frames/step/GPU on orbiting cameras, colour+depth+normal+distortion fwd+bwd",
                       "surfels": P, "resolution": RES, "frames_per_step_per_gpu": F, "instances_per_frame": R_inst,
                       "parallelism": f"frames sharded over {world} GPU(s), 1 NCCL all-reduce of {acc_flat_bytes >> 20} MiB/step" if world > 1 else "1 GPU",
                       "streams": NS, "mode": (args.mode if args.impl == "ours" else "reference: single-frame calls, legacy default stream"),
                       "value_step": value_mode, "split": (max(1, args.split) if args.impl == "ours" and args.mode == "batch" else None),
                       "l2": f"explicit flush (256 MiB write) between timed steps; per-step working set also exceeds the {L2_MB} MB L2"},
            "e2e": {"value": round(e2e_value, 2), "unit": "frames/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4,
                    "mode": e2e_mode, "check_vs_eager": e2e_check, "api": "render_loss_batch" if BATCH else ("render_fused" if render is render_fused else "render"),
                    "what": "render() -> L1+normal+distortion loss -> backward -> (all-reduce) -> fused Adam; per step the "
                            "cameras + target images come from pinned host memory, the loss is read back",
                    "model": "SurfelCloud, SH rows as " + ("_features_dc/_features_rest (torch.cat per step)" if args.split_features
                                                           else "one (P,16,3) parameter (both arms)")},
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "kernels_ms": kernels, "variants": variants,
            "cpu_baseline": cpu_baseline, "reference_cuda": reference_cuda, "wall_ms_timed_region": round(wall_ms, 1),
        }
        if args.impl == "reference":
            line["cpu_baseline"] = {"value": line["value"], "unit": "frames/s", "cores": 0, "kind": "reference",
                                    "sample": "the reference's only implementation of this path is CUDA: this arm runs "
                                              "oracle/_ref/_C.so on the GPU (no CPU cores involved); see --ref-device cpu for the oracle port"}
            line["e2e"]["h2d_bytes_per_step"] = int(h2d)
        emit(line)
    if world > 1:
        torch.distributed.destroy_process_group()
    return 0


def dump_outputs(dirname, fwd, grad_flat, views):
    """--dump-outputs (see the module docstring): fwd = the forward outputs (num_rendered, color, allmap, radii, ...) of
    the step's launches in frame order, grad_flat = the flat gradient buffer the step wrote."""
    color = torch.cat([o[1].reshape(-1, 3, o[1].shape[-2] * o[1].shape[-1]) for o in fwd])
    allmap = torch.cat([o[2].reshape(-1, 8, o[2].shape[-2] * o[2].shape[-1]) for o in fwd])
    radii = torch.cat([o[3].reshape(-1, o[3].shape[-1]) for o in fwd]).float()
    grads = dict(zip(GRAD_KEYS, views(grad_flat)))
    F, n_pix, n_surf = color.shape[0], color.shape[-1], radii.shape[-1]
    pixel_bytes = F * (3 + 8) * 4
    surfel_bytes = (F + sum(g[0].numel() for g in grads.values())) * 4
    n, m = n_pix, n_surf
    while n * pixel_bytes + m * surfel_bytes > DUMP_BYTES:
        n, m = (n + 1) // 2, (m + 1) // 2
    dev = color.device
    pix = torch.from_numpy(np.sort(np.random.default_rng(0).choice(n_pix, n, replace=False))).to(dev) if n < n_pix else None
    surf = torch.from_numpy(np.sort(np.random.default_rng(1).choice(n_surf, m, replace=False))).to(dev) if m < n_surf else None
    out = {"color": color, "allmap": allmap, "radii": radii, **grads}
    os.makedirs(dirname, exist_ok=True)
    for name, a in out.items():
        if name in ("color", "allmap"):
            a = a if pix is None else a.index_select(-1, pix)
        else:
            a = a if surf is None else a.index_select(-1 if name == "radii" else 0, surf)
        np.save(os.path.join(dirname, name + ".npy"), a.float().cpu().numpy())


def cpu_oracle_fps(scene, vms_h, pms_h, cps_h, RES, nframes, dLc, dLo):
    from oracle import surfel_oracle as so
    so.lib()
    # one untimed warm-up frame (page faults of the oracle's buffers, OpenMP thread start-up), then the sample
    st = so.forward(scene.means3D, scene.opacities, scene.scales, scene.rotations, shs=scene.shs, sh_degree=3, W=RES, H=RES,
                    tanfovx=TAN, tanfovy=TAN, bg=(0, 0, 0), viewmatrix=vms_h[63], projmatrix=pms_h[63], campos=cps_h[63])
    so.backward(st, dLc, dLo)
    t0 = time.perf_counter()
    for f in range(nframes):
        st = so.forward(scene.means3D, scene.opacities, scene.scales, scene.rotations, shs=scene.shs, sh_degree=3, W=RES, H=RES,
                        tanfovx=TAN, tanfovy=TAN, bg=(0, 0, 0), viewmatrix=vms_h[f], projmatrix=pms_h[f], campos=cps_h[f])
        so.backward(st, dLc, dLo)
    dt = time.perf_counter() - t0
    return {"value": round(nframes / dt, 4), "unit": "frames/s", "cores": so.num_threads(), "kind": "port",
            "sample": f"{nframes} full frames of the same workload (fwd+bwd) after 1 warm-up frame, oracle/surfel_oracle.c with OpenMP"}


def reference_cpu_arm(args, rank, world):
    """--impl reference when oracle/_ref is absent (or --ref-device cpu): the oracle port on the host cores."""
    if rank != 0:
        return 0
    scene = object_scene(args.surfels, seed=0, opacity=args.opacity, center=(0.0, 0.0, 0.0))
    vms_h, pms_h, cps_h = build_views(None)
    rng = np.random.default_rng(0)
    dLc = rng.normal(size=(3, args.res, args.res)).astype(np.float32)
    dLo = (0.1 * rng.normal(size=(8, args.res, args.res))).astype(np.float32)
    n = max(2, min(args.steps, 8))
    cb = cpu_oracle_fps(scene, vms_h, pms_h, cps_h, args.res, n, dLc, dLo)
    line = {"metric": "raster fwd+bwd frames/sec @512^2, 300K surfels", "value": cb["value"], "unit": "frames/s",
            "n_gpus": args.gpus, "steps": n, "warmup": 0, "ms_per_step": round(1e3 / cb["value"], 2), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": f"HL: {args.surfels} surfels, {args.res}x{args.res}; one frame per step on the host cores"},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)
    return 0


if __name__ == "__main__":
    sys.exit(main())
