#!/usr/bin/env python
"""Headline benchmark: reconstructed frames/s of the BDE2VID hot path (voxelise + UNet forward).

Workload (BASELINE.json configs[1]): one synthetic 346x260 event sequence per step, T windows of
31,500 events, 5-bin voxels, batch 1, assumed cfg of SURVEY.md section 8, seed-0 random weights,
fused voxelise + UNet on one B200.  With N GPUs every rank processes its own sequences (weak scaling).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--precision bf16|fp32] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.  Inputs and weights come from fixed seeds,
so runs with the same arguments compute on identical inputs; --dump-outputs DIR writes the frames of the last timed step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from bde2vid_b200 import synth  # noqa: E402

H, W, NEV, BINS = 260, 346, 31500, 5
# algorithmic work per frame of the reference graph at 264x352 (SURVEY.md 8(d)): conv + linear FLOPs
# are executed by the implicit-GEMM kernel, bmm FLOPs by the window-attention kernel.
GF_CONV, GF_LINEAR, GF_BMM = 125.79, 32.36, 5.19
VOXEL_BYTES_PER_WINDOW = 16 * NEV + 4 * BINS * H * W
# dram__bytes_read.sum + dram__bytes_write.sum of the voxeliser (memset + reduction kernels) from the committed ncu capture;
# filled in from profiles/ once measured (None = not captured for this build)
VOXEL_TRAFFIC = {
    # profiles/r02_ncu_voxel_traffic.csv (ncu --cache-control none over one 100-window call at 346x260, launches 6-11): the six
    # chained reduction kernels (each also zeroes the next chunk's grids) read 50.4 MB from DRAM (= the events, 16 B x 3.15 M:
    # the zeroed grids are still L2-resident, nothing is re-read); 143.6 MB of the 264x352 grids are written back while the
    # kernels run, the rest of the 185.9 MB after the last one -- every grid line goes to HBM once
    "bytes_per_100_windows": 50.4e6 + 185.9e6,
    "source": "ncu --cache-control none, dram__bytes_read.sum of the 6 chained reduction kernels of one call (50.4 MB = events) + one "
              "write-back of the padded grids (185.9 MB, of which 143.6 MB inside the kernels); profiles/r02_ncu_voxel_traffic.csv",
}


def cfg_dict():
    ns = {}
    exec(synth.ASSUMED_CFG_STR, ns)
    return ns["model"]


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm=d["hbm_gbs"], tc_burst=d["bf16_tflops"], tc_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tc_burst=1590.0, tc_sustained=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        if not sm:
            return None
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference path on the host cores (bounded sample)
# ------------------------------------------------------------------------------------------------

def reference_model_or_none(cfg):
    """The UNMODIFIED reference (BDE2VID from /root/reference or baseline/_ref, imported through oracle/ref_shim.py) when
    its tree is reachable at run time -- it is in the build container, it is not on the GPU box -- else None."""
    for root in (os.environ.get("BDE2VID_REFERENCE"), os.path.join(ROOT, "baseline", "_ref"), "/root/reference"):
        if root and os.path.isdir(os.path.join(root, "model", "BDE2VID")):
            try:
                os.environ["BDE2VID_REFERENCE"] = root
                from oracle import ref_shim
                ref_shim.REFERENCE_ROOT = root
                R = ref_shim.reference_modules()
                return R, ref_shim
            except Exception as e:          # missing third-party import etc.: fall back to the port, say why
                sys.stderr.write("reference at %s not importable (%s); timing the oracle port\n" % (root, e))
    return None, None


def cpu_reference_fps(T_sample, seq_id=0, threads=None, h=H, w=W, nev=NEV, return_frames=False):
    """frames/s of voxelise + forward on the host cores for T_sample windows of the bench workload: the reference's own
    code when its tree is present ('reference'), else the oracle port of the same algorithm ('port': numpy voxeliser +
    functional torch fp32)."""
    from oracle import oracle_torch as O
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    cfg = O.full_cfg(cfg_dict()["generator"])
    sd = synth.init_state_dict(cfg, 0)
    ev = synth.gen_events(seq_id, T_sample, h, w, nev)
    prm = O.croper_params(w, h, 3)
    R, shim = reference_model_or_none(cfg)
    kind = "port"
    if R is not None:
        kind = "reference"
        model = R.BDE2VID(generator=dict(cfg)).eval()
        model.load_state_dict(sd, strict=True)
        crop = R.Croper(3)
        crop.update_params(w, h)
    t0 = time.perf_counter()
    vox = []
    for wi in range(T_sample):
        xs, ys, ts, ps = synth.to_loader_format(ev, wi)
        if R is not None:
            v = R.events_to_voxel_torch(*(torch.from_numpy(a) for a in (xs, ys, ts, ps)), BINS, sensor_size=(h, w))
            vox.append(crop.pad(v[None]))
        else:
            vox.append(O.pad_voxel(torch.from_numpy(O.voxel_grid(xs, ys, ts, ps, BINS, (h, w)))[None], prm))
    with torch.no_grad():
        if R is not None:
            with shim.cpu_mode():
                out = model([{"events": v} for v in vox])
        else:
            out = O.bde2vid_forward(sd, cfg, vox)
    frames = [O.crop_image(o, prm) for o in out]
    dt = time.perf_counter() - t0
    if return_frames:
        return T_sample / dt, dt, threads, kind, torch.cat(frames, 0)
    return T_sample / dt, dt, threads, kind


def run_reference_arm(args, rank, world):
    """`--impl reference`: the reference's CPU implementation of the path on the box's host cores (all threads), on a
    bounded sample of the same workload.  Rank 0 alone works; the other ranks exit."""
    if rank != 0:
        return
    if args.full_cpu:
        # SURVEY 8(d) C1: one 240x180 sequence, T = 100, voxelise + model end to end
        fps, dt, threads, kind = cpu_reference_fps(100, h=180, w=240, nev=15000)
        T_s, times, sample = 100, [dt], "C1: 100 of 100 windows of one 240x180 sequence (BASELINE.json configs[0])"
    else:
        T_s = args.ref_windows
        for _ in range(max(0, min(args.warmup, 1))):
            cpu_reference_fps(2)
        times = []
        for _ in range(args.steps):
            fps, dt, threads, kind = cpu_reference_fps(T_s)
            times.append(dt)
        sample = "%d of %d windows of one 346x260 sequence" % (T_s, args.windows)
    dt = float(np.mean(times))
    val = T_s / dt
    what = ("the unmodified reference imported from its tree" if kind == "reference"
            else "oracle port of the reference path; the reference tree is not on this box")
    line = {
        "impl": "reference", "metric": "reconstructed frames/s (346x260, 5-bin)", "value": val, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": len(times), "warmup": min(args.warmup, 1), "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, T_s, note="CPU arm: bounded sample of the same workload"),
        "cpu_baseline": {"value": val, "unit": "frames/s", "cores": threads, "kind": kind, "sample": "%s (%s)" % (sample, what)},
        "e2e": {"value": val, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def workload_config(args, T, note=None):
    c = {"workload": "BDE2VID assumed-cfg, seed-0 weights, one synthetic %dx%d sequence per step, T=%d windows x %d "
                     "events, %d-bin voxels, batch 1, fused voxelise+UNet (BASELINE.json configs[1])" % (W, H, T, NEV, BINS),
         "windows_per_sequence": T, "events_per_window": NEV, "padded": "264x352",
         "sequences_in_flight_per_gpu": (getattr(args, "concurrent", 1) * getattr(args, "batch", 1)) if note is None else 1,
         "streams": getattr(args, "concurrent", 1) if note is None else 1,
         "sequences_per_call": getattr(args, "batch", 1) if note is None else 1,
         "step": "every stream submits `sequences_per_call` independent batch-1 sequences, which the engine executes as "
                 "one batched launch sequence (reconstruct_events_batch)",
         "l2_policy": "no flush: one step streams >2 GB of activations (>>126 MB L2) between re-reads of its inputs"}
    if note:
        c["note"] = note
    return c


DUMP_BYTES = 60 << 20


def dump_outputs(path, seqs):
    """Write the frames a caller of the timed path received (per sequence, in stream order, its T frames [1, 1, H, W]) so
    that two builds can be compared output for output.  ``frames.npy`` (float32 [sequences, T, K]) holds every frame at
    the same K pixels: all of them when the frames fit in DUMP_BYTES, else a sample drawn with seed 0, whose flat
    indices y * W + x are ``frame_pixels.npy`` (float64)."""
    os.makedirs(path, exist_ok=True)
    frames = torch.stack([torch.cat(f, 0) for f in seqs]).flatten(2)
    n, t, p = frames.shape
    k = min(p, DUMP_BYTES // (4 * n * t + 8))
    pix = np.sort(np.random.default_rng(0).permutation(p)[:k])
    np.save(os.path.join(path, "frames.npy"), frames[:, :, torch.from_numpy(pix).to(frames.device)].float().cpu().numpy())
    np.save(os.path.join(path, "frame_pixels.npy"), pix.astype(np.float64))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("BDE2VID_PRECISION", "bf16"))
    ap.add_argument("--windows", type=int, default=100, help="T: windows (= frames) per sequence")
    ap.add_argument("--ref-windows", type=int, default=6, help="windows of the bounded CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--full-cpu", action="store_true", help="CPU arm / cpu_baseline on SURVEY's C1: 240x180, T=100, whole sequence")
    ap.add_argument("--config", default="default", choices=["default", "e2vid16", "gen4", "shard64", "pair"],
                    help="default = BASELINE.json configs[1] (the headline); e2vid16 = configs[2]; shard64 = configs[3]; gen4 = configs[4]; pair = one sequence split over two GPUs (SURVEY 8 f4)")
    ap.add_argument("--no-single", action="store_true", help="skip the extra one-sequence-in-flight measurement")
    ap.add_argument("--no-kernel-timing", action="store_true")
    ap.add_argument("--concurrent", type=int, default=2, help="CUDA streams (independent model calls in flight) per GPU")
    ap.add_argument("--batch", type=int, default=8, help="independent sequences batched into each model call")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the frames of the last resident step to DIR/*.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config != "default"):
        ap.error("--dump-outputs writes the frames of the default GPU workload only")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from bde2vid_b200 import ops
    from bde2vid_b200.model import MODELS

    warm = max(3, args.warmup)
    T = args.windows
    if args.config != "default":
        import bench_configs
        line = getattr(bench_configs, "run_" + args.config)(args, rank, world, dev)
        if rank == 0:
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return
    model = MODELS.build(cfg_dict())
    model.load_state_dict(synth.init_state_dict(cfg_dict()["generator"], 0), strict=True)
    model = model.eval().to(dev)
    model.generator.precision = args.precision

    # per-rank sequences: rank r processes seq ids r, r+world, ... (independent units; no data-path collective).
    # One step = S streams x NB sequences: every stream submits NB independent batch-1 sequences that the
    # engine runs as one batched launch sequence (dynamic batching of independent requests).
    S = max(1, args.concurrent)
    NB = max(1, args.batch)
    n_seq = 2 * S * NB
    host = []
    for i in range(n_seq):
        ev = synth.gen_events(rank + i * world, T, H, W, NEV)
        xs, ys, ts, ps, off = synth.to_loader_format_seq(ev)
        host.append([torch.from_numpy(a).pin_memory() for a in (xs, ys, ts, ps, off)])
    resident = [[a.to(dev) for a in h] for h in host]
    h2d_bytes = S * NB * sum(a.numel() * a.element_size() for a in host[0])
    d2h_bytes = S * NB * T * H * W * 4
    streams = [torch.cuda.Stream(device=dev) for _ in range(S)]
    out_host = [torch.empty(NB, T, 1, 1, H, W).pin_memory() for _ in range(S)]

    def pick(pool, i, s):
        base = ((i * S + s) * NB) % n_seq
        return [pool[(base + b) % n_seq] for b in range(NB)]

    def fan_out(fn):
        main = torch.cuda.current_stream()
        res = []
        for s in range(S):
            streams[s].wait_stream(main)
            with torch.cuda.stream(streams[s]):
                res.append(fn(s))
        for s in range(S):
            main.wait_stream(streams[s])
        return res

    last_frames = None

    def step_resident(i):
        nonlocal last_frames
        last_frames = fan_out(lambda s: model.reconstruct_events_batch(pick(resident, i, s), (H, W), slot=s))
        return last_frames

    def step_e2e(i):
        # pinned host arrays go straight into the plan's static device buffers (async H2D on the stream);
        # the reconstructed frames come back to pinned host memory on the same stream
        def one(s):
            frames = model.reconstruct_events_batch(pick(host, i, s), (H, W), slot=s)
            out_host[s].copy_(torch.stack([torch.stack(f, 0) for f in frames], 0), non_blocking=True)
        fan_out(one)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    with torch.no_grad():
        for i in range(warm):
            step_resident(i)
        sampler = ClockSampler(local)
        sampler.start()
        ms = timed(step_resident, args.steps)
        clocks = sampler.stop()
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, [seq for per_stream in last_frames for seq in per_stream])
        for i in range(2):
            step_e2e(i)
        ms_e2e = timed(step_e2e, args.steps)

    eng = model.generator.engine()
    # launches of one model call: read from a plan this run executed (a freshly built one has not been enqueued yet, which is
    # what eng.plan() returns when the LRU plan cache evicted slot 0 under a very large sweep configuration)
    done = [q for k, q in eng.plans.items() if k[:4] == (T, NB, 264, 352) and getattr(q, "launches", 0)]
    plan = done[0] if done else eng.plan(T, NB, 264, 352)
    launches_per_step = getattr(plan, "launches", 0) * S
    plan_gb = sum(q.nbytes for q in eng.plans.values()) / 2 ** 30
    fps = world * args.steps * S * NB * T / (ms * 1e-3)
    fps_e2e = world * args.steps * S * NB * T / (ms_e2e * 1e-3)

    # checksum of the reconstructed frames, reduced over ranks (the path's only collective: metric reduction)
    with torch.no_grad():
        frames = step_resident(0)[0][0]
        chk = torch.stack([f.double().mean() for f in frames]).sum().reshape(1)
    if world > 1:
        dist.all_reduce(chk)
    chk = float(chk.item()) / (world * T)

    pk = peaks()
    roofline = None
    voxel_roof = None
    attn_roof = None
    shares = None
    if not args.no_kernel_timing:
        # live per-kernel timing of the dominant kernel (the tcgen05 implicit-GEMM engine): one eager
        # (non-graph) pass of the same step with a CUDA event pair recorded in C right around every launch on
        # the launching stream.  A spin kernel first puts the GPU ~150 ms behind the host so that launches
        # queue up and the event pairs measure kernel time, not Python launch gaps.
        import ctypes as C
        from bde2vid_b200 import _lib
        lib = _lib.load()
        torch.cuda.synchronize()
        lib.bde_profile_begin(200000)
        # the same pass also gives the live share of every kernel class: each ops.* entry point of the schedule is
        # bracketed by a CUDA event pair on the (single) launching stream
        klass = {"window_attention_fused": lambda a: "attention_level1" if a[4] == 64 else "attention_level3",
                 "mlp_fused": lambda a: "fused_mlp_c%d" % a[2], "gemm": lambda a: "bde_gemm_tcgen05_convs",
                 "head_conv": lambda a: "head_conv", "voxelize_seq_into": lambda a: "voxeliser",
                 "upsample2x_sum": lambda a: "elementwise", "pred_sigmoid": lambda a: "elementwise",
                 "add": lambda a: "elementwise", "cast": lambda a: "elementwise"}
        pairs, saved = [], {}

        def bracket(name, fn, cls_of):
            def wrapped(*a, **k):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                r = fn(*a, **k)
                e1.record()
                pairs.append((cls_of(a), e0, e1))
                return r
            return wrapped
        for name, cls_of in klass.items():
            saved[name] = getattr(ops, name)
            setattr(ops, name, bracket(name, saved[name], cls_of))
        torch.cuda._sleep(int(0.3 * 1.9e9))
        plan.overlap = False           # one stream: every launch is timed alone
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.no_grad():
            p0.record()
            plan._enqueue(True)
            p1.record()
        torch.cuda.synchronize()
        plan.overlap = True
        for name, fn in saved.items():
            setattr(ops, name, fn)
        pass_ms = p0.elapsed_time(p1)
        shares = {}
        for cls, e0, e1 in pairs:
            d = shares.setdefault(cls, {"ms": 0.0, "launches": 0})
            d["ms"] += e0.elapsed_time(e1)
            d["launches"] += 1
        for d in shares.values():
            d["share"] = d["ms"] / pass_ms
            d["avg_us"] = d["ms"] * 1e3 / d["launches"]
        shares["_pass"] = {"ms": pass_ms, "what": "one eager single-stream pass of one model call (%d sequences x %d windows), "
                                                 "every launch serialised; shares are of this pass" % (NB, T)}
        # level-1 attention (the largest share): its binding unit is the special-function pipe -- one ex2 per
        # (head, query, key) score: 16 heads x 49 x 147 per window; measured MUFU.EX2 rate 16 / clk / SM (DESIGN.md section 4)
        attn_roof = None
        if "attention_level1" in shares:
            a1 = shares["attention_level1"]
            nwin1 = plan.lv[0]["nwin"] if "nwin" in plan.lv[0] else 0
            ex2 = 16.0 * 49 * 147 * nwin1 * a1["launches"]
            sm = torch.cuda.get_device_properties(dev).multi_processor_count
            peak_ex2 = 16.0 * sm * (clocks.get("sm_mhz") or 1965.0) * 1e6
            attn_roof = {"kernel": "attn_fused_kernel<64,4,19> (level-1 window attention, head_dim 4)", "bound": "sfu (MUFU.EX2)",
                         "achieved": ex2 / (a1["ms"] * 1e-3) / 1e12, "peak": peak_ex2 / 1e12, "unit": "T ex2/s",
                         "frac": ex2 / (a1["ms"] * 1e-3) / peak_ex2, "avg_launch_us": a1["avg_us"], "windows_per_launch": nwin1,
                         "peak_source": "16 ex2 / clk / SM (tools/micro/mufu_probe.cu) x SMs x SM clock under load"}
        tot, cnt = C.c_double(0.0), C.c_int(0)
        lib.bde_profile_end(C.byref(tot), C.byref(cnt))
        gemm_ms, n_rec = float(tot.value), int(cnt.value)
        # algorithmic FLOPs of exactly the launches that were timed: 2 M N K summed in C from the descriptors (the
        # head conv, the fused attention and the fused MLP kernels do their share of GF_CONV / GF_LINEAR outside
        # bde_gemm and are neither timed nor counted here)
        fl = C.c_double(0.0)
        lib.bde_profile_flops(C.byref(fl))
        flops = float(fl.value)
        ach = flops / (gemm_ms * 1e-3) / 1e12
        peak = pk["tc_sustained"]
        roofline = {"kernel": "bde_gemm tcgen05 kernels: conv_tma_kernel (TMA-fed persistent convs: ConvLSTM gates, "
                              "decoders, stride-2 encoders) + gemm_tc_kernel (enc0, L3 proj)", "bound": "tensor",
                    "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                    # DRAM bytes (read + write) per launch from the committed ncu --set full capture of three
                    # consecutive ConvLSTM gate convs (profiles/r01_ncu_full_prof_conv_lstm.metrics.txt): 26.3 / 49.2 /
                    # 14.3 MB; operands are served from L2 (algorithmic operand bytes per launch: 24-48 MB)
                    "traffic": 29.9e6, "traffic_source": "ncu capture, mean of 3 ConvLSTM launches (not live)",
                    "launches": n_rec, "avg_launch_us": gemm_ms * 1e3 / max(1, n_rec),
                    "kernel_ms_per_step": gemm_ms, "peak_source": pk["src"] + " sustained bf16 (kernel timed inside a long step)",
                    "flops_per_step": flops}
        # voxeliser alone, all T windows in one launch (HBM-bound)
        xs, ys, ts, ps, off = resident[0]
        vout = torch.empty(T, BINS, 264, 352, device=dev)
        for _ in range(3):
            ops.voxelize_seq(xs, ys, ts, ps, off, BINS, H, W, 2, 3, 264, 352, out=vout)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(10):
            ops.voxelize_seq(xs, ys, ts, ps, off, BINS, H, W, 2, 3, 264, 352, out=vout)
        e.record()
        torch.cuda.synchronize()
        vms = s.elapsed_time(e) / 10
        vach = VOXEL_BYTES_PER_WINDOW * T / (vms * 1e-3) / 1e9
        voxel_roof = {"kernel": "voxel_atomic_kernel (global RED.ADD.F32 executed by L2 into L2-resident zeroed grids, in chunks of "
                                "windows; every launch zeroes the next chunk, launches chained with programmatic dependent launch; "
                                "128-bit event loads)", "bound": "hbm", "achieved": vach, "peak": pk["hbm"], "unit": "GB/s",
                      "frac": vach / pk["hbm"], "traffic": VOXEL_TRAFFIC.get("bytes_per_100_windows"),
                      "traffic_source": VOXEL_TRAFFIC.get("source"), "ms_per_launch": vms,
                      "bytes_per_launch": VOXEL_BYTES_PER_WINDOW * T}

    # one sequence in flight (BASELINE.json configs[1] says "batch 1"): the strict single-sequence rate, reported beside
    # the batched headline
    single = None
    if not args.no_single and (S, NB) != (1, 1):
        def step_single(i):
            return model.reconstruct_events_batch([resident[i % n_seq]], (H, W), slot=0)
        with torch.no_grad():
            for i in range(3):
                step_single(i)
            ms1 = timed(step_single, 3)
        single = {"value": world * 3 * T / (ms1 * 1e-3), "unit": "frames/s", "streams": 1, "sequences_per_call": 1,
                  "ms_per_sequence": ms1 / 3}

    cpu = None
    parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        if args.full_cpu:
            v, dt, threads, kind = cpu_reference_fps(100, h=180, w=240, nev=15000)
            cpu = {"value": v, "unit": "frames/s", "cores": threads, "kind": kind,
                   "sample": "SURVEY C1: 100 of 100 windows of one 240x180 sequence, voxelise + model, %.1f s" % dt}
        else:
            Ts = args.ref_windows
            v, dt, threads, kind, ref_frames = cpu_reference_fps(Ts, seq_id=0, return_frames=True)
            cpu = {"value": v, "unit": "frames/s", "cores": threads, "kind": kind,
                   "sample": "%d of %d windows of the same 346x260 sequence, %s, %.1f s"
                             % (Ts, T, "the unmodified reference" if kind == "reference" else
                                "oracle port (numpy voxeliser + functional torch fp32)", dt)}
            # parity of the TIMED path in the same run: the same Ts windows through reconstruct_events_batch with the bench's
            # batch size (same kernels / dispatch as the timed steps: B = NB sequences, CUDA graph) vs the CPU frames
            seqs = []
            for b in range(NB):
                evb = synth.gen_events(b, Ts, H, W, NEV)
                seqs.append([torch.from_numpy(a).to(dev) for a in synth.to_loader_format_seq(evb)])
            with torch.no_grad():
                for _ in range(3):
                    outp = model.reconstruct_events_batch(seqs, (H, W), slot=0)
            got = torch.cat(outp[0], 0).cpu()
            parity = {"max_abs": float((got - ref_frames).abs().max()), "mse": float(((got - ref_frames) ** 2).mean()),
                      "frames": Ts, "batch": NB, "vs": kind, "gate": 2e-3}

    if rank == 0:
        line = {
            "metric": "reconstructed frames/s (346x260, 5-bin)", "value": fps, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if args.precision.startswith("bf16") else "f32",
            "data": "synthetic", "config": workload_config(args, T),
            "e2e": {"value": fps_e2e, "unit": "frames/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches_per_step * args.steps,
            "clocks": clocks, "roofline": roofline, "roofline_voxeliser": voxel_roof, "roofline_attention": attn_roof,
            "kernel_shares": shares, "cpu_baseline": cpu,
            "tflops_algorithmic": fps / world * (GF_CONV + GF_LINEAR + GF_BMM) / 1e3,
            "frame_checksum": chk, "precision": args.precision,
            "single_sequence": single, "parity": parity, "resident_plan_gb": plan_gb,
            "parity_max_abs": None if parity is None else parity["max_abs"],
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
