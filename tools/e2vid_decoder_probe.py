"""E2VIDRecurrent decoders at the e2vid16 shape (B = 16, 272x352, 4 encoders, bf16): the upsample-conv form
(use_upsample_conv=True: bilinear x2 of skip + x, then a 5x5 conv on the x2 map) against the transposed form
(use_upsample_conv=False: one 3x3 phase conv with N = 4 Cout on the low-resolution map, then bde_shuffle2x_sum), in one
process.

  1. whole recurrent step, CUDA events around ``--steps`` steps with states carried, profiler off; the two models
     alternate for ``--rounds`` rounds after a warm-up of both;
  2. per decoder stage, in a torch.profiler run of its own: the decoder GEMM and its memory-bound partner kernel
     (upsample before the GEMM, shuffle after it), mean device time over the profiled steps;
  3. MACs of each form from the shapes, and the bytes / s of the shuffle kernel (bytes it must move over its time).

The working set of a step (~1 GB of activations) is larger than the L2; caches are not flushed between steps.
Usage: python tools/e2vid_decoder_probe.py [--steps 20] [--rounds 5] [--prof-steps 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bde2vid_b200 import synth  # noqa: E402
from bde2vid_b200.e2vid import E2VIDRecurrent  # noqa: E402

B, H, W, NE, BC = 16, 272, 352, 4, 32


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = "nvidia-smi not readable: %s" % e
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi " + q: out}


def make(upsample):
    m = E2VIDRecurrent({"num_bins": 5, "use_upsample_conv": upsample})
    m.load_state_dict(synth.random_state_dict_like(m.state_dict(), 0), strict=True)
    m = m.eval().cuda()
    m.unetrecurrent.precision = "bf16"
    return m


def levels():
    """(h, w, Cin) of decoder i's low-resolution input."""
    return [(H >> (NE - i), W >> (NE - i), BC * 2 ** (NE - i)) for i in range(NE)]


def macs(form, h, w, cin):
    cout = cin // 2
    return {"upsample": B * 4 * h * w * 25 * cin * cout,        # 5x5 conv on the x2 map: 100 Cin Cout per low-res pixel
            "transposed": B * h * w * 36 * cin * cout,         # 3x3 conv, N = 4 Cout: 36 Cin Cout per low-res pixel
            "transposed_nonzero": B * h * w * 25 * cin * cout}[form]


def shuffle_bytes(i, h, w, cin):
    """g read once, dst written once, the skip read when there is one (every decoder but the last)."""
    cout, es = cin // 2, 2
    return es * B * h * w * 4 * cout * (2 if i == NE - 1 else 3)


def upsample_bytes(h, w, cin):
    """skip and x read at low resolution, dst written at x2."""
    return 2 * B * h * w * cin * 2 + 2 * B * 4 * h * w * cin


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--prof-steps", type=int, default=3)
    ap.add_argument("--out")
    a = ap.parse_args()
    torch.cuda.set_device(0)
    models = {"upsample": make(True), "transposed": make(False)}
    g = torch.Generator().manual_seed(1)
    xs = [(torch.randn(B, 5, H, W, generator=g) * (torch.rand(B, 5, H, W, generator=g) < 0.3)).cuda() for _ in range(8)]

    def run(m, n):
        for t in range(n):
            m({"events": xs[t % len(xs)]})

    times = {k: [] for k in models}
    with torch.no_grad():
        for m in models.values():
            m.reset_states()
            run(m, 5)
        torch.cuda.synchronize()
        for _ in range(a.rounds):
            for k, m in models.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                run(m, a.steps)
                e1.record()
                e1.synchronize()
                times[k].append(e0.elapsed_time(e1) / a.steps)

        # per-stage device times from the profiler (separate run)
        from torch.autograd import DeviceType
        from torch.profiler import ProfilerActivity, profile
        stages = {}
        for k, m in models.items():
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                run(m, a.prof_steps)
                torch.cuda.synchronize()
            evs = sorted([e for e in prof.events() if e.device_type == DeviceType.CUDA], key=lambda e: e.time_range.start)
            us = lambda e: e.time_range.end - e.time_range.start  # noqa: E731
            gemm, mem = [0.0] * NE, [0.0] * NE
            j = 0
            for n, e in enumerate(evs):
                if k == "transposed" and "shuffle2x_sum_kernel" in e.name:
                    mem[j % NE] += us(e)
                    gemm[j % NE] += us(evs[n - 1])
                    j += 1
                elif k == "upsample" and "upsample2x_sum" in e.name:
                    mem[j % NE] += us(e)
                    gemm[j % NE] += us(evs[n + 1])
                    j += 1
            assert j == NE * a.prof_steps, (k, j)
            step_us = sum(us(e) for e in evs) / a.prof_steps
            stages[k] = dict(gemm_us=[v / a.prof_steps for v in gemm], mem_us=[v / a.prof_steps for v in mem],
                             kernel_us_per_step=step_us)

    lines = []
    out = {"card": card(), "shape": "B=%d %dx%d, %d encoders, bf16" % (B, H, W, NE), "steps": a.steps, "rounds": a.rounds,
           "step_ms": {k: v for k, v in times.items()}, "decoders": []}
    lines.append("card: %s" % json.dumps(out["card"]))
    lines.append("shape: %s; %d rounds x %d steps per form, alternating" % (out["shape"], a.rounds, a.steps))
    for k, v in times.items():
        s = sorted(v)
        lines.append("step %-10s median %.3f ms  (min %.3f, max %.3f)  = %.0f frames/s" % (k, s[len(s) // 2], s[0], s[-1],
                                                                                       B / (s[len(s) // 2] * 1e-3)))
    for k in models:
        lines.append("kernel time per step (profiler, sum of all kernels) %-10s %.1f us" % (k, stages[k]["kernel_us_per_step"]))
    lines.append("decoder  in(h x w x Cin)   form        GEMM us   MACs (G)  TMAC/s   mem-kernel us  mem GB/s   stage us")
    for i, (h, w, cin) in enumerate(levels()):
        for k in models:
            gu, mu = stages[k]["gemm_us"][i], stages[k]["mem_us"][i]
            mc = macs(k, h, w, cin)
            nb = shuffle_bytes(i, h, w, cin) if k == "transposed" else upsample_bytes(h, w, cin)
            lines.append("%d        %3d x %3d x %3d   %-10s  %7.1f   %8.1f  %6.0f   %7.1f        %6.0f     %7.1f" % (
                i, h, w, cin, k, gu, mc / 1e9, mc / gu / 1e6, mu, nb / mu / 1e3, gu + mu))
            out["decoders"].append(dict(i=i, h=h, w=w, cin=cin, form=k, gemm_us=gu, macs=mc, mem_kernel_us=mu, mem_bytes=nb,
                                        mem_gbps=nb / mu / 1e3))
        lines.append("         MACs transposed / upsample = %.2f (non-zero taps only: %.2f)" % (
            macs("transposed", h, w, cin) / macs("upsample", h, w, cin), macs("transposed_nonzero", h, w, cin) / macs("upsample", h, w, cin)))
    tot = {k: sum(stages[k]["gemm_us"]) + sum(stages[k]["mem_us"]) for k in models}
    lines.append("all decoder stages per step: upsample %.1f us, transposed %.1f us" % (tot["upsample"], tot["transposed"]))
    out["decoder_stage_us_per_step"] = tot
    text = "\n".join(lines)
    print(text)
    print(json.dumps(out))
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n" + json.dumps(out) + "\n")


if __name__ == "__main__":
    main()
