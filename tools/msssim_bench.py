"""MS-SSIM at 1216x2176 on one GPU: the fused kernel (csrc/msssim.cu), the same algorithm as the fp32 torch op
sequence pytorch_msssim 1.0 runs (oracle/msssim.py on float32 CUDA tensors), and PairStream end to end with
msssim on and off.

    python tools/msssim_bench.py [--iters 200] [--pairs 6] [--out profiles/r3_msssim_n1.json]

Kernel and torch times are CUDA events over `--iters` calls that rotate over `--pairs` distinct input pairs (each pair
63.5 MB, so the working set is larger than the 126 MB L2), after a device-side sleep that lets the host enqueue ahead.
PairStream rounds alternate msssim off / on on the same pipelined stream of pinned 8-bit host pairs.  Achieved FLOP/s
and bytes/s use the algorithm's operation and byte counts from shapes (`algorithm_counts`)."""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from masic_b200 import _lib, ops  # noqa: E402
from masic_b200.hsic import HSIC  # noqa: E402
from oracle import msssim as OM  # noqa: E402

HBM_TBS = 7.7        # data sheet, HGX B200, per GPU


def gpu_info(index: int) -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                                     # report, do not guess
        return {"gpu": torch.cuda.get_device_name(index), "power_limit": f"unavailable ({e})"}


def level_sizes(h, w, levels=5):
    out = [(h, w)]
    for _ in range(levels - 1):
        h, w = (h + h % 2) // 2, (w + w % 2) // 2
        out.append((h, w))
    return out


def algorithm_counts(planes, h, w, levels=5):
    """FP32 operations (an FMA counts 2) and HBM bytes MS-SSIM needs, per call on two images of `planes` planes.
    Per level: 3 products per input pixel, the 11-tap horizontal pass of 5 maps over h x (w - 10), the vertical pass
    over (h - 10) x (w - 10), ~20 operations per output for cs / ssim; between levels 4 operations per pooled pixel of
    each image.  Bytes: both images read once, each pooled level written once and read twice (statistics, next pool)."""
    flops = 0.0
    nbytes = 2 * planes * h * w * 4.0
    for l, (hl, wl) in enumerate(level_sizes(h, w, levels)):
        flops += planes * (3 * hl * wl + 2 * 55 * hl * (wl - 10) + 2 * 55 * (hl - 10) * (wl - 10)
                           + 20 * (hl - 10) * (wl - 10))
        if l:
            flops += 2 * planes * 4 * hl * wl
            nbytes += 2 * planes * hl * wl * 4.0 * 3
    return flops, nbytes


def timed(fn, iters):
    fn(0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda._sleep(20_000_000)
    e0.record()
    for i in range(iters):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--torch-iters", type=int, default=20)
    ap.add_argument("--pairs", type=int, default=6)
    ap.add_argument("--stream-pairs", type=int, default=60, help="pairs per PairStream round")
    ap.add_argument("--rounds", type=int, default=4, help="PairStream rounds per setting (alternating)")
    ap.add_argument("--height", type=int, default=1216)
    ap.add_argument("--width", type=int, default=2176)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_msssim_n1.json"))
    a = ap.parse_args()
    if a.pairs < 4:
        ap.error("--pairs must be >= 4 (the rotation has to exceed the L2)")
    if not torch.cuda.is_available():
        raise SystemExit("msssim_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    H, W = a.height, a.width
    lib = _lib.load()
    g = torch.Generator(device=dev).manual_seed(0)
    xs = [torch.rand(1, 3, H, W, generator=g, device=dev) for _ in range(a.pairs)]
    ys = [(x + 0.05 * torch.randn(x.shape, generator=g, device=dev)).clamp(0, 1).contiguous() for x in xs]

    # ---- the kernel: preallocated scratch and output, one masic_ms_ssim call (5 launches) per view
    import ctypes as C
    nbytes = lib.masic_ms_ssim_scratch_bytes(1, 3, H, W, 5)
    _lib.check(min(int(nbytes), 0), "masic_ms_ssim_scratch_bytes")
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    out = torch.empty(a.pairs, 3, device=dev)
    wts = (C.c_float * 5)(*ops.MS_SSIM_WEIGHTS)

    def kern(i):
        j = i % a.pairs
        _lib.check(lib.masic_ms_ssim(ys[j].data_ptr(), xs[j].data_ptr(), 1, 3, H, W, 5, 1.0, 0.01, 0.03, wts, 1,
                                     scratch.data_ptr(), out[j].data_ptr(), torch.cuda.current_stream().cuda_stream),
                   "masic_ms_ssim")
    k_ms = timed(kern, a.iters)
    k_err = max(float((out[j].double() - OM.ms_ssim_per_channel(ys[j].double(), xs[j].double(), 1.0)[0]).abs().max())
                for j in range(a.pairs))

    # ---- the same algorithm as pytorch_msssim's fp32 torch op sequence
    def tor(i):
        j = i % a.pairs
        OM.ms_ssim_per_channel(ys[j], xs[j], 1.0)
    t_ms = timed(tor, a.torch_iters)

    flops, hbm = algorithm_counts(3, H, W)
    info = gpu_info(0)
    try:
        clk_ghz = float(info["max_sm_clock"].split()[0]) / 1e3
        fma_peak = torch.cuda.get_device_properties(0).multi_processor_count * 128 * 2 * clk_ghz * 1e9
    except Exception:
        clk_ghz, fma_peak = None, None
    k_s = k_ms / 1e3
    bound_fma = flops / fma_peak if fma_peak else None
    bound_hbm = hbm / (HBM_TBS * 1e12)
    del xs, ys

    # ---- PairStream end to end, msssim off / on alternating
    torch.manual_seed(0)
    net = HSIC().eval().to(dev)
    ps = net.pair_stream(H, W, dev, depth=3)
    gh = torch.Generator().manual_seed(1)
    u = [(torch.randint(0, 256, (1, 3, H, W), generator=gh, dtype=torch.uint8).pin_memory(),
          torch.randint(0, 256, (1, 3, H, W), generator=gh, dtype=torch.uint8).pin_memory()) for _ in range(4)]
    Hm = torch.eye(3)[None].contiguous().pin_memory()

    def stream_round(msssim, n):
        t0 = time.perf_counter()
        tickets = []
        for i in range(n):
            tickets.append(ps.submit(u[i % 4][0], u[i % 4][1], Hm, msssim=msssim))
            if i >= ps.depth - 1:
                ps.result(tickets[i - ps.depth + 1])
        for t in tickets[max(0, n - ps.depth + 1):]:
            ps.result(t)
        return n / (time.perf_counter() - t0)
    stream_round(False, 10)
    stream_round(True, 10)
    rates = {False: [], True: []}
    for _ in range(a.rounds):
        for m in (False, True):
            rates[m].append(stream_round(m, a.stream_pairs))
    med = lambda v: sorted(v)[len(v) // 2]   # noqa: E731

    res = {
        "metric": "ms_ssim_1216x2176", "height": H, "width": W, "channels": 3, "levels": 5, "data_range": 1.0,
        **info,
        "kernel_ms_per_view": k_ms, "kernel_calls": a.iters, "distinct_input_pairs": a.pairs,
        "kernel_max_abs_err_vs_float64_oracle": k_err,
        "torch_fp32_ms_per_view": t_ms, "torch_fp32_calls": a.torch_iters,
        "torch_fp32_what": "oracle/msssim.py on float32 CUDA tensors: the op sequence of pytorch_msssim 1.0 "
                           "(grouped conv2d, avg_pool2d, elementwise)",
        "speedup_vs_torch_fp32": t_ms / k_ms,
        "algorithm_gflop_per_view": flops / 1e9, "algorithm_hbm_mb_per_view": hbm / 1e6,
        "kernel_tflops": flops / k_s / 1e12, "kernel_hbm_tbs": hbm / k_s / 1e12,
        "fp32_fma_peak_tflops": fma_peak / 1e12 if fma_peak else "not measured (no clock reading)",
        "fp32_fma_peak_basis": "148 SMs x 128 FP32 lanes x 2 x max SM clock (nvidia-smi)",
        "hbm_peak_tbs": HBM_TBS, "hbm_peak_basis": "HGX B200 data sheet, per GPU",
        "share_of_fma_bound": bound_fma / k_s if bound_fma else None,
        "share_of_hbm_bound": bound_hbm / k_s,
        "binding_bound": ("fp32 FMA" if bound_fma and bound_fma > bound_hbm else "HBM"),
        "pair_stream_pairs_per_s_msssim_off": rates[False], "pair_stream_pairs_per_s_msssim_on": rates[True],
        "pair_stream_median_off": med(rates[False]), "pair_stream_median_on": med(rates[True]),
        "pair_stream_setup": f"HSIC random init, depth {ps.depth}, pinned uint8 host pairs, criterion read back "
                             f"every pair, {a.rounds} alternating rounds of {a.stream_pairs} pairs per setting",
    }
    print(json.dumps(res))
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
