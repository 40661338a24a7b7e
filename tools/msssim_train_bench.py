"""What training for MS-SSIM costs on one GPU: the HSIC training step at 512x896, batch 2, with metric="mse" and
metric="ms-ssim" (rounds alternate between the two), and the MS-SSIM forward + backward kernels (csrc/msssim.cu) at
512x896x2 and 1216x2176x1.

    python tools/msssim_train_bench.py [--steps 30] [--rounds 5] [--iters 100] [--out profiles/r3_msssim_train_n1.json]

Step times: CUDA events around `--steps` graph replays of `step_grads` (no read-back) per round; the medians of the
rounds are compared.  Kernel times: CUDA events over `--iters` calls that rotate over distinct input pairs whose total
exceeds the 126 MB L2, after a device-side sleep that lets the host enqueue ahead.  The backward's bytes are counted from
shapes by `bwd_bytes`.  The card's name and power limit are read in the same run."""
import argparse
import json
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
from masic_b200 import train_ops as T  # noqa: E402
from masic_b200.hsic import HSIC  # noqa: E402
from msssim_bench import HBM_TBS, gpu_info, level_sizes, timed  # noqa: E402


def bwd_bytes(planes, h, w, addend=False):
    """HBM bytes of one masic_ms_ssim_bwd call.  Per level (h_l x w_l, maps of (h_l - 10) x (w_l - 10)): the map
    launch reads x and y and writes three maps; the gather launch reads the three maps, x and y, the coarser level's
    gradient (a quarter of the pixels) and writes the level's gradient (level 0: dx, plus the addend's read)."""
    total = 0.0
    sizes = level_sizes(h, w)
    for l, (hl, wl) in enumerate(sizes):
        px, mp = hl * wl, (hl - 10) * (wl - 10)
        total += 4.0 * planes * (2 * px + 3 * mp)                  # map launch
        total += 4.0 * planes * (3 * mp + 2 * px + px)             # gather launch: maps, x, y, write
        if l + 1 < len(sizes):
            total += 4.0 * planes * sizes[l + 1][0] * sizes[l + 1][1]
        if l == 0 and addend:
            total += 4.0 * planes * px
    return total


def kernel_times(n, h, w, iters, dev):
    planes = n * 3
    pair_mb = 2 * planes * h * w * 4 / 1e6
    pairs = max(4, int(300 / pair_mb) + 1)                        # rotate over more than twice the L2
    g = torch.Generator(device=dev).manual_seed(0)
    xs = [torch.rand(n, 3, h, w, generator=g, device=dev) for _ in range(pairs)]
    xh = [(x + 0.03 * torch.randn(x.shape, generator=g, device=dev)).clamp(0, 1).contiguous() for x in xs]
    scratch, work = T.ms_ssim_buffers(n, 3, h, w, dev)
    out = torch.empty(n, 3, device=dev)
    dx = torch.empty(n, 3, h, w, device=dev)

    def fwd(i):
        T.ms_ssim_fwd(xh[i % pairs], xs[i % pairs], scratch, out)

    def fwd_bwd(i):
        fwd(i)
        T.ms_ssim_grad(xh[i % pairs], xs[i % pairs], scratch, -1.0 / planes, dx, work=work)
    f_ms = timed(fwd, iters)
    fb_ms = timed(fwd_bwd, iters)
    f_ms2 = timed(fwd, iters)
    f = min(f_ms, f_ms2)
    b = fb_ms - f
    nb = bwd_bytes(planes, h, w)
    return {"size": f"{n}x3x{h}x{w}", "fwd_ms": [f_ms, f_ms2], "fwd_bwd_ms": fb_ms, "bwd_ms": b,
            "bwd_launches": 2 + 5, "bwd_model_mb": nb / 1e6, "bwd_hbm_tbs": nb / (b / 1e3) / 1e12,
            "bwd_share_of_hbm_bound": nb / (HBM_TBS * 1e12) / (b / 1e3),
            "distinct_input_pairs": pairs, "input_pair_mb": pair_mb,
            "work_mb": work.numel() / 1e6, "calls": iters}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_msssim_train_n1.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("msssim_train_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    B, H, W = 2, 512, 896
    torch.manual_seed(0)
    net = HSIC().to(dev).train()
    trainers = {m: net.trainer(B, H, W, dev, lmbda=0.01 if m == "mse" else 8.0, metric=m) for m in ("mse", "ms-ssim")}
    g = torch.Generator(device=dev).manual_seed(1)
    x1, x2 = (torch.rand(B, 3, H, W, generator=g, device=dev) for _ in range(2))
    Hm = torch.eye(3, device=dev).repeat(B, 1, 1)
    for tr in trainers.values():                       # eager warm-up, graph capture, one replay
        for _ in range(3):
            tr.step_grads(x1, x2, Hm)
    torch.cuda.synchronize()
    times = {m: [] for m in trainers}
    for _ in range(a.rounds):
        for m, tr in trainers.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.steps):
                tr.step_grads(x1, x2, Hm, read_back=False)
            e1.record()
            torch.cuda.synchronize()
            times[m].append(e0.elapsed_time(e1) / a.steps)
    med = {m: sorted(v)[len(v) // 2] for m, v in times.items()}
    losses = {m: tr.read_losses() for m, tr in trainers.items()}
    del trainers, net
    torch.cuda.empty_cache()

    res = {
        "metric": "msssim_training", **gpu_info(0),
        "step": {"batch": B, "height": H, "width": W, "steps_per_round": a.steps, "rounds": a.rounds,
                 "ms_per_step": times, "median_ms": med, "added_ms": med["ms-ssim"] - med["mse"],
                 "last_losses": losses,
                 "setup": "HSIC random init, step_grads replayed as one CUDA graph, no read-back, rounds alternate "
                          "mse / ms-ssim"},
        "kernels": [kernel_times(2, 512, 896, a.iters, dev), kernel_times(1, 1216, 2176, a.iters, dev)],
        "hbm_peak_tbs": HBM_TBS, "hbm_peak_basis": "HGX B200 data sheet, per GPU",
    }
    print(json.dumps(res))
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
