"""Training-step benchmark of the cross quality enhancement network (stage two: the codec frozen): 512x896 patches,
batch 2 per GPU, data-parallel with one NCCL all-reduce of the flat gradient buffer per step.

    python tools/cqe_train_bench.py [--steps 20] [--warmup 3] [--profile]
    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/cqe_train_bench.py

Prints one JSON line on rank 0: pairs/s (whole job), ms per step (device-timed, max over ranks), useful TFLOP/s (the
3x3 convolutions at their real channel counts: forward, data gradients except conv0's, weight gradients), and, on
rank 0's GPU, the same step through torch autograd on oracle/cqe.py's modules with cuDNN (bf16 autocast,
channels_last) as a library baseline.  --profile adds CUDA-event times per op group of one eager step."""
import argparse
import json
import os
import subprocess
import sys
from pathlib import Path

import torch
import torch.distributed as dist

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from masic_b200.cqe import Independent_EN  # noqa: E402

LMBDA = 0.01


def useful_flops_per_pair(h: int, w: int) -> float:
    """MACs per pixel and view: 3x3 convs, real channels.  Forward of all 21 convs, data gradient of all but conv0
    (conv1's feeds the mask-weight gradient), weight gradient of all."""
    eb = sum(6 * 9 * c * c for c in (32, 64, 96))
    conv0, conv1, conv2 = 9 * 3 * 32, 9 * 6 * 32, 9 * 96 * 3
    fwd = eb + conv0 + conv1 + conv2
    dgrad = eb + conv1 + conv2
    wgrad = fwd
    return 2.0 * 2 * h * w * (fwd + dgrad + wgrad)


def gpu_info(index: int) -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                                     # report, do not guess
        return {"gpu": torch.cuda.get_device_name(index), "power_limit": f"unavailable ({e})"}


def cudnn_baseline(dev, net, x1h, x2h, Hm, x1, x2, steps: int, warmup: int) -> float:
    """ms per step of oracle/cqe.py's modules under torch autograd (cuDNN convs, bf16 autocast, channels_last)."""
    from oracle.cqe import OracleIndependentEN
    ora = OracleIndependentEN()
    ora.load_state_dict({k: v.cpu() for k, v in net.state_dict().items()})
    ora = ora.to(dev).to(memory_format=torch.channels_last)
    opt = torch.optim.Adam(ora.parameters(), lr=1e-4, fused=True)
    fwd = OracleIndependentEN.forward.__wrapped__
    torch.backends.cudnn.benchmark = True
    a = [t.contiguous(memory_format=torch.channels_last) for t in (x1h, x2h)]

    def step():
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = fwd(ora, a[0], a[1], Hm)
            loss = LMBDA * 255.0 ** 2 * (torch.mean((out["x1_hat"].float() - x1) ** 2) +
                                         torch.mean((out["x2_hat"].float() - x2) ** 2))
        loss.backward()
        opt.step()
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--height", type=int, default=512)
    ap.add_argument("--width", type=int, default=896)
    ap.add_argument("--batch", type=int, default=2)
    ap.add_argument("--baseline-steps", type=int, default=5)
    ap.add_argument("--profile", action="store_true")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be >= 1")
    H, W, B = a.height, a.width, a.batch
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if not torch.cuda.is_available():
        raise SystemExit("cqe_train_bench needs a CUDA device")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    torch.manual_seed(0)
    net = Independent_EN().to(dev).train()
    tr = net.trainer(B, H, W, dev, lmbda=LMBDA)
    opt = torch.optim.Adam(net.parameters(), lr=1e-4, fused=True)
    g = torch.Generator().manual_seed(100 + rank)
    x1 = torch.rand(B, 3, H, W, generator=g)
    x2 = torch.rand(B, 3, H, W, generator=g)
    x1h = (x1 + 0.02 * torch.randn(x1.shape, generator=g)).to(dev)
    x2h = (x2 + 0.02 * torch.randn(x2.shape, generator=g)).to(dev)
    x1, x2 = x1.to(dev), x2.to(dev)
    Hm = torch.eye(3).repeat(B, 1, 1)
    Hm[:, 0, 2] = 12.0
    Hm = Hm.to(dev)
    losses = []
    for _ in range(max(1, a.warmup)):
        losses.append(tr.train_step(x1h, x2h, Hm, x1, x2, opt)["loss"])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        tr.train_step(x1h, x2h, Hm, x1, x2, opt)
    e1.record()
    torch.cuda.synchronize()
    losses.append(tr.read_losses()["loss"])
    ms = torch.tensor([e0.elapsed_time(e1) / a.steps], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms)
    res = None
    if rank == 0:
        flop = useful_flops_per_pair(H, W) * B
        base = cudnn_baseline(dev, net, x1h, x2h, Hm, x1, x2, a.baseline_steps, 2)
        res = {"metric": "cqe_train_step", "value": world * B / (ms / 1e3), "unit": "pairs/s", "n_gpus": world,
               "ms_per_step": ms, "steps": a.steps, "batch_per_gpu": B, "height": H, "width": W,
               "useful_tflops_per_gpu": flop / (ms / 1e3) / 1e12, "useful_gflop_per_step_per_gpu": flop / 1e9,
               "planned_gflop_per_step_per_gpu": tr.flops() / 1e9,
               "cudnn_autograd_ms_per_step": base, "speedup_vs_cudnn_autograd": base / ms,
               "loss_first": losses[0], "loss_last": losses[-1],
               "parallelism": f"dp{world}: one NCCL all-reduce of the flat fp32 gradient buffer "
                              f"({tr.flat_grad.numel()} floats) per step",
               **gpu_info(local)}
        if a.profile:
            tr.step_grads(x1h, x2h, Hm, x1, x2, refresh=True, read_back=False)
            res["profile_ms"] = {n: round(t, 4) for n, t in tr.profile()}
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if res is not None:
        print(json.dumps(res))


if __name__ == "__main__":
    main()
