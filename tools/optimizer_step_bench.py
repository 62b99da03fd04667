"""Training-step time per update rule: momentum, Adam, RMSProp and Adam + EMA on the fused CUDA step.

Settings of bench.py's training workload: 8 rotating device-resident batches, the front-end running ahead
(tcr_step_args::input_resident), --warmup steps, then --steps timed steps between two CUDA events; eager launches, as in
bench.py.  A separate, untimed pass with tcr_profile enabled gives the `update` kernel's mean time (CUDA events around every
launch, so it is not part of the ms/step figure).  One JSON line per (model, rule) on stdout; the first line names the GPU
and its power limit.  Under torch.distributed.run every rank steps (peer-memory exchange) and rank 0 prints.

    python tools/optimizer_step_bench.py [--steps 200 --warmup 20] [--shapes r8,r14]
    python -m torch.distributed.run --nproc-per-node=2 tools/optimizer_step_bench.py --shapes r8
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {"r8": ("TCResNet8", 1.0, 512), "r14": ("TCResNet14", 1.5, 1024)}


def gpu_identity(index):
    import torch
    info = {"gpu": torch.cuda.get_device_name(index)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit,power.max_limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout.strip()
        limit, max_limit, sm = (x.strip() for x in q.split(","))
        info.update(power_limit_w=float(limit), power_max_limit_w=float(max_limit), sm_max_mhz=float(sm))
    except Exception as e:                      # the query is informational only
        info["power_limit_w"] = f"unavailable ({type(e).__name__})"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--shapes", default="r8,r14")
    ap.add_argument("--rules", default="mom,adam,rmsprop,adam+ema")
    ap.add_argument("--profile-steps", type=int, default=20)
    a = ap.parse_args()

    import torch
    import tcresnet_b200  # noqa: F401
    from tcresnet_b200.engine import Engine, Optimizer

    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        print(json.dumps(dict(gpu_identity(local), n_gpus=world, steps=a.steps, warmup=a.warmup)), flush=True)
    rules = {"mom": Optimizer("mom", momentum=0.9), "adam": Optimizer.adam(), "rmsprop": Optimizer.rmsprop(),
             "adam+ema": Optimizer.adam(ema_decay=0.999)}

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    for shape in a.shapes.split(","):
        model, width, n = SHAPES[shape]
        eng = Engine(model=model, width_multiplier=width, max_batch=n, dropout_keep_prob=0.5, device=local)
        if world > 1:
            eng.attach_process_group()
        gen = torch.Generator(device=dev).manual_seed(1234 + rank)
        wavs = [torch.rand(n, 16000, device=dev, generator=gen) * 2 - 1 for _ in range(8)]
        labels = torch.randint(0, 12, (8, n), device=dev, generator=torch.Generator(device=dev).manual_seed(4321))
        hots = [torch.nn.functional.one_hot(labels[i], 12).float().contiguous() for i in range(8)]
        losses = torch.zeros(2, device=dev)
        for rule in a.rules.split(","):
            opt = rules[rule]
            params, slots, moving = eng.new_variables(seed=0)
            st = eng.new_optimizer_state(opt, params, slots)
            lr = 0.1 if opt.kind == "mom" else 1e-3

            def step(i):
                eng.train_step(wavs[i % 8], hots[i % 8], params, None, moving, lr, weight_decay=1e-3, dropout_seed=i * world + rank,
                               losses=losses, input_resident=True, optimizer=opt, state=st)
            for i in range(a.warmup):
                step(i)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(a.steps):
                step(a.warmup + i)
            e1.record()
            barrier()
            ms = e0.elapsed_time(e1) / a.steps
            eng.profile(True)
            for i in range(a.profile_steps):
                step(i)
            torch.cuda.synchronize()
            stats = eng.profile_read()
            eng.profile(False)
            upd_ms, upd_n = stats.get("update", (float("nan"), 0))
            if rank == 0:
                print(json.dumps({"model": f"{model}-{width}", "batch_per_gpu": n, "n_gpus": world, "rule": rule,
                                  "ms_per_step": round(ms, 4), "utt_per_s": round(n * world / (ms * 1e-3), 1),
                                  "update_kernel_us": round(upd_ms / max(upd_n, 1) * 1e3, 2),
                                  "update_kernel_note": "mean of a separate tcr_profile pass (events around each launch)",
                                  "final_total_loss": round(float(losses[0].item()), 5),
                                  "exchange": getattr(eng, "exchange", "none (1 GPU)") if world > 1 else "none (1 GPU)"}), flush=True)
            barrier()
        eng.close()
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
