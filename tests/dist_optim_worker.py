"""Worker for the 2-GPU optimizer test (launched by tests/test_optimizers_gpu.py under torch.distributed.run).

One rank per GPU, 16 utterances each, Adam with EMA through engine.train_step.  The step averages the ranks' gradients
(peer memory, or ncclAllReduce with TCR_P2P=0) and applies Adam to that mean: every step's update must equal the fp64 rule on
the mean gradient the step reports, the first step's mean gradient must equal the oracle's shard-wise mean, and after 4 steps
parameters, m, v, the beta powers and the shadows must be bit-identical on every rank.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import tcresnet_b200  # noqa: E402,F401
from oracle import optim_oracle as OO  # noqa: E402
from oracle import tcr_oracle as O  # noqa: E402
from parity_cases import perturbed_variables  # noqa: E402


def rel(a, b):
    b = np.asarray(b, np.float64)
    return float(np.abs(np.asarray(a, np.float64) - b).max() / max(np.abs(b).max(), 1e-30))


def main():
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    per = 16
    spec = O.build_spec("TCResNet8", 1.0, 49)
    params, moving = perturbed_variables(spec)
    wav, onehot = O.synthetic_batch(per * world)
    feat = O.mfcc(wav, 640, 320)
    lr, wd = 0.01, 1e-3
    from tcresnet_b200.engine import Engine, Optimizer
    eng = Engine(max_batch=per, dropout_keep_prob=1.0)
    eng.attach_process_group()
    dev = eng.device
    opt = Optimizer.adam(ema_decay=0.999)
    p = torch.from_numpy(O.flatten_vars(spec, params)).to(dev)
    mv = torch.from_numpy(O.flatten_moving(spec, moving)).to(dev)
    st = eng.new_optimizer_state(opt, p)
    lo, hi = rank * per, (rank + 1) * per
    x, y = torch.from_numpy(wav[lo:hi]).to(dev), torch.from_numpy(onehot[lo:hi]).to(dev)
    un = lambda t: O.unflatten_vars(spec, t.cpu().numpy())
    p_ref = un(p)
    s_ref = dict(m=un(st.slots), v=un(st.slots2), beta1_power=np.float64(np.float32(0.9)), beta2_power=np.float64(np.float32(0.999)),
                 ema=un(st.ema))
    errs = {}
    for step in range(4):
        before = O.unflatten_vars(spec, p.cpu().numpy())
        out = eng.train_step(x, y, p, None, mv, lr, weight_decay=wd, dropout_seed=step, want_grads=True, optimizer=opt, state=st)
        torch.cuda.synchronize()
        g = out["grads"].cpu().numpy().astype(np.float64)
        if step == 0:
            shard = []
            for r in range(world):
                logits, cache = O.forward(spec, before, moving, feat[r * per:(r + 1) * per], True)
                shard.append(O.flatten_vars(spec, O.backward(spec, before, cache, logits, onehot[r * per:(r + 1) * per], wd), np.float64))
            errs["grad0"] = rel(g, np.mean(shard, axis=0))
        p_new, s_new = OO.adam_update(p_ref, O.unflatten_vars(spec, g), s_ref, lr)
        s_new["ema"] = OO.ema_update(s_ref["ema"], p_new, 0.999)
        p_ref, s_ref = p_new, s_new
        fl = lambda d: O.flatten_vars(spec, d, np.float64)
        errs[f"params{step}"] = rel(p.cpu().numpy(), fl(p_ref))
        errs[f"m{step}"] = rel(st.slots.cpu().numpy(), fl(s_ref["m"]))
        errs[f"v{step}"] = rel(st.slots2.cpu().numpy(), fl(s_ref["v"]))
        errs[f"ema{step}"] = rel(st.ema.cpu().numpy(), fl(s_ref["ema"]))
        errs[f"powers{step}"] = rel(st.scalars.cpu().numpy(), [s_ref["beta1_power"], s_ref["beta2_power"]])
    assert all(v < 1e-4 for v in errs.values()), f"rank {rank}: {errs}"
    for name, t in (("params", p), ("m", st.slots), ("v", st.slots2), ("powers", st.scalars), ("ema", st.ema)):
        gathered = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(gathered, t)
        assert all(torch.equal(a, gathered[0]) for a in gathered), f"replicas diverged in {name}"
    if rank == 0:
        worst = max(errs.items(), key=lambda kv: kv[1])
        print(f"exchange={eng.exchange} world={world}: adam+ema, worst rel err {worst[0]} {worst[1]:.2e}, replicas bit-identical "
              f"after 4 steps")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
