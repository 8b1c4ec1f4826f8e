"""One rank of the multi-rank Ranger test (launched by torchrun from test_ranger.py): Ranger through
``train.make_optimizer`` on ``train_dist.train_step``, with clipping and dropout 0.5, for 13 steps (rectification and
the first Lookahead at step 6, the second Lookahead at 12); the last step has one site, so the other ranks contribute
no gradient there.  Rank 0 prints one JSON line with every rank's parameter digest."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from deepsignal_plant_b200 import synthetic  # noqa: E402
from deepsignal_plant_b200 import freq_dist as fd  # noqa: E402
from deepsignal_plant_b200 import train as tr  # noqa: E402
from deepsignal_plant_b200 import train_dist as td  # noqa: E402
from train_dist_worker import KEYS, build, emit  # noqa: E402

STEPS = 13


def main():
    dist.init_process_group("gloo")
    device = int(os.environ.get("LOCAL_RANK", "0")) % torch.cuda.device_count()
    torch.cuda.set_device(device)
    grp = fd.TorchGroup()
    world, rank = grp.world, grp.rank
    dev = torch.device("cuda", device)
    torch.cuda.manual_seed(99 + rank)
    model = build(64, 0.5, dev, state_mode="philox", seed=rank).train()
    n = 96
    f = synthetic.make_features(n, 13, 16, seed=3)
    data = {k: torch.from_numpy(f[k]).to(dev) for k in KEYS}
    data["labels"] = torch.from_numpy(np.random.default_rng(4).integers(0, 2, n)).to(dev)
    params = list(model.parameters())
    ex = td.GradientExchange(rank, world, device, sum(q.numel() for q in params), grp.all_gather_object)
    opt = tr.make_optimizer("Ranger", params, 1e-3)
    weight = torch.tensor([1.0, 1.7], device=dev)
    losses = []
    for s in range(STEPS):
        idx = torch.arange(n, device=dev) if s < STEPS - 1 else torch.tensor([n - 1], device=dev)
        losses.append(float(td.train_step(model, params, data, idx, weight, rank, world, ex, opt, KEYS)))
    ex.close()
    steps = sorted({opt.state[p]["step"] for p in params})
    emit(grp, {"digest": td.param_digest(model), "losses": losses, "steps": steps},
         lambda every: {"ok": len({e["digest"] for e in every}) == 1 and all(e["steps"] == [STEPS] for e in every)})
    grp.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
