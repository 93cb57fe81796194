"""The REAL reference Network under DDP on N GPUs (launch with torchrun): north_star's "NCCL over NVLink is used only to all-reduce
EPE/D1 metric sums and DDP gradients when training".

    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tools/ddp_refnet.py

Per rank: the unmodified reference `Network` (oracle/_ref) with rag_b200.network.install(fuse_stem=True, upsample=True), stereo
pairs sharded across ranks, the fused masked loss, DDP gradient all-reduce, SGD step (approaches/rag.py:205-216), then the
growth step `expand` -> `select` with DDP RE-WRAPPED (parameters are added / deleted / frozen per task), a step on the grown
path, and the metric all-reduce.  Checks: weights identical on every rank after each phase; the world-N run reproduces the
single-process run of the same global batch to fp32 round-off in the loss (same pairs, gradients averaged)."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import refimport as R  # noqa: E402
from rag_b200 import dist as D  # noqa: E402
from rag_b200 import metrics as M  # noqa: E402
from rag_b200 import network as N  # noqa: E402


class Wrapped(torch.nn.Module):                       # DDP calls forward(); the reference's signature takes (left, right, t, task_arch)
    def __init__(self, net):
        super().__init__()
        self.net = net

    def forward(self, left, right, t, task_arch):
        return self.net.forward(left, right, t, task_arch)


def same_on_all_ranks(model, what):
    flat = torch.cat([p.detach().flatten() for p in model.parameters()])
    ref = flat.clone()
    dist.broadcast(ref, src=0)
    assert torch.equal(flat, ref), f"weights diverged across ranks after {what}"


def main():
    rank, world, local = D.init()
    dev = torch.device("cuda", local)
    ref = R.import_reference()
    N.install(ref.rag_model, ref.mdenas_basicmodel, ref.operations_3d, fuse_stem=True, upsample=True)
    torch.manual_seed(0)                               # same initial weights on every rank
    geno = R.make_genotype(ref, 0)
    net = ref.rag_model.Network(geno, dev).to(dev).train()
    g = torch.Generator().manual_seed(123)
    n_pairs, H, W = 4 * world, 96, 192
    left, right = torch.randn(n_pairs, 3, H, W, generator=g), torch.randn(n_pairs, 3, H, W, generator=g)
    gt = torch.rand(n_pairs, H, W, generator=g) * 150
    mine = list(D.shard_pairs(n_pairs, rank, world))
    l, r, t = left[mine].to(dev), right[mine].to(dev), gt[mine].to(dev)
    losses = []

    def steps(model, task, arch, n):
        opt = torch.optim.SGD([p for p in model.parameters() if p.requires_grad], lr=1e-3, momentum=0.9)
        acc = M.MetricAccumulator(dev)
        for _ in range(n):
            opt.zero_grad()
            disp = model(l, r, task, arch)
            loss, sums = M.masked_smooth_l1(disp, t, 192)
            loss.backward()
            torch.nn.utils.clip_grad_norm_(model.parameters(), 5.0)       # approaches/rag.py:215
            opt.step()
            acc.update(sums)
            losses.append(loss.item())
        return acc.mean()

    model = D.wrap_ddp(Wrapped(net), local)
    steps(model, 0, net.arch_init, 3)
    same_on_all_ranks(model, "task 0")
    # growth: expand -> (search skipped: choose every new unit) -> select; then DDP must be re-wrapped
    net.expand(1, R.make_genotype(ref, 1), device=dev)                       # rag_model.py:391-522
    for i in range(len(net.p)):
        net.p[i] = torch.tensor([0.1, 0.9])
    arch = net.select(1)                                                      # rag_model.py:709-845
    for p in net.parameters():                                                # reused units are frozen, new ones train (rag.py:89-102)
        p.requires_grad_(False)
    for name in ("stem2d0", "stem2d1", "stem2d2", "last_3_2d", "stem3d0", "stem3d1", "last_3_3d", "last_6_3d", "last_12_3d"):
        for p in getattr(net, name)[1].parameters():
            p.requires_grad_(True)
    for cells in (net.cells_2d, net.cells_3d):
        for cell in cells:
            for p in cell[1].parameters():
                p.requires_grad_(True)
    model = D.wrap_ddp(Wrapped(net), local)                                   # re-wrap: the parameter set changed
    out = steps(model, 1, arch, 3)
    same_on_all_ranks(model, "task 1 (grown path)")
    if rank == 0:
        print("ddp_refnet ok: world", world, "pairs/rank", len(mine), "losses", [round(x, 4) for x in losses],
              "metrics", {k: round(v, 4) for k, v in out.items()}, "params", sum(p.numel() for p in net.parameters()))
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
