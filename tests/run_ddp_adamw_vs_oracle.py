"""Multi-GPU AdamW parity helper (launched under torchrun by test_multi_gpu_adamw_matches_oracle,
or by hand:  torchrun --nproc-per-node 2 tests/run_ddp_adamw_vs_oracle.py).

The AdamW rows of run_ddp_vs_oracle.py's scheme: N ranks train the toy 2-task model with
``decoupled_weight_decay=True`` through NCCL + K2 (with and without clip) and through the fused
NVLS kernel K7 where multicast is available; rank 0 checks the weights against single-process
``torch.optim.AdamW`` on the CPU fed the concatenated batch, and the K7 run against the NCCL run."""
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import frl_b200  # noqa: E402,F401
from frl_b200 import fused_optim, grad_sync, synthetic  # noqa: E402
from frl_b200.arena import ParamArena  # noqa: E402
from frl_b200.types import OptAlgorithm, OptimOpts  # noqa: E402
from oracle import ref_loop  # noqa: E402
from adamw_oracle import make_optimizer  # noqa: E402

LR, WD = 0.02, 0.05


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    torch.backends.cuda.matmul.allow_tf32 = False
    ns = synthetic.api_namespace("frl_b200")
    from frl_b200.symm import make_link, try_make_allocator
    alloc = try_make_allocator(dev, world)
    if rank == 0:
        print("NVLS_AVAILABLE", alloc is not None, flush=True)
    combos = [(0.0, False), (0.05, False)] + ([(0.0, True)] if alloc is not None else [])
    nccl_weights = None
    for clip, nvls in combos:
        torch.manual_seed(123 + rank)                 # different init per rank: broadcast must fix
        problem = synthetic.make_toy_problem(ns, "/tmp/unused")
        model = problem.get_model().to(dev)
        crit = problem.get_criterion().to(dev)
        arena = ParamArena(model.parameters(), crit.parameters(), device=dev,
                           shared_allocator=alloc if nvls else None)
        opt = fused_optim.create_fused_optimizer(
            arena, OptimOpts(algo=OptAlgorithm.ADAM, lr=LR, weightDecay=WD), decoupled_weight_decay=True)
        link = make_link(alloc, arena.grad, arena.master, max_blocks=8) if nvls else None
        pipe = grad_sync.GradBucketPipeline(arena, opt, world_size=world, clip_norm=clip,
                                            bucket_cap_mb=0.02, first_bucket_mb=0.005, nvls_link=link)
        assert (pipe.nvls is not None) == bool(nvls)
        pipe.broadcast_parameters(0)
        assert len(pipe.buckets) >= 3
        g = torch.Generator().manual_seed(7)
        B = 32 * world
        batches = [(torch.rand(B, 64, generator=g), torch.randn(B, 4, generator=g),
                    torch.randint(0, 10, (B,), generator=g)) for _ in range(4)]
        model.train()
        for x, yr, yc in batches:
            sl = slice(rank, None, world)
            out = model([x[sl].to(dev)])
            total, _ = crit(out, [(yr[sl].to(dev),), (yc[sl].to(dev),)])
            pipe.begin_step()
            total.backward()
            pipe.finish_step()
        torch.cuda.synchronize()
        mine = torch.cat([p.detach().reshape(-1).float() for p in model.parameters()])
        gathered = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(gathered, mine)
        if rank == 0:
            for other in gathered[1:]:
                assert torch.equal(other, gathered[0]), "replicas diverged"
            torch.manual_seed(123)
            ref_problem = synthetic.make_toy_problem(ns, "/tmp/unused")
            ref = ref_problem.get_model()
            rc = ref_problem.get_criterion()
            ropt = make_optimizer(ref.parameters(), ref_loop.OptimSpec(algo="adam", lr=LR, weight_decay=WD),
                                  decoupled_weight_decay=True)
            ref.train()
            for x, yr, yc in batches:
                out = ref([x])
                total, _ = ref_loop.parallel_criterion(list(rc.loss_modules), list(rc.loss_weights),
                                                       list(rc.loss_names), out, [(yr,), (yc,)])
                ropt.zero_grad()
                total.backward()
                if clip:
                    torch.nn.utils.clip_grad_norm_(ref.parameters(), clip)
                ropt.step()
            want = torch.cat([p.detach().reshape(-1) for p in ref.parameters()])
            # the Adam bound of run_ddp_vs_oracle.py: m/(sqrt(v)+eps) amplifies fp32 rounding where
            # v is tiny; the decoupled decay itself is a single rounding of p * (1 - lr*wd)
            np.testing.assert_allclose(mine.cpu().numpy(), want.numpy(), rtol=1e-3, atol=5e-5)
            if clip == 0.0 and not nvls:
                nccl_weights = mine.clone()
            if nvls:
                torch.testing.assert_close(mine, nccl_weights, rtol=1e-4, atol=5e-6)
            print("DDP_ADAMW_PARITY_OK", clip, "nvls" if nvls else "nccl", "world", world, flush=True)
        pipe.sync_sharded_state()
        pipe.remove_hooks()
        dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
