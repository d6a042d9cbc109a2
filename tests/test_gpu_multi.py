"""Two-GPU run of the sampler surface (SURVEY.md §8e): one process per GPU under NCCL, the reference's ceil(bs / world)
slicing (sampler.py:273-277), ONE weight broadcast (rank 1 starts from different weights), a final all-gather — all of it
through resshift_b200.parallel, the same code bench.py --gpus N runs.  Every shard of the gathered batch must equal, bit
for bit, the single-GPU run of that slice on rank 0 (image shards are independent: nothing inside the loop communicates),
and the whole-batch run to rounding.
Skipped on machines with fewer than two devices."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    from resshift_b200 import parallel
    from resshift_b200.config import preset
    from resshift_b200.sampler import ResShiftSampler, make_configs
    from resshift_b200.weights import random_state_dict
    try:
        ucfg, dcfg = preset("tiny")
        dcfg.sf = 1
        # rank r loads different weights: only the broadcast from rank 0 can make the shards agree
        configs = make_configs(ucfg, dcfg, autoencoder=None, state_dict=random_state_dict(ucfg, rank))
        s = ResShiftSampler(configs, sf=1, use_amp=True, seed=7, chop_size=64, chop_stride=64, padding_offset=16)
        assert s.num_gpus == world and dist.is_initialized() and dist.get_backend() == "nccl"
        s.broadcast_weights(src=0)
        batch = 5                                             # uneven: rank 0 gets 3 images, rank 1 gets 2
        g = torch.Generator(device="cuda").manual_seed(99)
        y_all = torch.rand(batch, 3, 64, 64, device="cuda", generator=g) * 2 - 1   # (latent = LQ size: sf 1; 64 = 8 * 2^(levels-1))
        a, b = parallel.shard_range(batch, world, rank)
        s.setup_seed(1234)                                    # same noise stream on every rank ...
        noise_all = torch.randn(s.base_diffusion.num_timesteps + 1, batch, 3, 64, 64, device="cuda")

        def run(y, noise):      # the hot path proper with explicit noise: prior sample + T denoise steps inside librs_b200
            return s.base_diffusion.sample_latent(y, s.model, {"lq": y}, noises=noise).clone()
        local = run(y_all[a:b].contiguous(), noise_all[:, a:b].contiguous())
        full = s.gather_results(local, batch)
        ok, info = True, ""
        if rank == 0:
            # every rank's slice re-run on rank 0 AT THE SLICE'S OWN BATCH SIZE must reproduce the gathered shard bit for bit
            # (same weights after the broadcast, kernels bit-reproducible across GPUs, gather in rank order); the planner
            # picks other tile shapes / split-K factors for other batch sizes, so the whole-batch run agrees to rounding
            # only (see test_batch_independence_at_bench_size)
            ok = full.shape == y_all.shape
            for rr in range(world):
                aa, bb = parallel.shard_range(batch, world, rr)
                again = run(y_all[aa:bb].contiguous(), noise_all[:, aa:bb].contiguous())
                ok = ok and bool(torch.equal(full[aa:bb], again))
            whole = run(y_all, noise_all)
            dmax = (full - whole).abs().max().item()
            ok = ok and dmax <= 2e-2
            info = f"shards bit-identical: {ok}; vs the whole-batch plan max |d| = {dmax:.3e}"
        q.put((rank, ok, info))
    except Exception as exc:                                  # noqa: BLE001 — report instead of hanging the parent
        import traceback
        q.put((rank, False, traceback.format_exc()))
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpu_sampler_shards_equal_single_gpu_run():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=600) for _ in procs)
    for p in procs:
        p.join(timeout=120)
    assert [r[:2] for r in res] == [(0, True), (1, True)], res
