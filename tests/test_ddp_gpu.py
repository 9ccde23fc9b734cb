"""GPU, 2 NCCL ranks (skipped on a box with fewer than 2 GPUs): one utterance-sharded data-parallel step of the hot path
equals "N independent micro-batches with averaged gradients" (SURVEY.md §8e) — on the hardware path, not only on gloo."""
import os
import sys

import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _Enc(torch.nn.Module):
    def forward(self, *a, **k):
        raise AssertionError("encoders are not used by hot_path_loss")


def _worker(rank, world, port, q):
    try:
        sys.path.insert(0, ROOT)
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                          LOCAL_RANK=str(rank))
        import torch.distributed as dist
        import multimodal_av_model_b200 as pkg
        from multimodal_av_model_b200 import ddp
        from multimodal_av_model_b200.synthetic import CharTokenizer, make_features
        ddp.init_distributed("nccl")
        dev = torch.device("cuda", rank)
        torch.manual_seed(rank)                     # different init per rank on purpose: the trainer must broadcast rank 0's
        fus = pkg.CrossAttentionFusion(512, 1024, 512)
        dec = pkg.CTCDecoder(1024, 800, blank_id=3)
        tr = pkg.MultimodalTrainer(_Enc(), _Enc(), fus, dec, CharTokenizer(800), device=dev)
        assert tr._reducer is not None and tr.world_size == world
        feats = [make_features(pairs=2, t_v=40, t_enc=99, seed=50 + r, n_samples=32000, dtype=torch.bfloat16)
                 for r in range(world)]

        def loss_of(r):
            fd = {k: [t.to(dev) for t in v] for k, v in feats[r].items()}
            with torch.autocast("cuda", dtype=torch.bfloat16):
                return tr.hot_path_loss(fd["visual"], fd["audio"], fd["middle"], fd["masks"], fd["texts"], fd["lens"])[0]

        named = list(fus.named_parameters()) + [("dec." + k, p) for k, p in dec.named_parameters()]
        got = None
        for _ in range(2):                          # two steps: the second runs with the "unused parameter" set known
            tr._reducer.zero_grad()
            loss_of(rank).backward()
            tr._reducer.finish()
            got = {k: (None if p.grad is None else p.grad.clone()) for k, p in named}
        # parameters are identical on every rank after the constructor's broadcast
        w = fus.fusion_proj.weight.detach().clone()
        ws = [torch.empty_like(w) for _ in range(world)]
        dist.all_gather(ws, w)
        same_params = all(torch.equal(ws[0], t) for t in ws)
        tr._reducer.close()
        acc = {}
        for r in range(world):
            for _, p in named:
                p.grad = None
            loss_of(r).backward()
            for k, p in named:
                if p.grad is not None:
                    acc[k] = acc.get(k, 0) + p.grad / world
        worst = 0.0
        for k, p in named:
            if k not in acc:
                assert got[k] is None, k           # cross_attn_visual: outside the graph, .grad stays None under DDP too
                continue
            err = ((got[k] - acc[k]).abs().max() / (acc[k].abs().max() + 1e-12)).item()
            worst = max(worst, err)
        q.put((rank, same_params, worst, None))
        dist.barrier()
        dist.destroy_process_group()
    except Exception as e:          # surface the failure in the parent instead of a queue timeout
        import traceback
        q.put((rank, False, float("inf"), traceback.format_exc()))


def test_two_rank_nccl_step_equals_mean_of_single_gpu_gradients():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, 29641, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=600) for _ in procs)
    for p in procs:
        p.join(timeout=120)
    for rank, same, worst, tb in res:
        assert tb is None, tb
        assert same, "parameters differ across ranks after the constructor broadcast"
        # same kernels on both sides; the difference is fp32 summation order (split-K atomics, NCCL ring order)
        assert worst < 2e-3, (rank, worst)
