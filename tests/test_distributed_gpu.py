"""2-rank NCCL equivalence of the PRODUCT path (BASELINE.md 3.C, SURVEY.md 8e): one optimizer step of the CUDA model under torch DDP on
two GPUs, each rank on its half of a batch, must equal the 1-rank step on the concatenated batch (dropout off).

Every per-token computation is identical in both runs (sequences never interact); only the token-dimension reductions (weight /
bias / LayerNorm gradients, the loss mean) are split across ranks.  With fp32 parameters those reductions are fp32 sums of identical
bf16 products in a different order, so gradients, LAMB moments and parameters agree to ~1e-6 (bar: 1e-5, the north_star's LAMB
tolerance).  With bf16 parameters each rank's gradient is rounded to bf16 before the allreduce, so the bar is the bf16 one.
Skipped when fewer than two GPUs are visible (gpurun --gpus 2 runs it)."""
import os
import socket

import pytest
import torch

pytestmark = pytest.mark.gpu

CFG = dict(hidden_size=256, num_hidden_layers=2, num_attention_heads=4, intermediate_size=1024, vocab_size=1024,
           max_position_embeddings=128, type_vocab_size=2, hidden_act="gelu", initializer_range=0.02,
           hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
B, S, P = 8, 128, 10


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _one_step(dtype, device, distributed, batch):
    from deeplearningexamples_b200 import ops, training as T
    ops.manual_seed(7)
    model, opt, scaler, sched, crit, _ = T.prepare_model_and_optimizer(CFG, device, learning_rate=1e-3, max_steps=10, warmup_proportion=0.1,
                                                                      distributed=distributed, dtype=dtype, seed=11, init_loss_scale=2 ** 10)
    model.train()
    loss = T.take_training_step(scaler, model, crit, batch)
    core = model.module if hasattr(model, "module") else model
    grads = {k: p.grad.detach().float().clone() for k, p in core.named_parameters() if p.grad is not None}
    T.take_optimizer_step(sched, opt, scaler)
    torch.cuda.synchronize()
    state, masters = {}, {}
    named = dict(core.named_parameters())
    name_of = {id(p): k for k, p in named.items()}
    for g, g32 in zip(opt.param_groups, opt.param_groups_fp32):
        for p, p32 in zip(g["params"], g32["params"]):
            k = name_of[id(p)]
            st = opt.state[p]
            state[k] = (st["exp_avg"].clone(), st["exp_avg_sq"].clone())
            masters[k] = (p32 if p32 is not None else p.data).detach().float().clone()
    return loss.detach().float().item(), grads, state, masters, int(opt.param_groups[0]["step"].item())


def _worker(rank, world, port, dtype_name, out_path):
    import torch.distributed as dist
    from deeplearningexamples_b200 import training as T
    dtype = getattr(torch, dtype_name)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    device = torch.device("cuda", rank)
    dist.init_process_group(backend="nccl", init_method="env://", world_size=world, rank=rank, device_id=device)
    full = T.synthetic_batch(B, S, CFG["vocab_size"], P, seed=5, full_mask=False)
    half = B // world
    mine = {k: v[rank * half:(rank + 1) * half].to(device) for k, v in full.items()}
    loss, grads, state, masters, step = _one_step(dtype, device, True, mine)
    losses = [None] * world
    dist.all_gather_object(losses, loss)
    if rank == 0:
        torch.save(dict(losses=losses, grads={k: v.cpu() for k, v in grads.items()},
                        state={k: (a.cpu(), b.cpu()) for k, (a, b) in state.items()},
                        masters={k: v.cpu() for k, v in masters.items()}, step=step), out_path)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("dtype_name,tol", [("float32", 1e-5), ("bfloat16", 2e-2)])
def test_two_rank_ddp_step_equals_one_rank_step_on_concatenated_batch(tmp_path, dtype_name, tol):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from deeplearningexamples_b200 import training as T
    out = str(tmp_path / "rank0.pt")
    mp.spawn(_worker, args=(2, _free_port(), dtype_name, out), nprocs=2, join=True)
    two = torch.load(out, weights_only=False)
    device = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    full = {k: v.to(device) for k, v in T.synthetic_batch(B, S, CFG["vocab_size"], P, seed=5, full_mask=False).items()}
    loss, grads, state, masters, step = _one_step(getattr(torch, dtype_name), device, False, full)
    assert step == two["step"] == 1
    # equal-sized shards with equally many masked positions: the global loss is the mean of the rank losses
    assert abs(sum(two["losses"]) / 2 - loss) < 1e-4 * abs(loss)

    def rel(a, b):
        return ((a.float().cpu() - b.float().cpu()).norm() / b.float().cpu().norm().clamp_min(1e-20)).item()

    for k, g1 in grads.items():
        if k.endswith("key.bias"):
            continue                                    # analytically zero gradient
        assert rel(two["grads"][k], g1) < max(tol, 2e-5), ("grad", k, rel(two["grads"][k], g1))
        m2, v2 = two["state"][k]
        m1, v1 = state[k]
        assert rel(m2, m1) < max(tol, 2e-5) and rel(v2, v1) < max(2 * tol, 4e-5), ("moments", k, rel(m2, m1), rel(v2, v1))
        # parameters.  fp32: identical up to summation order.  bf16: the first LAMB step is sign-like (m^ / sqrt(v^) = g / |g|), so a
        # gradient entry that rounds to opposite signs on the two paths moves that element by up to 2 * lr * trust-ratio; zero-initialised
        # parameters (biases) consist of nothing but this update, hence an absolute bound of two step sizes next to the relative one
        diff = (two["masters"][k].float().cpu() - masters[k].float().cpu()).abs().max().item()
        if dtype_name == "float32":
            assert rel(two["masters"][k], masters[k]) < 1e-5, ("param", k, rel(two["masters"][k], masters[k]))
        else:
            assert diff <= 2.2e-3 * max(1.0, masters[k].float().abs().max().item()), ("param", k, diff)
