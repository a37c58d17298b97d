"""GPU parity: multi-tensor LAMB (3 launches) vs the CPU oracle (oracle/lamb_oracle.*), through the
FusedLAMBAMP boundary.  Tolerance 1e-5 rel on moments (north_star), 1e-5 on parameters."""
import copy
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SHAPES = [[(1024, 1024), (4096, 1024), (333, 77), (5,), (2, 1024)], [(1024,), (2,), (4096,), (3, 3, 3)]]


def _make(dtype, seed=0):
    rng = np.random.default_rng(seed)
    params = [[torch.nn.Parameter(torch.from_numpy(rng.standard_normal(s).astype(np.float32) * 0.05).cuda().to(dtype))
               for s in grp] for grp in SHAPES]
    return params, rng


def _oracle_groups(params, wds=(0.01, 0.0), lr=2e-3):
    return [dict(params=[p.detach().float().cpu().numpy().copy() for p in grp], grads=None,
                 exp_avg=[np.zeros(tuple(p.shape), np.float32) for p in grp],
                 exp_avg_sq=[np.zeros(tuple(p.shape), np.float32) for p in grp],
                 lr=lr, betas=(0.9, 0.999), eps=1e-6, weight_decay=wd, step=0, bias_correction=True, grad_averaging=True)
            for grp, wd in zip(params, wds)]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("scale", [1.0, 65536.0])
def test_lamb_matches_oracle(dtype, scale):
    from deeplearningexamples_b200.lamb import FusedLAMBAMP
    from oracle import lamb_oracle as LO
    params, rng = _make(dtype)
    opt = FusedLAMBAMP([{'params': params[0], 'weight_decay': 0.01}, {'params': params[1], 'weight_decay': 0.0}], lr=2e-3)
    opt.setup_fp32_params()
    og = _oracle_groups(params)
    scaler = torch.amp.GradScaler("cuda", init_scale=scale, growth_interval=10**9)
    for it in range(5):
        gmag = 10.0 if it == 2 else 1e-2          # iteration 2 exercises global-norm clipping
        for grp, ogrp in zip(params, og):
            ogrp["grads"] = []
            for p in grp:
                g = (rng.standard_normal(tuple(p.shape)).astype(np.float32) * gmag)
                gt = (torch.from_numpy(g).cuda() * scale).to(dtype)
                p.grad = gt
                ogrp["grads"].append(gt.float().cpu().numpy())
        scaler._lazy_init_scale_growth_tracker(torch.device("cuda")) if scaler._scale is None else None
        opt.step(grad_scaler=scaler)
        r = LO.lamb_step(og, scale=scale)
        assert not r["found_inf"] and opt._found_inf.item() == 0.0
        assert opt._global_grad_norm.item() == pytest.approx(r["global_grad_norm"], rel=1e-5)
    for gi, (grp, ogrp) in enumerate(zip(params, og)):
        assert opt.param_groups[gi]['step'].item() == ogrp["step"] == 5
        for pi, p in enumerate(grp):
            st = opt.state[p]
            np.testing.assert_allclose(st['exp_avg'].cpu().numpy(), ogrp["exp_avg"][pi], rtol=1e-5, atol=1e-9)
            np.testing.assert_allclose(st['exp_avg_sq'].cpu().numpy(), ogrp["exp_avg_sq"][pi], rtol=1e-5, atol=1e-12)
            master = opt.param_groups_fp32[gi]['params'][pi] if dtype == torch.bfloat16 else p.data
            np.testing.assert_allclose(master.cpu().numpy(), ogrp["params"][pi], rtol=1e-5, atol=1e-7)
            if dtype == torch.bfloat16:   # model copy is the bf16 rounding of the fp32 master
                assert torch.equal(p.data, master.to(torch.bfloat16))


def test_lamb_overflow_skips_step_and_registers_found_inf():
    from deeplearningexamples_b200.lamb import FusedLAMBAMP
    params, rng = _make(torch.bfloat16, seed=1)
    opt = FusedLAMBAMP([{'params': params[0]}, {'params': params[1], 'weight_decay': 0.0}], lr=1e-3)
    opt.setup_fp32_params()
    scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 20)
    for grp in params:
        for p in grp:
            p.grad = torch.randn_like(p)
    params[0][1].grad[7, 3] = float("inf")
    before = [p.detach().clone() for grp in params for p in grp]
    scaler._lazy_init_scale_growth_tracker(torch.device("cuda"))
    scaler.step(opt)                       # GradScaler sees _step_supports_amp_scaling and passes itself
    found = scaler._found_inf_per_device(opt)
    assert sum(v.item() for v in found.values()) == 1.0
    scaler.update()
    assert scaler.get_scale() == 2.0 ** 19
    assert all(torch.equal(a, p) for a, p in zip(before, [p for grp in params for p in grp]))
    assert all(g['step'].item() == 0 for g in opt.param_groups)
    assert all((opt.state[p]['exp_avg'] == 0).all() for grp in params for p in grp)


def test_lamb_state_dict_round_trip_keeps_fp32_moments():
    from deeplearningexamples_b200.lamb import FusedLAMBAMP
    params, rng = _make(torch.bfloat16, seed=2)
    mk = lambda ps: FusedLAMBAMP([{'params': ps[0]}, {'params': ps[1], 'weight_decay': 0.0}], lr=1e-3)
    opt = mk(params); opt.setup_fp32_params()
    for grp in params:
        for p in grp:
            p.grad = torch.randn_like(p) * 1e-2
    opt.step()
    sd = opt.state_dict()
    assert sd['param_groups'][0]['step'].dtype == torch.int32 and sd['param_groups'][0]['lr'].is_cuda
    params2 = copy.deepcopy(params)
    opt2 = mk(params2); opt2.load_state_dict(sd); opt2.setup_fp32_params()
    for g1, g2 in zip(opt.param_groups, opt2.param_groups):
        assert g2['step'].item() == g1['step'].item() == 1
        for p1, p2 in zip(g1['params'], g2['params']):
            assert opt2.state[p2]['exp_avg'].dtype == torch.float32
            assert torch.equal(opt.state[p1]['exp_avg_sq'], opt2.state[p2]['exp_avg_sq'])
    # the driver zeroes step / refills lr in the *saved* dict when changing phase (run_pretraining.py:442-445)
    for group in sd['param_groups']:
        group['step'].zero_(); group['lr'].fill_(5e-5)


def test_lamb_full_bert_large_shape_list_properties():
    """BASELINE full size (398 tensors, 336M params): size-independent properties -- zero gradient with zero
    moments leaves decayed weights shrinking by exactly lr (trust ratio 1/wd * wd) and no-decay ones unchanged;
    the model copy equals bf16(master)."""
    from deeplearningexamples_b200.lamb import FusedLAMBAMP
    from oracle import bert_oracle as O
    shapes = O.param_shapes(O.BERT_LARGE)
    no_decay = ['bias', 'gamma', 'beta', 'LayerNorm']
    decay, nodecay = [], []
    g = torch.Generator(device="cuda").manual_seed(0)
    for name, shp in shapes.items():
        p = torch.nn.Parameter((torch.randn(shp, device="cuda", generator=g) * 0.02 + 0.01).to(torch.bfloat16))
        (nodecay if any(nd in name for nd in no_decay) else decay).append(p)
    assert len(decay) == 150 and len(nodecay) == 248
    opt = FusedLAMBAMP([{'params': decay, 'weight_decay': 0.01}, {'params': nodecay, 'weight_decay': 0.0}], lr=1e-2)
    opt.setup_fp32_params()
    for p in decay + nodecay:
        p.grad = torch.zeros_like(p)
    masters0 = [m.clone() for grp in opt.param_groups_fp32 for m in grp['params']]
    opt.step()
    torch.cuda.synchronize()
    assert opt._global_grad_norm.item() == 0.0
    masters1 = [m for grp in opt.param_groups_fp32 for m in grp['params']]
    for i, (m0, m1) in enumerate(zip(masters0, masters1)):
        if i < 150:      # u = wd*p, |u| = wd|p|, ratio = lr/wd, p_new = p - lr*p
            torch.testing.assert_close(m1, m0 * (1 - 1e-2), rtol=2e-6, atol=1e-8)
        else:            # u = 0 => p unchanged
            assert torch.equal(m1, m0)
    for p, m in zip(decay + nodecay, masters1):
        assert torch.equal(p.data, m.to(torch.bfloat16))


def test_oracle_vs_reference_kernel(golden_dir):
    """Pins the CPU oracle (and our kernel) to the reference's OWN CUDA kernels: fused_lamb_CUDA.multi_tensor_l2norm /
    multi_tensor_lamb driven exactly as fused_lamb.py:166-258 does, on a B200, for this sequence of steps.  What they computed is
    stored in tests/golden/lamb_reference_kernel.npz (tests/golden/make_lamb_golden.py), at fixed positions of each tensor."""
    from deeplearningexamples_b200.lamb import FusedLAMBAMP
    from oracle import lamb_oracle as LO
    gold = np.load(os.path.join(golden_dir, "lamb_reference_kernel.npz"))
    rng = np.random.default_rng(int(gold["seed"]))
    shapes = [tuple(int(d) for d in gold[f"shape{i}"]) for i in range(sum(k.startswith("shape") for k in gold.files))]
    host_p = [rng.standard_normal(s).astype(np.float32) * 0.05 for s in shapes]
    wd, lr, scale = float(gold["wd"]), float(gold["lr"]), float(gold["scale"])
    # --- ours
    ours = [torch.nn.Parameter(torch.from_numpy(a.copy()).cuda()) for a in host_p]
    opt = FusedLAMBAMP([{'params': ours, 'weight_decay': wd}], lr=lr)
    opt.setup_fp32_params()
    scaler = torch.amp.GradScaler("cuda", init_scale=scale, growth_interval=10 ** 9)
    scaler._lazy_init_scale_growth_tracker(torch.device("cuda"))
    # --- oracle
    og = [dict(params=[a.copy() for a in host_p], grads=None, exp_avg=[np.zeros_like(a) for a in host_p],
               exp_avg_sq=[np.zeros_like(a) for a in host_p], lr=lr, betas=(0.9, 0.999), eps=1e-6, weight_decay=wd, step=0,
               bias_correction=True, grad_averaging=True)]
    for it in range(int(gold["steps"])):
        gs = [(rng.standard_normal(s).astype(np.float32) * (5.0 if it == 1 else 1e-2) * scale) for s in shapes]
        for p, g in zip(ours, gs):
            p.grad = torch.from_numpy(g.copy()).cuda()
        og[0]["grads"] = [g.copy() for g in gs]
        opt.step(grad_scaler=scaler)
        LO.lamb_step(og, scale=scale)
        assert float(gold["gnorm"][it]) == pytest.approx(LO.sumsq(np.concatenate([g.ravel() for g in gs]))[0] ** 0.5, rel=1e-5)
    for i in range(len(shapes)):
        # reference kernel is built with --use_fast_math (approximate div/sqrt): compare at 1e-4 to the IEEE oracle,
        # ours at 1e-5 (north_star tolerance on fp32 LAMB moments)
        idx = gold[f"idx{i}"]
        np.testing.assert_allclose(gold[f"exp_avg{i}"], og[0]["exp_avg"][i].ravel()[idx], rtol=1e-4, atol=1e-9)
        np.testing.assert_allclose(gold[f"exp_avg_sq{i}"], og[0]["exp_avg_sq"][i].ravel()[idx], rtol=1e-4, atol=1e-12)
        np.testing.assert_allclose(gold[f"param{i}"], og[0]["params"][i].ravel()[idx], rtol=1e-4, atol=1e-6)
        np.testing.assert_allclose(opt.state[ours[i]]['exp_avg'].cpu().numpy(), og[0]["exp_avg"][i], rtol=1e-5, atol=1e-9)
        np.testing.assert_allclose(opt.state[ours[i]]['exp_avg_sq'].cpu().numpy(), og[0]["exp_avg_sq"][i], rtol=1e-5, atol=1e-12)
        np.testing.assert_allclose(ours[i].detach().cpu().numpy(), og[0]["params"][i], rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_fused_adam_matches_oracle(dtype):
    """dle_adam_step (SQuAD fine-tune optimizer: clip + Adam, bias_correction=False) vs the CPU oracle."""
    from deeplearningexamples_b200.adam import FusedAdam
    from oracle import lamb_oracle as LO
    params, rng = _make(dtype, seed=7)
    opt = FusedAdam([{'params': params[0], 'weight_decay': 0.01}, {'params': params[1], 'weight_decay': 0.0}], lr=3e-3,
                    bias_correction=False, max_grad_norm=1.0)
    opt.setup_fp32_params()
    og = [dict(params=[p.detach().float().cpu().numpy().copy() for p in grp], grads=None,
               exp_avg=[np.zeros(tuple(p.shape), np.float32) for p in grp], exp_avg_sq=[np.zeros(tuple(p.shape), np.float32) for p in grp],
               lr=3e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=wd, step=0, bias_correction=False) for grp, wd in zip(params, (0.01, 0.0))]
    for it in range(4):
        mag = 5.0 if it == 1 else 1e-2                    # iteration 1 clips
        for grp, ogrp in zip(params, og):
            ogrp["grads"] = []
            for p in grp:
                g = torch.from_numpy(rng.standard_normal(tuple(p.shape)).astype(np.float32) * mag).cuda().to(dtype)
                p.grad = g
                ogrp["grads"].append(g.float().cpu().numpy())
        opt.step()
        r = LO.adam_step_numpy(og, max_grad_norm=1.0)
        assert opt._global_grad_norm.item() == pytest.approx(r["global_grad_norm"], rel=1e-5)
    for gi, (grp, ogrp) in enumerate(zip(params, og)):
        for pi, p in enumerate(grp):
            st = opt.state[p]
            np.testing.assert_allclose(st['exp_avg'].cpu().numpy(), ogrp["exp_avg"][pi], rtol=1e-5, atol=1e-9)
            np.testing.assert_allclose(st['exp_avg_sq'].cpu().numpy(), ogrp["exp_avg_sq"][pi], rtol=1e-5, atol=1e-12)
            master = opt.param_groups_fp32[gi]['params'][pi] if dtype == torch.bfloat16 else p.data
            np.testing.assert_allclose(master.cpu().numpy(), ogrp["params"][pi], rtol=2e-5, atol=2e-6)
