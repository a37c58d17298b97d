"""Record what the reference's OWN fused LAMB CUDA kernels compute for the sequence of
tests/test_lamb_gpu.py::test_oracle_vs_reference_kernel, so that test runs without them.

    python tests/golden/make_lamb_golden.py [out.npz]        # default: tests/golden/lamb_reference_kernel.npz

Needs a B200 and the reference's fused_lamb_CUDA extension, built from the reference sources into oracle/_ref by
oracle/build_ref.py.  fused_lamb_CUDA.multi_tensor_l2norm / multi_tensor_lamb are driven as fused_lamb.py:148-258 drives
them (fp32 4-list form) for three steps; iteration 1 has large gradients so global-norm clipping is exercised.

Stored (float32 unless noted): the case (seed, shapes, lr, wd, scale), the global gradient norm the reference kernel
computed at each step, and exp_avg / exp_avg_sq / param after the last step at fixed positions of each tensor (all of a
tensor of at most 4096 elements, else 4096 positions drawn with seed 0; idx<i> is int32).
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

CASE = dict(seed=5, shapes=[(1024, 512), (300, 7), (4096,), (2,)], wd=0.01, lr=3e-3, scale=1024.0, steps=3)
SAMPLE = 4096


def inputs(case):
    """Initial parameters and the scaled gradients of every step, in the order the test draws them."""
    rng = np.random.default_rng(case["seed"])
    params = [rng.standard_normal(s).astype(np.float32) * 0.05 for s in case["shapes"]]
    grads = [[rng.standard_normal(s).astype(np.float32) * (5.0 if it == 1 else 1e-2) * case["scale"] for s in case["shapes"]]
             for it in range(case["steps"])]
    return params, grads


def main(out):
    from oracle import build_ref
    ext = build_ref.load_module()
    if ext is None:
        raise SystemExit("oracle/_ref/fused_lamb_CUDA.so is not built (python oracle/build_ref.py)")
    params, grads = inputs(CASE)
    rp = [torch.from_numpy(a.copy()).cuda() for a in params]
    rm, rv = [torch.zeros_like(a) for a in rp], [torch.zeros_like(a) for a in rp]
    rstep = torch.zeros(1, dtype=torch.int, device="cuda")
    noop = torch.zeros(1, dtype=torch.int, device="cuda")
    lr_t = torch.tensor(CASE["lr"], device="cuda")
    gnorms = []
    for gs in grads:
        rg = [torch.from_numpy(g.copy()).cuda() for g in gs]
        found_inf = torch.zeros(1, device="cuda")
        sc = torch.full((1,), CASE["scale"], device="cuda")
        inv_scale = sc.double().reciprocal().float()
        gnorm = ext.multi_tensor_l2norm(65536, noop, [rg], False)[0]
        rstep += (noop != 1).int()
        ext.multi_tensor_lamb(65536, noop, [rg, rp, rm, rv], lr_t, 0.9, 0.999, 1e-6, rstep, 1, CASE["wd"], 1, 1, gnorm, 1.0 * sc, False,
                              found_inf, inv_scale)
        gnorms.append(gnorm.item())
    rec = dict(seed=np.int64(CASE["seed"]), lr=np.float64(CASE["lr"]), wd=np.float64(CASE["wd"]), scale=np.float64(CASE["scale"]),
               steps=np.int64(CASE["steps"]), gnorm=np.array(gnorms, np.float32))
    gen = torch.Generator().manual_seed(0)
    for i, s in enumerate(CASE["shapes"]):
        n = int(np.prod(s))
        idx = torch.randperm(n, generator=gen)[:SAMPLE].sort().values if n > SAMPLE else torch.arange(n)
        rec[f"shape{i}"] = np.array(s, np.int64)
        rec[f"idx{i}"] = idx.numpy().astype(np.int32)
        for name, t in (("exp_avg", rm[i]), ("exp_avg_sq", rv[i]), ("param", rp[i])):
            rec[f"{name}{i}"] = t.reshape(-1)[idx.cuda()].cpu().numpy()
    np.savez(out, **rec)
    print("wrote", out, "global grad norms", gnorms)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "lamb_reference_kernel.npz"))
