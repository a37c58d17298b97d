#!/usr/bin/env python
"""bench.py -- BERT-large pretraining step throughput (training_sequences_per_second, the reference's own metric:
run_pretraining.py:748) on N B200s of one node, synthetic data, bf16, LAMB.

  python bench.py --gpus 1 --steps 8 --warmup 3                      # our arm (default)
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
  python bench.py --impl reference ...                               # CPU arm: the oracle restatement on the host cores

One "step" = H2D of one synthetic batch (e2e pass only) + forward + loss + backward (+ DDP bucketed NCCL allreduce)
+ FusedLAMBAMP step + zero_grad, i.e. take_training_step + take_optimizer_step of the reference driver with
gradient_accumulation_steps = 1.  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "training_sequences_per_second"
_T0 = time.time()


def log(msg):
    print(f"[bench +{time.time() - _T0:7.1f}s] {msg}", file=sys.stderr, flush=True)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="pretrain", choices=["pretrain", "squad"], help="pretrain = BERT-large pretraining step (headline); squad = SQuAD fine-tuning "
                         "step, seq 384, QA head, FusedAdam + clip (BASELINE.json configs[3])")
    ap.add_argument("--seq", type=int, default=0, help="0 = 512 (phase 2, headline) for pretrain / 384 for squad; 128 = phase 1")
    ap.add_argument("--batch", type=int, default=0, help="per-GPU micro-batch (0 = 128 @512, 512 @128 -- 65536 tokens per GPU per step; the reference ran 32 @512 / 256 @128 on 80 GB "
                         "A100s, SURVEY.md 8d; 180 GB fits 4x that and the LAMB / allreduce cost per sequence halves again vs 64)")
    ap.add_argument("--max-pred", type=int, default=0)
    ap.add_argument("--no-dropout", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-batch", type=int, default=0, help="sequences per CPU step (bounded sample)")
    ap.add_argument("--bucket-mb", type=int, default=100)
    ap.add_argument("--dynamic-mlm-gather", action="store_true", help="use torch.nonzero (host sync per step) like the reference instead of nonzero_static(batch*max_pred)")
    ap.add_argument("--no-reference-gpu", action="store_true", help="skip the reference-GPU leg (the unmodified reference step timed on this GPU after our arm, N=1 only)")
    ap.add_argument("--no-cuda-graphs", action="store_true", help="enqueue every step eagerly instead of replaying one captured CUDA graph of the whole step "
                         "(the reference driver's --cuda_graphs, run_pretraining.py:602-640,669)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="after the timed resident pass, write what its last step computed as DIR/<name>.npy "
                         "(float32, see dump_outputs); inputs and weights are seeded, so two builds run with the same arguments can be compared array by array")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return a


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d.get("hbm_gbs"), tf_burst=d.get("bf16_tflops"), tf_sustained=d.get("bf16_tflops_sustained"), source="measured")
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi sampled every 200 ms DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()          # exact PID we started
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        rows = [r for t, r in self.rows if t0 <= t <= t1 and len(r) >= 8] or [r for _, r in self.rows if len(r) >= 8]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(float(r[1]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[4 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][2]), "power_w_max": max(float(r[3]) for r in rows),
                "samples": len(rows), "reasons": reasons}


def dump_outputs(out_dir, model, opt, loss, per_tensor=4096):
    """Write what one training step hands its caller, as float32 .npy files in out_dir:
      loss.npy               the step's loss, shape [1]
      global_grad_norm.npy   the optimizer's global gradient norm of that step, shape [1]
      params.npy, master_params.npy, exp_avg.npy, exp_avg_sq.npy
                             every parameter the step updated (named_parameters() order) after the update: the 16-bit model weights,
                             their fp32 masters and the two moments, each sampled at the same at most `per_tensor` positions and concatenated.
    The positions come from a fixed seed and the tensor sizes only, so they are the same in every run; for BERT-large
    (398 tensors) each array holds about 0.94M values, about 14 MB in all.  Compare two builds with a tolerance: split-K GEMMs
    accumulate with fp32 atomics in no fixed order, so two runs of one build already differ slightly (on a B200 at its 1000 W
    limit, the loss of the default workload by 4e-5 relative)."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    net = model.module if hasattr(model, "module") else model
    masters = {id(p): m for g, g32 in zip(opt.param_groups, opt.param_groups_fp32) for p, m in zip(g["params"], g32["params"])}
    gen = torch.Generator().manual_seed(0)
    cols = {"params": [], "master_params": [], "exp_avg": [], "exp_avg_sq": []}
    for _, p in net.named_parameters():
        st = opt.state.get(p, {})
        if "exp_avg" not in st:                     # no gradient, so the step did not touch it
            continue
        n = p.numel()
        idx = (torch.randperm(n, generator=gen)[:per_tensor].sort().values if n > per_tensor else torch.arange(n)).to(p.device)
        master = masters.get(id(p))
        for name, t in (("params", p), ("master_params", p if master is None else master),
                        ("exp_avg", st["exp_avg"]), ("exp_avg_sq", st["exp_avg_sq"])):
            cols[name].append(t.detach().reshape(-1)[idx].float().cpu())
    arrays = {k: torch.cat(v).numpy() for k, v in cols.items()}
    arrays["loss"] = loss.detach().float().reshape(1).cpu().numpy()
    arrays["global_grad_norm"] = opt._global_grad_norm.detach().float().reshape(1).cpu().numpy()
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))
    log(f"wrote {len(arrays)} arrays ({sum(a.nbytes for a in arrays.values()) / 2**20:.1f} MB) to {out_dir}")


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle (reference algorithm restated for CPU, oracle/) on a bounded sample
# ------------------------------------------------------------------------------------------------
def usable_cores():
    """Host cores this process may actually use: affinity mask capped by the cgroup CPU quota (a container that
    *sees* 128 CPUs but is throttled to a fraction of them collapses under 128 spinning OpenMP threads)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    return n


def cpu_reference_run(cfg, S, P, ref_batch, steps, warmup):
    threads = int(os.environ.get("DLE_CPU_THREADS", 0)) or min(usable_cores(), 64)
    os.environ["OMP_NUM_THREADS"] = str(threads)          # read by libgomp when oracle/liblamb_oracle.so first runs
    import numpy as np
    import torch
    from oracle import bert_oracle as O
    from oracle import lamb_oracle as LO
    torch.set_num_threads(threads)
    sd = {k: v.requires_grad_(True) for k, v in O.init_params(cfg, seed=42).items()}
    no_decay = ['bias', 'gamma', 'beta', 'LayerNorm']
    names = list(sd.keys())
    groups = []
    for decay, wd in ((True, 0.01), (False, 0.0)):
        ks = [k for k in names if (not any(nd in k for nd in no_decay)) == decay]
        groups.append(dict(keys=ks, params=[sd[k].detach().numpy() for k in ks], grads=None,
                           exp_avg=[np.zeros(tuple(sd[k].shape), np.float32) for k in ks],
                           exp_avg_sq=[np.zeros(tuple(sd[k].shape), np.float32) for k in ks],
                           lr=6e-3, betas=(0.9, 0.999), eps=1e-6, weight_decay=wd, step=0, bias_correction=True, grad_averaging=True))
    batches = [O.synthetic_batch(ref_batch, S, cfg["vocab_size"], P, seed=42 + i) for i in range(2)]

    def step(i):
        t_a = time.perf_counter()
        loss, *_ = O.forward_loss(sd, cfg, batches[i % 2])
        loss.backward()
        log(f"  cpu fwd+bwd {time.perf_counter() - t_a:.1f}s")
        for g in groups:
            g["grads"] = [sd[k].grad.numpy() for k in g["keys"]]
        LO.lamb_step(groups)                       # updates the numpy views of the torch parameters in place
        for k in names:
            sd[k].grad = None
        return loss.item()

    log(f"cpu arm: params built, {torch.get_num_threads()} threads")
    for i in range(warmup):
        step(i)
        log(f"cpu warm-up {i} done")
    t0 = time.perf_counter()
    for i in range(steps):
        step(i)
        log(f"cpu step {i} done")
    dt = time.perf_counter() - t0
    return dict(value=ref_batch * steps / dt, ms_per_step=1000.0 * dt / steps, cores=threads, threads=torch.get_num_threads(),
                sample=f"{threads} threads of {os.cpu_count()} visible CPUs; {steps} steps x {ref_batch} sequences (S={S}) of the same workload after {warmup} warm-up; fp32 torch-CPU "
                       f"forward/backward (oracle/bert_oracle.py) + OpenMP LAMB (oracle/lamb_oracle.c)")


def reference_gpu_leg(S, steps, warmup):
    """The unmodified reference step (its modeling.py, its fused_lamb_CUDA kernels, its run_pretraining.py functions) timed on this GPU
    by tools/bench_reference_gpu.py in a fresh process, at the reference's own micro-batch (32 @512 / 256 @128, README.md:813-816) and at
    twice that; eager and with the reference's own --cuda_graphs.  Returns the list of result lines (or a one-line reason)."""
    tool = os.path.join(ROOT, "tools", "bench_reference_gpu.py")
    if not os.path.exists(os.path.join(ROOT, "baseline", "_ref", "BERT", "run_pretraining.py")):
        return {"unavailable": "baseline/_ref/BERT is not installed (python baseline/install_ref.py needs /root/reference)"}
    base = 32 if S >= 384 else 256
    runs, out = [(base, False), (base, True), (2 * base, True)], []
    for batch, graphs in runs:
        cmd = [sys.executable, tool, "--arm", "reference", "--seq", str(S), "--batch", str(batch), "--steps", str(steps), "--warmup", str(warmup)]
        if graphs:
            cmd.append("--cuda-graphs")
        env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT")}
        try:
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=420, env=env)
            lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
            if r.returncode == 0 and lines:
                j = json.loads(lines[-1])
                out.append({"micro_batch": batch, "cuda_graphs": graphs, "value": j["value"], "e2e": j["e2e"]["value"], "ms_per_step": j["ms_per_step"],
                            "dtype": j["dtype"], "hbm_peak_gb": j.get("hbm_peak_gb")})
            else:
                out.append({"micro_batch": batch, "cuda_graphs": graphs, "failed": (r.stderr or r.stdout).strip().splitlines()[-1:][0][:300] if (r.stderr or r.stdout).strip() else "no output"})
        except subprocess.TimeoutExpired:
            out.append({"micro_batch": batch, "cuda_graphs": graphs, "failed": "timeout"})
        log(f"reference gpu leg: {out[-1]}")
    return {"runs": out}


def workload(args):
    from deeplearningexamples_b200 import training as T
    if args.workload == "squad":
        cfg = dict(T.BERT_LARGE)
        cfg["vocab_size"] = 30528
        return cfg, args.seq or 384, args.batch or 32, 0          # reference micro-batch 32 at seq 384 (README.md:841-842)
    S = args.seq or 512
    B = args.batch or (128 if S >= 384 else 512)
    P = args.max_pred or (80 if S >= 384 else 20)
    cfg = dict(T.BERT_LARGE)
    cfg["vocab_size"] = 30528                     # 30522 padded to a multiple of 8 (run_pretraining.py:383-384)
    return cfg, S, B, P


def config_dict(args, cfg, S, B, P, n):
    if args.workload == "squad":
        return {"workload": f"BERT-large SQuAD fine-tuning step seq{S} bf16 FusedAdam + global-norm clip (BASELINE.json configs[3] per-GPU shape)",
                "seq_len": S, "micro_batch_per_gpu": B, "global_batch": B * n, "gradient_accumulation_steps": 1,
                "dropout": 0.0 if args.no_dropout else 0.1, "parallelism": f"dp{n}", "attention_mask": "all ones (padded to full length)",
                "cuda_graphs": not args.no_cuda_graphs,
                "l2_policy": "per-step working set (weights 0.67 GB + activations) exceeds the 126 MB L2; no explicit flush"}
    phase = "phase-2" if S >= 384 else "phase-1"
    return {"workload": f"BERT-large {phase} pretraining step seq{S} bf16 LAMB (BASELINE.json configs[{2 if S >= 384 else 1}] per-GPU shape)",
            "seq_len": S, "micro_batch_per_gpu": B, "global_batch": B * n, "max_predictions_per_seq": P,
            "gradient_accumulation_steps": 1, "dropout": 0.0 if args.no_dropout else 0.1, "parallelism": f"dp{n}",
            "attention_mask": "all ones (padded to full length)", "mlm_gather": "torch.nonzero (sync)" if args.dynamic_mlm_gather else "nonzero_static(batch*max_pred), sync-free",
            "cuda_graphs": not (args.no_cuda_graphs or args.dynamic_mlm_gather),
            "l2_policy": "per-step working set (weights 0.67 GB + activations >10 GB) exceeds the 126 MB L2; no explicit flush"}


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    cfg, S, B, P = workload(args)
    ref_batch = args.ref_batch or 2
    steps, warm = args.steps, args.warmup
    r = cpu_reference_run(cfg, S, P, ref_batch, steps, warm)
    n = args.gpus
    line = {"impl": "reference", "metric": METRIC, "value": round(r["value"], 4), "unit": "sequences/s", "n_gpus": n, "steps": steps,
            "warmup": warm, "ms_per_step": round(r["ms_per_step"], 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": config_dict(args, cfg, S, B, P, n),
            "cpu_baseline": {"value": round(r["value"], 4), "unit": "sequences/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]},
            "e2e": {"value": round(r["value"], 4), "unit": "sequences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "reference run_pretraining.py asserts CUDA (run_pretraining.py:325) and cannot run on CPU; this arm times the CPU "
                    "restatement of the same step (oracle/) on the box's host cores"}
    print(json.dumps(line), flush=True)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from deeplearningexamples_b200 import _lib as L
    from deeplearningexamples_b200 import kernels as K
    from deeplearningexamples_b200 import ops
    from deeplearningexamples_b200 import training as T

    world = int(os.environ.get("WORLD_SIZE", 1))
    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=ours) needs a B200: there is no CPU path")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        if not (args.no_cuda_graphs or args.dynamic_mlm_gather):
            # whole-step capture under DDP: NCCL's async error handling must be off, as the reference sets it (run_pretraining.py:334-335)
            os.environ.setdefault("NCCL_ASYNC_ERROR_HANDLING", "0")
            os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "0")
        # record what NCCL sets up (algorithms, channels, NVLS) without touching stdout: rank 0 writes its INIT log to a file
        nccl_log = None
        if rank == 0 and os.environ.get("NCCL_DEBUG", "VERSION").upper() in ("VERSION", "WARN"):
            nccl_log = f"/tmp/dle_nccl_init_{os.getpid()}.log"
            os.environ.update(NCCL_DEBUG="INFO", NCCL_DEBUG_SUBSYS="INIT,ENV,TUNING", NCCL_DEBUG_FILE=nccl_log)
        dist.init_process_group(backend="nccl", init_method="env://", device_id=device)
    else:
        nccl_log = None
    L.load()
    cfg, S, B, P = workload(args)
    if args.no_dropout:
        cfg["hidden_dropout_prob"] = cfg["attention_probs_dropout_prob"] = 0.0
    ops.manual_seed(42 + rank)
    squad = args.workload == "squad"
    if squad:
        from deeplearningexamples_b200 import squad as SQ
        model, opt, sched = SQ.prepare_squad_model_and_optimizer(cfg, device, distributed=world > 1, seed=42, total_steps=10000)
        scaler = crit = None
        host = [SQ.synthetic_squad_batch(B, S, cfg["vocab_size"], seed=T.rank_seed(42, rank) + 100 * i, pin=True) for i in range(4)]
    else:
        model, opt, scaler, sched, crit, _ = T.prepare_model_and_optimizer(cfg, device, distributed=world > 1, bucket_cap_mb=args.bucket_mb,
                                                                          seed=42, static_masked_count=None if args.dynamic_mlm_gather else B * P)
        host = [T.synthetic_batch(B, S, cfg["vocab_size"], P, seed=T.rank_seed(42, rank) + 100 * i, pin=True) for i in range(4)]
    model.train()
    dev = [{k: v.to(device) for k, v in hb.items()} for hb in host[:2]]
    stage = {k: torch.empty_like(v, device=device) for k, v in host[0].items()}
    loss_host = torch.zeros(1, dtype=torch.float32).pin_memory()
    loss_acc = torch.zeros(1, dtype=torch.float32, device=device)
    h2d = sum(v.numel() * v.element_size() for v in host[0].values())

    use_graphs = not (args.no_cuda_graphs or args.dynamic_mlm_gather)
    graph = {"g": None, "loss": None}

    def one_step():                                    # take_training_step + take_optimizer_step on the static batch
        if squad:
            graph["loss"] = SQ.squad_training_step(model, opt, sched, stage, loss_acc)
            return
        graph["loss"] = T.take_training_step(scaler, model, crit, stage, loss_acc)
        T.take_optimizer_step(sched, opt, scaler)

    def run_step():
        if graph["g"] is not None:
            graph["g"].replay()
        else:
            one_step()
        return graph["loss"]

    def step_resident(i):                              # inputs already in HBM: device-to-device into the static batch
        db = dev[i % 2]
        for k in stage:
            stage[k].copy_(db[k], non_blocking=True)
        return run_step()

    def step_e2e(i):                                   # inputs in pinned host memory, loss read back
        hb = host[i % 4]
        for k in stage:
            stage[k].copy_(hb[k], non_blocking=True)
        loss = run_step()
        loss_host.copy_(loss.detach().float().reshape(1), non_blocking=True)
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t_host = time.perf_counter()
        for i in range(steps):
            fn(i)
        e1.record()
        t_host = time.perf_counter() - t_host          # host time to ENQUEUE the steps (no sync inside)
        barrier()
        log(f"  host enqueue {1000 * t_host / steps:.2f} ms/step vs device {e0.elapsed_time(e1) / steps:.2f} ms/step")
        return T.max_over_ranks(e0.elapsed_time(e1), device), 1000 * t_host / steps

    log(f"model built: B={B} S={S} world={world}")
    n_warm = max(args.warmup, 3)
    launches_per_step = None
    if use_graphs:
        # the reference's recipe (run_pretraining.py:611-626): eager warm-up on a side stream (11 iterations under DDP), then capture
        for k in stage:
            stage[k].copy_(dev[0][k])
        n_eager = max(n_warm, 11 if world > 1 else 3)
        n_before = L.launch_count["n"]
        try:
            graph["g"] = T.capture_step_graph(one_step, warmup_iters=n_eager)
            launches_per_step = (L.launch_count["n"] - n_before) // (n_eager + 1)
            torch.cuda.synchronize()
            log(f"captured the step into a CUDA graph after {n_eager} eager warm-up steps ({launches_per_step} kernels of libdle_b200.so per step)")
        except Exception as e:                      # report, then measure the eager path rather than nothing
            graph["g"], launches_per_step, use_graphs = None, None, False
            log(f"CUDA-graph capture failed ({type(e).__name__}: {str(e)[:200]}); continuing with eager launches")
            torch.cuda.synchronize()
        n_warm = n_eager
        for i in range(2):
            step_resident(i)
    else:
        for i in range(n_warm):
            step_resident(i)
            torch.cuda.synchronize()
            log(f"warm-up step {i} done")
    step_e2e(0)
    torch.cuda.synchronize()
    log("warm-up done")
    sampler = ClockSampler(local) if rank == 0 else None
    t_start = time.time()
    if sampler:
        sampler.start()
        time.sleep(0.3)
    n0 = L.launch_count["n"]
    torch.cuda.nvtx.range_push("timed_resident")
    torch.cuda.profiler.start()          # ncu --profile-from-start off: capture exactly the timed region (all threads)
    ms_res, host_res = timed(step_resident, args.steps)
    torch.cuda.profiler.stop()
    torch.cuda.nvtx.range_pop()
    log(f"resident pass: {ms_res / args.steps:.2f} ms/step")
    if args.dump_outputs and rank == 0:            # before the passes below train the model further
        dump_outputs(args.dump_outputs, model, opt, graph["loss"])
    launches = (L.launch_count["n"] - n0) if launches_per_step is None else launches_per_step * args.steps
    ms_e2e, host_e2e = timed(step_e2e, args.steps)
    log(f"e2e pass: {ms_e2e / args.steps:.2f} ms/step")
    final_loss = loss_host.item()
    # per-launch GEMM timing for the roofline: CUDA events cannot bracket launches inside a replayed graph, so the same step is
    # enqueued eagerly once more (same kernels, same shapes, same stream) with an event pair around every GEMM launch
    graph["g"] = None
    K.gemm_profile = []
    ms_prof, _ = timed(step_e2e, max(2, min(args.steps, 4)))
    prof_steps = max(2, min(args.steps, 4))
    prof, K.gemm_profile = K.gemm_profile, None
    t_end = time.time()
    clocks = sampler.stop(t_start, t_end) if sampler else None
    ops.check_device_errors()
    if not squad:
        (model.module if hasattr(model, "module") else model).cls.check_mlm_overflow()

    n = world
    value = T.global_throughput(B, n, args.steps, ms_res)
    e2e = T.global_throughput(B, n, args.steps, ms_e2e)
    pk = peaks()
    traffic, traffic_src = None, None
    tensor_active = None
    tpath = os.path.join(ROOT, "profiles", "r02_gemm_traffic.json")
    if os.path.exists(tpath):                     # dram__bytes_read.sum + dram__bytes_write.sum per launch, from the committed ncu capture
        tj = json.load(open(tpath))
        traffic, traffic_src = tj["avg_dram_traffic_bytes_per_launch"], (
            "profiles/r02_gemm_traffic.json (ncu --set full, 12 forward GEMM launches of this command; the same 12 launches move "
            f"{tj.get('avg_algorithmic_bytes_per_launch', 0)} algorithmic bytes on average -- algorithmic_bytes_per_launch_avg below averages ALL timed launches)")
        ls_ = tj.get("launches", [])
        if ls_:                                   # time-weighted sm__pipe_tensor_cycles_active of the same 12 launches (ncu, not live)
            tensor_active = round(sum(l["tensor_active_pct"] * l["time_us"] for l in ls_) / sum(l["time_us"] for l in ls_), 1)
    by_shape = {}
    for a_, b_, f_, tag in prof:
        d = by_shape.setdefault(tag, [0, 0.0, 0.0])
        d[0] += 1; d[1] += a_.elapsed_time(b_); d[2] += f_
    epi_names = ["bias", "bias_gelu", "bias_dropout_residual", "dgelu", "add", "atomic_f32", "f32", "bias_tanh"]
    gemm_table = sorted(({"M": t[0], "N": t[1], "K": t[2], "a_mn": t[3], "b_mn": t[4], "epilogue": epi_names[t[5]], "launches": d[0],
                          "ms_total": round(d[1], 3), "tflops": round(d[2] / d[1] / 1e9, 1)} for t, d in by_shape.items()), key=lambda r: -r["ms_total"])
    for row in gemm_table[:24]:
        log(f"  gemm {row}")
    gemm_ms = sum(a.elapsed_time(b) for a, b, _, _ in prof)
    gemm_flops = sum(f for _, _, f, _ in prof)
    ach = gemm_flops / (gemm_ms / 1000.0) / 1e12 if gemm_ms > 0 else 0.0
    flops_seq = SQ.squad_flops_per_seq(cfg, S) if squad else T.train_flops_per_seq(cfg, S, P)
    line = {"metric": METRIC, "value": round(value, 2), "unit": "sequences/s", "n_gpus": n, "steps": args.steps, "warmup": n_warm,
            "ms_per_step": round(ms_res / args.steps, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic", "config": config_dict(args, cfg, S, B, P, n),
            "e2e": {"value": round(e2e, 2), "unit": "sequences/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": round(ms_e2e / args.steps, 3)},
            "host_enqueue_ms_per_step": {"resident": round(host_res, 3), "e2e": round(host_e2e, 3)},
            "gpu_launches": launches, "hbm_peak_gb": round(torch.cuda.max_memory_allocated() / 2**30, 1),
            "roofline": {"kernel": "gemm_bf16_tcgen05_kernel (all dense projections/FFN, fwd+dgrad+wgrad)", "bound": "tensor",
                         "achieved": round(ach, 1), "peak": pk["tf_sustained"], "unit": "TFLOP/s", "frac": round(ach / pk["tf_sustained"], 4),
                         "peak_source": pk["source"] + " (bf16_tflops_sustained: kernel timed inside a long step)",
                         "traffic": traffic, "traffic_source": traffic_src, "tensor_pipe_active_pct_ncu": tensor_active,
                         "algorithmic_bytes_per_launch_avg": int(sum(2.0 * (m * k + n * k + m * n) for _, _, _, (m, n, k, *_r) in prof) / max(len(prof), 1)),
                         "launches_timed": len(prof), "share_of_step": round((gemm_ms / prof_steps) / (ms_e2e / args.steps), 4),
                         "by_shape_top": gemm_table[:12],
                         "how": "CUDA events around every GEMM launch on the launching stream during an eager pass of the same step "
                                f"({prof_steps} steps, {round(ms_prof / prof_steps, 2)} ms/step incl. the host cost of recording two events per launch) run right after the "
                                "timed passes (events cannot bracket launches inside a replayed graph); algorithmic flops = 2*M*N*K per launch; "
                                "share_of_step = GEMM ms per step of that pass / ms per step of the timed e2e pass"},
            "model_flops_utilisation": {"train_gflop_per_seq": round(flops_seq / 1e9, 1),
                                        "achieved_tflops_per_gpu": round(value / n * flops_seq / 1e12, 1),
                                        "frac_of_sustained_peak": round(value / n * flops_seq / 1e12 / pk["tf_sustained"], 4)},
            "final_loss": round(final_loss, 4)}
    line["config"]["cuda_graphs"] = bool(use_graphs)
    if clocks is not None:
        line["clocks"] = clocks
    if nccl_log and os.path.exists(nccl_log):
        keep = [l.strip() for l in open(nccl_log, errors="replace") if any(k in l for k in ("NVLS", "Channel", "channels", "Connected", "NCCL version", "nRanks", "nranks", "Algo", "threadThresholds", "P2P", "NCCL_"))]
        brief = [l.split("NCCL INFO", 1)[-1].strip()[:160] for l in keep]
        summary = {"nvls": any("NVLS" in l for l in brief), "lines": len(brief), "tail": brief[-12:],
                   "channels": next((l for l in reversed(brief) if "channels" in l.lower() or "coll channels" in l.lower()), None)}
        line["nccl"] = summary
        for l in brief[-25:]:
            log("  nccl: " + l)
    if rank == 0 and n == 1 and not args.no_cpu_baseline and not squad:
        del model, opt
        torch.cuda.empty_cache()
        log("cpu baseline ...")
        r = cpu_reference_run(cfg, S, P, args.ref_batch or 2, 2, 1)
        log("cpu baseline done")
        line["cpu_baseline"] = {"value": round(r["value"], 4), "unit": "sequences/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]}
    if rank == 0 and n == 1 and not args.no_reference_gpu and not squad:
        try:
            del model, opt
        except NameError:
            pass
        graph.clear()
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        log(f"reference gpu leg ... ({torch.cuda.memory_allocated() / 2**30:.1f} GB still allocated by this process)")
        rg = reference_gpu_leg(S, max(3, min(args.steps, 6)), 3)
        ok = [x for x in rg.get("runs", []) if "value" in x]
        if ok:
            best = max(ok, key=lambda x: x["e2e"])
            rg.update({"value": best["value"], "e2e": best["e2e"], "micro_batch": best["micro_batch"], "unit": "sequences/s",
                       "what": "UNMODIFIED reference step (reference modeling.py + fused_lamb_CUDA kernels + run_pretraining.py take_training_step / "
                               "take_optimizer_step, --fp16 --allreduce_post_accumulation --allreduce_post_accumulation_fp16, eager torch ops, no TorchScript) "
                               "timed on THIS GPU with the same CUDA-event harness; best of the runs listed"})
            line["vs_reference_gpu"] = {"e2e_ratio": round(e2e / best["e2e"], 3), "value_ratio": round(value / best["value"], 3),
                                        "ours_micro_batch": B, "reference_micro_batch": best["micro_batch"]}
        line["reference_gpu"] = rg
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
