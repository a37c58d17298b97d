"""The drop-in claim, executed: the reference's OWN run_pretraining.py (byte-for-byte the file installed from /root/reference by
baseline/install_ref.py -- checked against the manifest hash) trains over the B200 mirror (shims/ours) with its own flags, writes its
own checkpoints and resumes from them (run_pretraining.py:388-410,489-515), eagerly and with its own --cuda_graphs.  The same script
also runs over the reference's own modeling.py + fused_lamb_CUDA kernels (the GPU baseline arm) so that arm is known to work here.

Launched as the reference's scripts launch it: a (1-rank) distributed job, --fp16 --allreduce_post_accumulation
--allreduce_post_accumulation_fp16 (model.half() -> bf16 on this path, see modeling.BertPreTrainedModel.half), and the driver's own
--disable_jit_fusions (custom autograd Functions cannot be TorchScript-ed)."""
import hashlib
import json
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "baseline", "_ref", "BERT")
SMALL = dict(attention_probs_dropout_prob=0.1, hidden_act="gelu", hidden_dropout_prob=0.1, hidden_size=256, initializer_range=0.02,
             intermediate_size=1024, max_position_embeddings=128, num_attention_heads=4, num_hidden_layers=2, type_vocab_size=2,
             vocab_size=30522)


def _need_ref():
    if not os.path.exists(os.path.join(REF, "run_pretraining.py")):
        pytest.skip("baseline/_ref/BERT not installed (python baseline/install_ref.py where the reference tree exists)")


def _run(arm, out, extra, steps, tmp_path, timeout=600):
    """`steps` optimizer steps of a 100-step schedule (--steps_this_run): the reference's --cuda_graphs warm-up trains 11 extra steps
    before the first counted one (run_pretraining.py:611-616), which a schedule as short as the run itself would push past its end
    (poly decay of a negative base = NaN learning rate, in the reference as well)."""
    cfg = tmp_path / "small.json"
    cfg.write_text(json.dumps(SMALL))
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    env = dict(os.environ, RANK="0", WORLD_SIZE="1", LOCAL_RANK="0", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    cmd = [sys.executable, os.path.join(ROOT, "tools", "run_reference_driver.py"), "--arm", arm, "--",
           "--input_dir", "synthetic?seq_len=128&max_pred=20&samples=512&bin_size=0", "--config_file", str(cfg), "--output_dir", str(out), "--vocab_file", "vocab.txt",
           "--train_batch_size", "8", "--max_seq_length", "128", "--max_predictions_per_seq", "20", "--max_steps", "100", "--steps_this_run", str(steps),
           "--warmup_proportion", "0.1", "--learning_rate", "1e-3", "--seed", "42", "--do_train", "--fp16", "--allreduce_post_accumulation",
           "--allreduce_post_accumulation_fp16", "--disable_jit_fusions", "--num_steps_per_checkpoint", "5", "--log_freq", "1",
           "--json-summary", str(out / "dllogger.json"), "--disable_progress_bar"] + extra
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env, cwd=str(tmp_path))
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    recs = [json.loads(l[5:]) for l in open(out / "dllogger.json") if l.startswith("DLLL ")]
    return r, recs


def _final(recs, key):
    vals = [rec["data"][key] for rec in recs if rec.get("type") == "LOG" and key in rec.get("data", {})]
    assert vals, key
    return vals[-1]


def test_installed_reference_script_is_the_reference_file():
    _need_ref()
    manifest = json.load(open(os.path.join(REF, "MANIFEST.json")))
    for rel in ("run_pretraining.py", "modeling.py", "lamb_amp_opt/fused_lamb/fused_lamb.py"):
        assert hashlib.sha256(open(os.path.join(REF, rel), "rb").read()).hexdigest() == manifest[rel]


@pytest.mark.parametrize("graphs", [False, True])
def test_unmodified_reference_driver_trains_checkpoints_and_resumes_over_the_b200_mirror(tmp_path, graphs):
    _need_ref()
    out = tmp_path / "results"
    # the reference's own --cuda_graphs cannot capture its dense-sequence-output path (torch.nonzero at modeling.py:590 and the boolean
    # label indexing of ITS criterion, run_pretraining.py:89, synchronise): like the reference model itself, the mirror is driven with
    # the script's --no_dense_sequence_output when graphs are on
    extra = ["--cuda_graphs", "--no_dense_sequence_output"] if graphs else []
    r, recs = _run("ours", out, extra, 10, tmp_path)
    assert os.path.exists(out / "ckpt_10.pt") and os.path.exists(out / "ckpt_5.pt")
    assert _final(recs, "training_sequences_per_second") > 0
    loss10 = _final(recs, "final_loss")
    assert 0 < loss10 < 12.0 and loss10 == loss10
    ck = torch.load(out / "ckpt_10.pt", map_location="cpu", weights_only=False)
    assert set(ck) >= {"model", "optimizer", "grad_scaler", "epoch"}
    assert "bert.encoder.layer.0.attention.self.query.weight" in ck["model"] and ck["model"]["bert.encoder.layer.0.attention.self.query.weight"].dtype == torch.bfloat16
    assert int(ck["optimizer"]["param_groups"][0]["step"].item()) == 10 + (11 if graphs else 0)     # the reference's 11 graph warm-up iterations also step the optimizer (:611-616)
    some = next(iter(ck["optimizer"]["state"].values()))
    assert some["exp_avg"].dtype == torch.float32
    # resume: picks the newest ckpt_*.pt of output_dir, continues to max_steps, keeps at most three checkpoints
    r2, recs2 = _run("ours", out, extra + ["--resume_from_checkpoint"], 15, tmp_path)
    assert "resume step from  10" in r2.stdout
    assert os.path.exists(out / "ckpt_15.pt")
    ck2 = torch.load(out / "ckpt_15.pt", map_location="cpu", weights_only=False)
    assert int(ck2["optimizer"]["param_groups"][0]["step"].item()) >= 15
    assert len([f for f in os.listdir(out) if f.startswith("ckpt_")]) <= 3


def test_reference_arm_runs_on_this_box(tmp_path):
    """The GPU baseline arm: the same script over the reference's own modeling.py and fused_lamb_CUDA kernels (fp16)."""
    _need_ref()
    from oracle import build_ref
    if build_ref.built_path() is None:
        pytest.skip("oracle/_ref/fused_lamb_CUDA.so not present")
    out = tmp_path / "results_ref"
    r, recs = _run("reference", out, [], 10, tmp_path)
    assert os.path.exists(out / "ckpt_10.pt")
    loss = _final(recs, "final_loss")
    assert 0 < loss < 12.0
    ck = torch.load(out / "ckpt_10.pt", map_location="cpu", weights_only=False)
    assert ck["model"]["bert.encoder.layer.0.attention.self.query.weight"].dtype == torch.float16
