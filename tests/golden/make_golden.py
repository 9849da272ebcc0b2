"""Generates tests/golden/reference_vectors.npz by RUNNING THE REFERENCE'S OWN PYTHON.

The reference is pure Python over mlx.core (mlx==0.25.0), which this project does not depend on.  This script
puts oracle/mlx_numpy_shim (a float32 NumPy stand-in for the handful of mlx primitives involved) on
sys.path, imports the reference's modules unmodified, feeds them seeded inputs and records inputs +
outputs.  tests/test_oracle_golden.py then checks oracle/reference_math.py against these vectors, and
the -m gpu tests check the CUDA path against them too.  Run with a checkout of the reference:

    python tests/golden/make_golden.py <reference checkout>

The FlashAttention projection weights are not stored, which keeps the file under 1 MB: tests regenerate them
from the seed set before each FlashAttention is built (tests/test_oracle_golden.py, attn_proj_weights).

What is exercised (reference file:line):
  optimizers/muon.py:54-83     Muon.zeropower_via_newtonschulz5        (wide, tall, square, batched)
  optimizers/muon.py:85-141    Muon.update on a flat-named module, 2 steps, callable lr
  optimizers/shampoo.py:88-126 MatrixSqrt.matrix_inverse_pth_root
  optimizers/shampoo.py:229-312 Shampoo._update_statistics/_compute_preconditioners/
                               _apply_preconditioners/_apply_grafting
  arch/flash_attention.py:78-194 FlashAttention._flash_attention and __call__ (MHA/GQA/MQA, causal)
  arch/llama.py:44-56,142-151,322-412 RMSNorm, MLP, Model.__call__ (tiny config, tied embeddings)
  mlx_lm_utils.py:5-56         linear_schedule / cosine_decay / join_schedules
  core/training.py:324-543     TokenizerManager (byte level) and DataManager (chunking, length sort, shuffles,
                               padded batches, validation walk) on tests/golden/tiny_corpus.jsonl, seeded as
                               Trainer.setup_system does (:966-968)
  core/training.py:1195-1234   Trainer.compute_loss (masked token-mean cross-entropy) on the tiny Model
  core/training.py:764-856     OptimizationManager.create_scheduler (all three types) and the Shampoo branch of
                               create_optimizer (factory defaults -> ShampooParams)
  core/training.py:621-668     EarlyStoppingMonitor: stop decisions / counter / best over validation-loss sequences
  core/training.py:52-166      Config.from_yaml on this repo's configs/c*.yaml -> tests/golden/ref_config_parse.json
  distributed/hybrid_distributed.py:303-354,430-452  HybridDeviceManager._aggregate_gradients /
                               distribute_batch (the data-parallel contract: unweighted mean, remainder
                               rows to the last shard)
"""
import os
import sys
import tempfile
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
REPO = HERE.parents[1]
if len(sys.argv) != 2:
    raise SystemExit("usage: python tests/golden/make_golden.py <reference checkout>")
REF = Path(sys.argv[1]).resolve()

# the reference's package names (optimizers, arch, core) collide with this repo's drop-in shims:
# make sure only the reference and the mlx shim are importable
sys.path = [p for p in sys.path if p not in ("", str(REPO)) and Path(p or ".").resolve() != REPO]
sys.path.insert(0, str(REF))
sys.path.insert(0, str(REPO / "oracle" / "mlx_numpy_shim"))
os.chdir(tempfile.gettempdir())

import mlx.core as mx  # noqa: E402  (the shim)
import mlx.nn as nn  # noqa: E402
import mlx_lm_utils as ref_sched  # noqa: E402
from arch.flash_attention import FlashAttention  # noqa: E402
from arch.llama import MLP, Model, ModelArgs, RMSNorm  # noqa: E402
from optimizers.muon import Muon  # noqa: E402
from optimizers.shampoo import MatrixSqrt, Shampoo, ShampooParams  # noqa: E402

rng = np.random.default_rng(1234)
out = {}


def f32(*shape, scale=1.0):
    return (rng.standard_normal(shape) * scale).astype(np.float32)


# ---- Newton-Schulz ---------------------------------------------------------------------------
muon = Muon(learning_rate=0.02)
for tag, shape in (("wide", (48, 96)), ("tall", (96, 32)), ("square", (64, 64))):
    g = f32(*shape, scale=0.02)
    out[f"ns_{tag}_in"] = g
    out[f"ns_{tag}_out"] = np.asarray(muon.zeropower_via_newtonschulz5(mx.array(g), 5))
# (the reference's mx.transpose(G, axes=(-1, -2)) only accepts 2-D inputs; a batch is a loop)
gb = f32(3, 32, 80, scale=0.02)
out["ns_batched_in"] = gb
out["ns_batched_out"] = np.stack([np.asarray(muon.zeropower_via_newtonschulz5(mx.array(gb[i]), 5)) for i in range(3)])

# ---- Muon.update on a flat module (names are flat, so gradients.get(name) works as intended) ---
shapes = {"w_wide": (32, 64), "w_tall": (80, 16), "gain": (64,)}
params = {k: f32(*s, scale=0.1) for k, s in shapes.items()}
model = nn.Module({k: mx.array(v) for k, v in params.items()})
sched = lambda step: 0.01 * (step + 1)  # noqa: E731
opt = Muon(learning_rate=sched, momentum=0.95, nesterov=True, ns_steps=5)
for step in range(2):
    grads = {k: f32(*s, scale=0.05) for k, s in shapes.items()}
    upd = opt.update(model, {k: mx.array(v) for k, v in grads.items()})
    for k in shapes:
        out[f"muon_s{step}_grad_{k}"] = grads[k]
        out[f"muon_s{step}_upd_{k}"] = np.asarray(upd[k])
        out[f"muon_s{step}_buf_{k}"] = np.asarray(opt.state[k]["momentum_buffer"])
for k, v in params.items():
    out[f"muon_param_{k}"] = v

# ---- Shampoo pieces ----------------------------------------------------------------------------
a = f32(40, 64, scale=0.3)
spd = (a @ a.T).astype(np.float32)
out["root_in"] = spd
out["root_out_p075"] = np.asarray(MatrixSqrt.matrix_inverse_pth_root(mx.array(spd), p=0.75, epsilon=1e-6))
out["root_out_p05"] = np.asarray(MatrixSqrt.matrix_inverse_pth_root(mx.array(spd), p=0.5, epsilon=1e-6))
sh = Shampoo(learning_rate=0.01, params=ShampooParams(beta2=0.95, start_preconditioning_step=1, update_period=1,
                                                      max_preconditioner_dim=32))
p0 = mx.array(f32(48, 40, scale=0.1))
st = sh._init_state(p0, "w")
g1, g2 = f32(48, 40, scale=0.05), f32(48, 40, scale=0.05)
sh._update_statistics(st, mx.array(g1))
sh._update_statistics(st, mx.array(g2))
sh._compute_preconditioners(st, 2)
pre = sh._apply_preconditioners(st, mx.array(g2), 2)
out["sh_g1"], out["sh_g2"] = g1, g2
out["sh_stat0"], out["sh_stat1"] = np.asarray(st["statistics"][0]), np.asarray(st["statistics"][1])
out["sh_pre0"], out["sh_pre1"] = np.asarray(st["preconditioners"][0]), np.asarray(st["preconditioners"][1])
out["sh_preconditioned"] = np.asarray(pre)
gu, su = f32(48, 40, scale=0.01), f32(48, 40, scale=0.3)
out["graft_in_graft"], out["graft_in_shampoo"] = gu, su
out["graft_out"] = np.asarray(sh._apply_grafting(mx.array(gu), mx.array(su)))

# ---- attention (the reference test matrix: B=2, S=16, hidden=128, head_dim=32; 4/4, 4/1, 4/2) ---
S = 16
mask = np.triu(np.full((S, S), -np.inf, dtype=np.float32), k=1)[None, None]
for tag, (H, Hk) in (("mha", (4, 4)), ("mqa", (4, 1)), ("gqa", (4, 2))):
    np.random.seed(7)           # the only draws from this seed are the q/k/v/o_proj weights (not stored)
    attn = FlashAttention(hidden_size=128, num_heads=H, num_kv_heads=Hk, head_dim=32)
    q, k, v = f32(2, S, H, 32), f32(2, S, Hk, 32), f32(2, S, Hk, 32)
    out[f"attn_{tag}_q"], out[f"attn_{tag}_k"], out[f"attn_{tag}_v"] = q, k, v
    out[f"attn_{tag}_causal"] = np.asarray(attn._flash_attention(mx.array(q), mx.array(k), mx.array(v), mx.array(mask)))
    out[f"attn_{tag}_nomask"] = np.asarray(attn._flash_attention(mx.array(q), mx.array(k), mx.array(v), None))
    x = f32(2, S, 128)
    out[f"attn_{tag}_x"] = x
    out[f"attn_{tag}_call"] = np.asarray(attn(mx.array(x), mask=mx.array(mask)))

# ---- RMSNorm / MLP / whole model ----------------------------------------------------------------
x = f32(2, 5, 64)
rn = RMSNorm(64, eps=1e-5)
rn.weight = mx.array((rng.random(64) + 0.5).astype(np.float32))
out["rms_x"], out["rms_w"], out["rms_y"] = x, np.asarray(rn.weight), np.asarray(rn(mx.array(x)))
np.random.seed(11)
mlp = MLP(64, 96)
out["mlp_x"] = x
for nm in ("gate_proj", "up_proj", "down_proj"):
    out[f"mlp_{nm}"] = np.asarray(getattr(mlp, nm).weight)
out["mlp_y"] = np.asarray(mlp(mx.array(x)))

np.random.seed(13)
args = ModelArgs(model_type="llama", hidden_size=64, num_hidden_layers=2, intermediate_size=96,
                 num_attention_heads=4, head_dim=16, vocab_size=67, num_key_value_heads=2,
                 tie_word_embeddings=True, use_flash_attention=True)
model = Model(args)
from mlx.utils import tree_flatten  # noqa: E402
for name, value in tree_flatten(model.parameters()):
    out[f"model_param::{name}"] = np.asarray(value)
tokens = rng.integers(0, 67, size=(2, 12))
out["model_tokens"] = tokens.astype(np.int64)
out["model_logits"] = np.asarray(model(mx.array(tokens)))

# ---- schedules ----------------------------------------------------------------------------------
warm = ref_sched.linear_schedule(0, 3e-4, steps=10)
cos = ref_sched.cosine_decay(3e-4, 100, 3e-5)
joined = ref_sched.join_schedules([warm, cos], [10])
steps = np.array([0, 1, 5, 9, 10, 11, 50, 109, 110, 500])
out["sched_steps"] = steps
out["sched_values"] = np.array([float(joined(int(s))) for s in steps], dtype=np.float64)

# ---- data-parallel contract -------------------------------------------------------------------------
from distributed.hybrid_distributed import HybridDeviceManager  # noqa: E402


class _Devices:  # distribute_batch only looks at the device names
    device_queues = {"mlx:0": None, "cuda:0": None, "cuda:1": None}


dp_batch = rng.integers(0, 100, size=(10, 6)).astype(np.int64)
out["dp_batch"] = dp_batch
for i, (_, sub) in enumerate(HybridDeviceManager.distribute_batch(_Devices(), mx.array(dp_batch))):
    out[f"dp_shard_{i}"] = np.asarray(sub)
dp_grads = [{"w": f32(4, 5), "b": f32(7)} for _ in range(3)]
for i, gd in enumerate(dp_grads):
    for k, v in gd.items():
        out[f"dp_grad_{i}_{k}"] = v
# _aggregate_gradients accumulates IN PLACE into the first worker's arrays: hand it copies
agg = HybridDeviceManager._aggregate_gradients(None, [{k: mx.array(v.copy()) for k, v in gd.items()} for gd in dp_grads])
for k, v in agg.items():
    out[f"dp_mean_{k}"] = np.asarray(v)

# ---- tokenizer + data path (core/training.py:324-543) ----------------------------------------------
import contextlib  # noqa: E402
import io  # noqa: E402
import random as _random  # noqa: E402

import core.training as ref_training  # noqa: E402

data_cfg = ref_training.DataConfig(
    input_file=str(HERE / "tiny_corpus.jsonl"), validation_file=str(HERE / "tiny_val.jsonl"),
    preprocessing={"max_context_size": 96, "chunk_overlap": 16},
    tokenizer={"normal_vocab_size": 256, "special_tokens": {"pad": "<pad>", "bos": "<bos>", "eos": "<eos>"}})
_random.seed(42)
np.random.seed(42)
tok = ref_training.TokenizerManager(data_cfg)
with contextlib.redirect_stdout(io.StringIO()):          # _create_batch prints every batch shape
    dm = ref_training.DataManager(data_cfg, tok, batch_size=3)
    out["data_special"] = np.array([tok.PAD_TOKEN, tok.BOS_TOKEN, tok.EOS_TOKEN, tok.VOCAB_SIZE], dtype=np.int64)
    out["data_num_docs"] = np.array([len(dm.train_docs), len(dm.val_docs), len(dm.train_batch_idx),
                                     dm.num_validation_batches], dtype=np.int64)
    out["data_tokenize_doc"] = np.array(tok.tokenize_doc("naïve 東京 ok"), dtype=np.int64)
    for step in range(8):
        out[f"data_batch_{step}"] = np.asarray(dm.generate_batch(step)).astype(np.int64)
    for i in range(3):
        out[f"data_val_{i}"] = np.asarray(dm.generate_validation_batch(i)).astype(np.int64)

# ---- Trainer.compute_loss (core/training.py:1195-1234) on the tiny model above --------------------------
import logging  # noqa: E402
import types  # noqa: E402

PAD = 66
loss_batch = rng.integers(0, 66, size=(3, 13)).astype(np.int64)
loss_batch[0, 9:] = PAD          # padded tails, as DataManager._create_batch produces them
loss_batch[2, 5:] = PAD
_self = types.SimpleNamespace(
    logger=logging.getLogger("golden"), distributed=False, device_mgr=None,
    config=types.SimpleNamespace(model=types.SimpleNamespace(
        attention={"num_heads": 4, "head_dim": 16, "max_position_embeddings": 64}, dimensions={"hidden_size": 64})),
    mixed_precision=ref_training.MixedPrecisionManager(False), tokenizer=types.SimpleNamespace(PAD_TOKEN=PAD))
loss_val, loss_ntoks = ref_training.Trainer.compute_loss(_self, model, mx.array(loss_batch[:, :-1]),
                                                          mx.array(loss_batch[:, 1:]))
out["loss_batch"] = loss_batch
out["loss_value"] = np.array(float(loss_val), dtype=np.float64)
out["loss_ntoks"] = np.array(int(loss_ntoks), dtype=np.int64)

# ---- scheduler composition and the Shampoo factory defaults (core/training.py:764-856) -------------------
import dataclasses  # noqa: E402


def _tc(scheduler, optimization, lr=1e-2, iters=8000):
    return ref_training.TrainingConfig(hyperparameters={"batch_size": 16, "learning_rate": lr, "weight_decay": 0.01,
                                                        "iters": iters}, scheduler=scheduler, optimization=optimization)


om_steps = np.array([0, 1, 10, 799, 800, 801, 2500, 4000, 7999, 8000, 8799, 9500])
out["om_steps"] = om_steps
for tag, sc in (("warmcos", {"type": "cosine_with_warmup", "min_lr_ratio": 0.05, "warmup_steps": 800}),
                ("cos", {"type": "cosine", "min_lr_ratio": 0.01}), ("lin", {"type": "linear"})):
    sched_fn = ref_training.OptimizationManager(_tc(sc, {"optimizer": "adamw"}), 8000).create_scheduler()
    out[f"om_sched_{tag}"] = np.array([float(sched_fn(int(s))) for s in om_steps], dtype=np.float64)
sh = ref_training.OptimizationManager(_tc({"type": "cosine", "min_lr_ratio": 0.1}, {"optimizer": "shampoo"}, lr=1e-3),
                                      5000)
sh_opt = sh.create_optimizer(sh.create_scheduler())       # every Shampoo knob left to the factory's default
for k, v in dataclasses.asdict(sh_opt.params).items():
    out[f"om_shampoo::{k}"] = np.array(v)

# ---- EarlyStoppingMonitor (core/training.py:621-668): stop decisions over validation-loss sequences -------------
es_rng = np.random.default_rng(77)            # its own generator: the arrays above do not move
es_cases = [
    ({"enabled": True, "patience": 3, "min_delta": 0.001}, np.concatenate([np.linspace(5.0, 3.0, 6), 3.0 + 0.0005 * np.arange(6)])),
    ({"enabled": True, "patience": 2, "min_delta": 0.01}, 4.0 - 0.02 * np.arange(10) + 0.03 * es_rng.standard_normal(10)),
    ({"enabled": True, "patience": 2, "min_delta": 0.0, "mode": "max", "metric": "val_loss"}, np.array([1.0, 1.5, 1.5, 1.4, 1.6, 1.6, 1.6])),
    ({"enabled": False, "patience": 1}, np.array([3.0, 3.1, 3.2, 3.3])),
    ({"enabled": True}, 3.0 + 0.1 * np.abs(es_rng.standard_normal(8))),       # all defaults
]
for i, (es_cfg, seq) in enumerate(es_cases):
    mon = ref_training.EarlyStoppingMonitor(dict(es_cfg))
    stops, counters, bests = [], [], []
    for v in seq:
        stops.append(int(bool(mon.update({"val_loss": float(v)}))))
        counters.append(mon.counter)
        bests.append(mon.best_value)
    out[f"es{i}_seq"] = np.asarray(seq, dtype=np.float64)
    out[f"es{i}_stop"] = np.asarray(stops)
    out[f"es{i}_counter"] = np.asarray(counters)
    out[f"es{i}_best"] = np.asarray(bests, dtype=np.float64)
    out[f"es{i}_cfg"] = np.array(repr(sorted(es_cfg.items())))

# ---- YAML schema: this repo's configs/*.yaml parsed by the REFERENCE's Config dataclasses (core/training.py:52-166)
import json  # noqa: E402

ref_cfg = {p.name: dataclasses.asdict(ref_training.Config.from_yaml(str(p))) for p in sorted((REPO / "configs").glob("c*.yaml"))}
(HERE / "ref_config_parse.json").write_text(json.dumps(ref_cfg, indent=1, sort_keys=True) + "\n")

np.savez_compressed(HERE / "reference_vectors.npz", **out)
print(f"wrote {HERE / 'reference_vectors.npz'} with {len(out)} arrays")
