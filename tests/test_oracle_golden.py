"""CPU: the oracle (oracle/reference_math.py) against golden vectors produced by running the
reference's own Python over the NumPy mlx shim (tests/golden/make_golden.py).  fp32 both sides, so
tolerances are fp32 round-off (different summation order only)."""
import numpy as np
import torch

from oracle import reference_math as R

RTOL = 2e-5


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30)


def t(x):
    return torch.from_numpy(np.asarray(x))


def test_newton_schulz_matches_reference(golden):
    for tag in ("wide", "tall", "square", "batched"):
        x = R.newton_schulz5(t(golden[f"ns_{tag}_in"]), 5)
        assert rel(x.numpy(), golden[f"ns_{tag}_out"]) < 5e-5, tag


def test_muon_update_matches_reference(golden):
    shapes = ("w_wide", "w_tall", "gain")
    params = {k: t(golden[f"muon_param_{k}"]).clone() for k in shapes}
    opt = R.MuonOracle(lambda step: 0.01 * (step + 1), momentum=0.95, nesterov=True, ns_steps=5)
    for step in range(2):
        grads = {k: t(golden[f"muon_s{step}_grad_{k}"]) for k in shapes}
        upd = opt.update(params, grads)
        for k in shapes:
            assert rel(upd[k].numpy(), golden[f"muon_s{step}_upd_{k}"]) < 5e-5, (step, k)
            assert rel(opt.state[k]["momentum_buffer"].numpy(), golden[f"muon_s{step}_buf_{k}"]) < 1e-6, (step, k)


def test_inverse_pth_root_matches_reference(golden):
    m = t(golden["root_in"])
    assert rel(R.matrix_inverse_pth_root(m, 0.75).numpy(), golden["root_out_p075"]) < RTOL
    assert rel(R.matrix_inverse_pth_root(m, 0.5).numpy(), golden["root_out_p05"]) < RTOL


def test_shampoo_statistics_preconditioning_grafting(golden):
    g1, g2 = t(golden["sh_g1"]), t(golden["sh_g2"])
    cap, b2 = 32, 0.95
    L = torch.zeros(cap, cap)
    Rm = torch.zeros(40 if 40 < cap else cap, 40 if 40 < cap else cap)
    for g in (g1, g2):
        lg = g[:cap, :cap]
        L = b2 * L + (1 - b2) * lg @ lg.T
        Rm = b2 * Rm + (1 - b2) * lg.T @ lg
    assert rel(L.numpy(), golden["sh_stat0"]) < RTOL
    assert rel(Rm.numpy(), golden["sh_stat1"]) < RTOL
    PL, PR = R.matrix_inverse_pth_root(L, 0.75), R.matrix_inverse_pth_root(Rm, 0.75)
    assert rel(PL.numpy(), golden["sh_pre0"]) < 1e-4
    assert rel(PR.numpy(), golden["sh_pre1"]) < 1e-4
    pre = g2.clone()
    pre[:cap, :cap] = PL @ g2[:cap, :cap] @ PR
    assert rel(pre.numpy(), golden["sh_preconditioned"]) < 1e-4
    gu, su = t(golden["graft_in_graft"]), t(golden["graft_in_shampoo"])
    assert rel((su * (gu.norm() / su.norm())).numpy(), golden["graft_out"]) < RTOL


def attn_proj_weights(H, Hk, D=32, hidden=128):
    """q/k/v/o_proj weights of the FlashAttention tests/golden/make_golden.py built: mlx's Linear init (uniform in
    +-1/sqrt(fan_in)), drawn in construction order from NumPy's legacy generator seeded with 7.  Regenerated here
    rather than stored; a wrong draw fails the `attn_*_call` comparison below."""
    rs = np.random.RandomState(7)
    w = {}
    for n, (fan_out, fan_in) in (("q", (H * D, hidden)), ("k", (Hk * D, hidden)), ("v", (Hk * D, hidden)),
                                 ("o", (hidden, H * D))):
        s = 1.0 / np.sqrt(fan_in)
        w[n] = t(rs.uniform(-s, s, (fan_out, fan_in)).astype(np.float32))
    return w


def test_attention_matches_reference(golden):
    S = 16
    mask = R.causal_mask(S)
    for tag in ("mha", "mqa", "gqa"):
        q, k, v = (t(golden[f"attn_{tag}_{n}"]) for n in "qkv")
        scale = 32 ** -0.5
        assert rel(R.attention(q, k, v, scale, mask).numpy(), golden[f"attn_{tag}_causal"]) < RTOL, tag
        assert rel(R.attention(q, k, v, scale, None).numpy(), golden[f"attn_{tag}_nomask"]) < RTOL, tag
        # FlashAttention.__call__: projections + attention + o_proj
        x = t(golden[f"attn_{tag}_x"])
        lin = torch.nn.functional.linear
        H = 4
        Hk = k.shape[2]
        w = attn_proj_weights(H, Hk)
        qq = lin(x, w["q"]).reshape(2, S, H, 32)
        kk = lin(x, w["k"]).reshape(2, S, Hk, 32)
        vv = lin(x, w["v"]).reshape(2, S, Hk, 32)
        y = lin(R.attention(qq, kk, vv, scale, mask).reshape(2, S, H * 32), w["o"])
        assert rel(y.numpy(), golden[f"attn_{tag}_call"]) < RTOL, tag


def test_rmsnorm_mlp_match_reference(golden):
    y = R.rmsnorm(t(golden["rms_x"]), t(golden["rms_w"]), 1e-5)
    assert rel(y.numpy(), golden["rms_y"]) < RTOL
    y = R.mlp(t(golden["mlp_x"]), t(golden["mlp_gate_proj"]), t(golden["mlp_up_proj"]), t(golden["mlp_down_proj"]))
    assert rel(y.numpy(), golden["mlp_y"]) < RTOL


def _model_params(golden):
    # mlx tree_flatten names -> oracle names (identical by construction)
    return {k.split("::", 1)[1]: t(golden[k]) for k in golden.files if k.startswith("model_param::")}


def test_llama_forward_matches_reference(golden):
    params = _model_params(golden)
    d = R.LlamaDims(64, 96, 2, 4, 2, 16, 67)
    assert set(R.param_shapes(d)) == set(params), "flattened parameter names differ from the reference's"
    for name, shape in R.param_shapes(d).items():
        assert tuple(params[name].shape) == shape, name
    logits = R.llama_forward(params, t(golden["model_tokens"]), d)
    assert rel(logits.numpy(), golden["model_logits"]) < 5e-5


def test_compute_loss_matches_reference(golden):
    """Trainer.compute_loss (core/training.py:1195-1234) called from the reference's source on the tiny model:
    fp32 cross-entropy, PAD-masked, summed and divided by the number of real tokens."""
    params = _model_params(golden)
    d = R.LlamaDims(64, 96, 2, 4, 2, 16, 67)
    batch = t(golden["loss_batch"])
    logits = R.llama_forward(params, batch[:, :-1], d)
    loss, ntoks = R.compute_loss(logits, batch[:, 1:], pad_token=66)
    assert int(ntoks) == int(golden["loss_ntoks"])
    assert abs(float(loss) - float(golden["loss_value"])) < 2e-5


def test_schedule_matches_reference(golden):
    sched = R.make_schedule({"type": "cosine_with_warmup", "warmup_steps": 10, "min_lr_ratio": 0.1}, 3e-4, 100)
    got = np.array([sched(int(s)) for s in golden["sched_steps"]])
    np.testing.assert_allclose(got, golden["sched_values"], rtol=1e-6, atol=1e-12)


def test_newton_schulz_properties():
    """Self-authored known-answer properties (SURVEY section 4): singular values of NS5 output for
    full-rank Gaussian wide matrices fall in [0.68, 1.14]; tall == transpose of wide."""
    g = torch.Generator().manual_seed(0)
    for shape in ((256, 512), (512, 128)):
        G = torch.randn(shape, generator=g)
        X = R.newton_schulz5(G)
        sv = torch.linalg.svdvals(X)
        assert 0.66 < sv.min() and sv.max() < 1.16, (shape, sv.min(), sv.max())
        assert rel(R.newton_schulz5(G.T).numpy(), X.T.numpy()) < 1e-5


def test_dp_contract_matches_reference(golden):
    """distributed/hybrid_distributed.py:303-354 (_aggregate_gradients) and :430-452 (distribute_batch), run
    from the reference's own source: unweighted mean over workers, remainder rows to the last shard -- for the
    oracle AND for the product's host-side helper."""
    from mlx_cuda_distributed_pretraining_b200.distributed import dp
    per_dev = [{k: torch.from_numpy(golden[f"dp_grad_{i}_{k}"]) for k in ("w", "b")} for i in range(3)]
    mean = R.mean_gradients(per_dev)
    for k in ("w", "b"):
        assert rel(mean[k].numpy(), golden[f"dp_mean_{k}"]) < 1e-6
    batch = torch.from_numpy(golden["dp_batch"])
    for r in range(3):
        assert torch.equal(dp.shard_batch(batch, r, 3), torch.from_numpy(golden[f"dp_shard_{r}"]))
    # the CUDA path reaches the same mean as sum-all-reduce * (1/world) folded into the optimizer's gradient scale
    flat_sum = sum(torch.cat([d["w"].flatten(), d["b"]]) for d in per_dev)
    want = torch.cat([torch.from_numpy(golden["dp_mean_w"]).flatten(), torch.from_numpy(golden["dp_mean_b"])])
    assert rel((flat_sum * (1.0 / 3)).numpy(), want.numpy()) < 1e-6


def test_tokenizer_and_data_path_match_reference(golden):
    """core/training.py:324-543 run from the reference's own source on tests/golden/tiny_corpus.jsonl: byte-level
    special-token ids, document chunking with overlap, length-sorted + shuffled batch order (same global RNG
    calls under the seeds Trainer.setup_system sets), padding / truncation, and the validation walk."""
    import random
    import numpy as np
    from pathlib import Path
    from mlx_cuda_distributed_pretraining_b200.core.training import DataConfig, DataManager, TokenizerManager
    here = Path(__file__).resolve().parent / "golden"
    cfg = DataConfig(input_file=str(here / "tiny_corpus.jsonl"), validation_file=str(here / "tiny_val.jsonl"),
                     preprocessing={"max_context_size": 96, "chunk_overlap": 16},
                     tokenizer={"normal_vocab_size": 256,
                                "special_tokens": {"pad": "<pad>", "bos": "<bos>", "eos": "<eos>"}})
    random.seed(42)
    np.random.seed(42)
    tok = TokenizerManager(cfg)
    dm = DataManager(cfg, tok, batch_size=3)
    assert [tok.PAD_TOKEN, tok.BOS_TOKEN, tok.EOS_TOKEN, tok.VOCAB_SIZE] == golden["data_special"].tolist()
    assert [len(dm.train_docs), len(dm.val_docs), len(dm.train_batch_idx), dm.num_validation_batches] == \
        golden["data_num_docs"].tolist()
    assert tok.tokenize_doc("naïve 東京 ok") == golden["data_tokenize_doc"].tolist()
    for step in range(8):
        assert torch.equal(dm.generate_batch(step), torch.from_numpy(golden[f"data_batch_{step}"])), step
    for i in range(3):
        assert torch.equal(dm.generate_validation_batch(i), torch.from_numpy(golden[f"data_val_{i}"])), i
    assert tok.detokenize(golden["data_tokenize_doc"][1:-1]) == "naïve 東京 ok"


def test_scheduler_and_shampoo_factory_match_reference(golden):
    """core/training.py:764-856 run from the reference's own OptimizationManager: the three scheduler types as
    composed there (cosine sees step - warmup, total_steps not reduced by the warm-up) and the ShampooParams the
    factory builds when the YAML leaves every knob at its default -- for the oracle and for the product."""
    import dataclasses
    from mlx_cuda_distributed_pretraining_b200.core.training import OptimizationManager, TrainingConfig
    steps = golden["om_steps"]

    def tc(scheduler, optimization, lr=1e-2, iters=8000):
        return TrainingConfig(hyperparameters={"batch_size": 16, "learning_rate": lr, "weight_decay": 0.01,
                                               "iters": iters}, scheduler=scheduler, optimization=optimization)

    for tag, sc in (("warmcos", {"type": "cosine_with_warmup", "min_lr_ratio": 0.05, "warmup_steps": 800}),
                    ("cos", {"type": "cosine", "min_lr_ratio": 0.01}), ("lin", {"type": "linear"})):
        fn = OptimizationManager(tc(sc, {"optimizer": "adamw"}), 8000).create_scheduler()
        got = np.array([float(fn(int(s))) for s in steps])
        assert np.allclose(got, golden[f"om_sched_{tag}"], rtol=1e-6, atol=1e-12), tag
    want = golden["om_sched_warmcos"]
    sched = R.make_schedule({"type": "cosine_with_warmup", "min_lr_ratio": 0.05, "warmup_steps": 800}, 1e-2, 8000)
    assert np.allclose([sched(int(s)) for s in steps], want, rtol=1e-6, atol=1e-12)
    om = OptimizationManager(tc({"type": "cosine", "min_lr_ratio": 0.1}, {"optimizer": "shampoo"}, lr=1e-3), 5000)
    params = dataclasses.asdict(om.create_optimizer(om.create_scheduler()).params)
    ref = {k.split("::", 1)[1]: golden[k] for k in golden.files if k.startswith("om_shampoo::")}
    assert set(params) == set(ref)
    for k, v in params.items():
        assert str(v) == str(ref[k].item()) or float(v) == float(ref[k]), (k, v, ref[k])


def test_dp_contract():
    g = [{"w": torch.ones(2, 2) * i} for i in (1.0, 3.0)]
    assert torch.equal(R.mean_gradients(g)["w"], torch.ones(2, 2) * 2.0)
    assert abs(R.token_weighted_loss([1.0, 3.0], [10, 30]) - 2.5) < 1e-12
