"""GPU parity at BASELINE.json's REAL dimensions (pytest -m gpu): merlot.yaml sizes -- H=768, 12 heads, 12+12+12 layers,
V=50370 (model/configs/merlot.yaml:28-57, merlot_5segments.yaml:20-33) -- against the oracle on identical weights and inputs.

  cfg1  1 frame 192x320 + 32 tokens, 2-D ids, forward                          (configs[0])
  cfg2  4-segment pretrain step 192x352, batch 2: forward, bit-exact masks, the three losses, every gradient (configs[1])
  cfg4  5 x 384x384 sort_story forward + all-pairs temporal softmax, 2 rows      (configs[3])
  cfg5  K2/K3/K4 at S=3608 with a ragged key mask                                (configs[4])

Every measured error goes into fullsize_parity.json under pytest's temporary directory (pin it with --basetemp).
Tolerances are stated next to each assert: integer paths bit-exact; losses <= 1e-3 relative (north star); bf16 hidden states
rel-Frobenius <= 1.5e-2 after 12(+12) bf16 layers; gradients rel-Frobenius <= 5e-2 per tensor against the fp32 oracle on the
same bf16-rounded weights (bf16 activations on the GPU, fp32 in the oracle: the bound is the bf16 noise of the graph).
"""
import json
import os

import pytest
import torch

from oracle import merlot_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rel(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


@pytest.fixture(scope="module")
def record(tmp_path_factory):
    report = tmp_path_factory.mktemp("fullsize") / "fullsize_parity.json"

    def rec(section, payload):
        d = json.loads(report.read_text()) if report.exists() else {}
        d[section] = payload
        report.write_text(json.dumps(d, indent=1, sort_keys=True))
    return rec


def full_cfg(**over):
    import sys
    sys.path.insert(0, ROOT)
    import bench
    cfg = dict(bench.load_config().model)
    cfg["hidden_dropout_prob"] = 0.0
    cfg.update(over)
    return cfg


OCFG = dict(type="adam_optimizer", learning_rate=3e-4, num_train_steps=460000, num_warmup_steps=10000, weight_decay_rate=0.1,
            beta_2=0.98, clip_norm=0.0, use_bfloat16_adam=True,
            param_overrides=[[["LayerNorm", "layer_norm", "GroupNorm", "bias"], {"weight_decay_rate": 0}]])


@pytest.fixture(scope="module")
def full_model():
    """One parameter set shared by the whole module (223 M parameters; the oracle gets the same bf16-rounded matrices)."""
    from merlot_b200.params import ParamStore
    cfg = full_cfg()
    torch.set_num_threads(min(32, os.cpu_count() or 8))
    params = O.init_params(cfg, seed=1, perturb=0.05)
    params = {k: (v.bfloat16().float() if (k.endswith("kernel") or k.endswith("word_embeddings")) else v) for k, v in params.items()}
    store = ParamStore(cfg, device=DEV, optimizer_cfg=OCFG)
    store.load_tf_dict(params)
    return cfg, params, store


def synth(batch, nc, Lc, h0, w0, seed, ncg):
    g = torch.Generator().manual_seed(seed)
    image = torch.rand(batch * nc, h0, w0, 3, generator=g).bfloat16().float()
    ids = torch.randint(100, 50357, (batch, nc, Lc), generator=g)
    ids[:, :, 0] = O.START
    lens = torch.randint(Lc // 2, Lc + 1, (batch, nc), generator=g)
    ids = (ids * (torch.arange(Lc)[None, None] < lens[..., None])).int()
    B = batch * nc // ncg
    shuf = torch.arange(ncg).repeat(B)
    shuf[:ncg] = 16 + torch.randperm(ncg, generator=g)
    vid = torch.zeros(B, ncg, dtype=torch.int32)
    if B > 1:
        vid[1, ncg // 2:] = 1
    return image, ids, shuf.int(), vid


def test_cfg1_forward_one_segment(full_model, record):
    """configs[0]: MerlotModel forward, 1 frame 192x320 + 32 text tokens, batch 1, 2-D ids (model/modeling.py:72-77)."""
    from merlot_b200.modeling import MerlotModel
    cfg, params, store = full_model
    image, ids, _, _ = synth(1, 1, 32, 192, 320, 11, 1)
    m = MerlotModel(cfg, is_training=False, use_tpu=False, image=image.to(DEV), input_ids=ids[:, 0].to(DEV), params=store)
    om = O.MerlotOracle(cfg, params, image, ids[:, 0])
    assert (m.B, m.L, m.P) == (1, 32, 61) and m.P == om.P  # SURVEY 8: Sv 242, viz_chunk 61, Sj 93
    errs = {n: rel(m.encoder_hidden_states[n], om.encoder_hidden_states[n]) for n in ("viz", "lang")}
    record("cfg1_forward_1x192x320_32tok", errs)
    for n, e in errs.items():
        assert e < 1.5e-2, (n, e)  # rel-Frobenius, 12 ViT + 12 joint bf16 layers vs fp32 oracle


def test_cfg2_pretrain_step_full_size(full_model, record):
    """configs[1] at batch 2 (8 segments): forward, bit-exact masking, three losses, all gradients."""
    from merlot_b200.modeling import MerlotModel
    cfg, params, store = full_model
    batch, nc, Lc = 2, 4, 32
    image, ids, shuf, vid = synth(batch, nc, Lc, 192, 352, 0, 4)
    B, Lj = batch, Lc * 4
    draws = O.make_mask_draws(B, Lj, int(Lj * 0.2), cfg["vocab_size"], seed=5)
    m = MerlotModel(cfg, is_training=False, use_tpu=False, image=image.to(DEV), input_ids=ids.to(DEV), mask_input=True,
                    shuffled_idx_img=shuf.to(DEV), params=store, mask_draws=draws, save_for_backward=True)
    leaf = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    om = O.MerlotOracle(cfg, leaf, image, ids, mask_input=True, shuffled_idx_img=shuf, mask_draws=draws)
    rep = {"dims": dict(Sv=266, Sj=m._dims["Sj"], P=m.P, L=m.L, B=m.B)}
    assert (m.P, m.L, m._dims["Sj"]) == (268, 128, 396)
    rep["attention_summs_rel"] = rel(m.lang_transformer_info["attention_summs"], om.attention_summs)
    assert rep["attention_summs_rel"] < 5e-3
    gm = {"masked_ids": m.lang_mask_info["masked_ids"].cpu().reshape(B, Lj), "masked_idx": m.lang_mask_info["masked_idx"].cpu()}
    same = torch.equal(gm["masked_ids"], om.lang_mask_info["masked_ids"]) and torch.equal(gm["masked_idx"], om.lang_mask_info["masked_idx"])
    rep["masks_bit_exact_from_own_attention"] = bool(same)
    # the masking algorithm itself is bit-exact given the same attention sums (integer path)
    oi = O.mask_inputs(ids.reshape(B, Lj), m.lang_transformer_info["attention_summs"].cpu(), cfg, draws)
    assert torch.equal(gm["masked_ids"], oi["masked_ids"]) and torch.equal(gm["masked_idx"], oi["masked_idx"])
    if not same:  # a near-tie in the bf16 attention sums picked another token: continue from the GPU's masks
        om = O.MerlotOracle(cfg, leaf, image, ids, mask_input=True, shuffled_idx_img=shuf, mask_override=gm)
    for name in ("viz", "lang"):
        rep[f"hidden_{name}_rel"] = rel(m.encoder_hidden_states[name], om.encoder_hidden_states[name])
        assert rep[f"hidden_{name}_rel"] < 1.5e-2, name
    rep["attention_log_abs"] = {k: abs(float(m.attention_log[k]) - float(v)) for k, v in om.attention_log.items()}
    assert max(rep["attention_log_abs"].values()) < 2e-3
    ll, _ = m.mask_loss()
    cl, cinfo = m.contrastive_loss()
    tl, tinfo = m.temporal_loss(shuf.to(DEV), vid.to(DEV))
    total_ref, oinfo = O.pretrain_losses(om, shuf, vid)
    pairs = {"lang": (ll, oinfo["lang"]["loss"]), "contr_lang_to_viz": (cinfo["lang_to_viz"], oinfo["contr"]["lang_to_viz"]),
             "contr_viz_to_lang": (cinfo["viz_to_lang"], oinfo["contr"]["viz_to_lang"]), "contr": (cl, oinfo["contr"]["loss_all"]),
             "temporal_lang_viz": (tinfo["lang_viz_loss"], oinfo["temporal"]["lang_viz_loss"]),
             "temporal_viz_viz": (tinfo["viz_viz_loss"], oinfo["temporal"]["viz_viz_loss"]), "temporal": (tl, oinfo["temporal"]["loss"])}
    rep["losses"] = {k: dict(gpu=float(a), oracle=float(b), rel=abs(float(a) - float(b)) / abs(float(b))) for k, (a, b) in pairs.items()}
    total = float(ll) + float(cl) + float(tl)
    rep["losses"]["total"] = dict(gpu=total, oracle=float(total_ref), rel=abs(total - float(total_ref)) / abs(float(total_ref)))
    record("cfg2_pretrain_step_batch2", rep)
    for k, v in rep["losses"].items():
        assert v["rel"] <= (1e-3 if k in ("lang", "contr", "temporal", "total") else 3e-3), (k, v)  # north star: 1e-3 on the losses
    store.g.zero_()
    m.backward()
    total_ref.backward()
    grads = store.to_tf_dict("g")
    table = {}
    for k, v in leaf.items():
        if v.grad is None or float(v.grad.norm()) < 1e-7:
            continue
        table[k] = rel(grads[k], v.grad)
    worst = sorted(table.items(), key=lambda kv: -kv[1])[:12]
    vals = sorted(table.values())
    rep["grad_rel"] = dict(n=len(vals), median=vals[len(vals) // 2], p90=vals[int(len(vals) * 0.9)], max=vals[-1], worst=worst)
    rep["grad_table"] = table
    record("cfg2_pretrain_step_batch2", rep)
    assert vals[-1] < 5e-2, worst
    assert vals[len(vals) // 2] < 2e-2
    store.g.zero_()


def test_cfg4_sort_story_forward_full_size(full_model, record):
    """configs[3]: 5 x 384x384 frames per story, eval forward, shuffled idx + 64, all-pairs temporal softmax
    (downstream/sort_story/get_zero_shot_logits.py:55-90, merlot_5segments.yaml:20,33)."""
    from merlot_b200.modeling import MerlotModel
    cfg0, params, store = full_model
    cfg = dict(cfg0, num_chunks_in_group=5, image_size=[384, 384])
    rows = 2
    image, ids, _, _ = synth(rows, 5, 32, 384, 384, 4, 5)
    shuf = (torch.stack([torch.randperm(5, generator=torch.Generator().manual_seed(i)) for i in range(rows)]) + 64).int().reshape(-1)
    m = MerlotModel(cfg, is_training=False, use_tpu=False, image=image.to(DEV), input_ids=ids.to(DEV), mask_input=False,
                    shuffled_idx_img=shuf.to(DEV), params=store)
    om = O.MerlotOracle(cfg, params, image, ids, mask_input=False, shuffled_idx_img=shuf)
    assert (m.viz_chunk_length, m.P, m.L, m._dims["Sv"], m._dims["Sj"]) == (145, 725, 160, 578, 885)
    H = cfg["hidden_size"]
    rep = {n: rel(m.encoder_hidden_states[n], om.encoder_hidden_states[n]) for n in ("viz", "lang")}
    h_lang = m.encoder_hidden_states["lang"].reshape(m.B, 5, m.lang_chunk_length, H)[:, :, 0]
    h_viz = m.encoder_hidden_states["viz"].reshape(m.B, 5, m.viz_chunk_length, H)[:, :, 0]
    logits = m.allpairs_temporal_logits(h_lang, h_viz, scope_name="lang_viz_temporal")
    ol = om.encoder_hidden_states["lang"].reshape(om.B, 5, om.lang_chunk_length, H)[:, :, 0]
    ov = om.encoder_hidden_states["viz"].reshape(om.B, 5, om.viz_chunk_length, H)[:, :, 0]
    ref = om.allpairs_temporal_logits(ol, ov, "lang_viz_temporal")
    pg, pr = torch.softmax(logits.float(), -1)[:, 1:].cpu(), torch.softmax(ref, -1)[:, 1:]
    rep["temporal_probs_rel"] = rel(pg, pr)
    rep["temporal_probs_maxabs"] = float((pg - pr).abs().max())
    record("cfg4_sort_story_forward_2x5x384x384", rep)
    assert rep["viz"] < 1.5e-2 and rep["lang"] < 1.5e-2
    assert rep["temporal_probs_rel"] < 1e-2


@pytest.mark.parametrize("masked", [True, False])
def test_cfg5_attention_S3608(masked, record):
    """configs[4] joint sequence (8 x 384 tokens + 8 x 67 viz = 3608): K2 forward, K3 backward and K4 column sums against
    O.attention_core (utils/transformer.py:98-127) with a ragged key mask (padding inside every 384-token caption)."""
    from merlot_b200 import ops
    B, S, heads, H = 2, 3608, 2, 128
    g = torch.Generator().manual_seed(7)
    qkv = (torch.randn(B * S, 3 * H, generator=g) * 0.6).bfloat16()
    dctx = (torch.randn(B * S, H, generator=g) * 0.5).bfloat16()
    valid = torch.ones(B, S, dtype=torch.uint8)
    if masked:
        for b in range(B):
            for c in range(8):  # ragged captions: each 384-token chunk keeps a random-length prefix
                n = int(torch.randint(40, 385, (1,), generator=g))
                valid[b, 536 + c * 384 + n:536 + (c + 1) * 384] = 0
    qkv_d, dctx_d = qkv.to(DEV), dctx.to(DEV)
    vd = valid.to(DEV).reshape(-1) if masked else None
    ctx, lse = ops.attention_fwd(qkv_d, B, S, heads, valid=vd)
    # oracle (fp32 on the same bf16 inputs)
    x = qkv.float().reshape(B, S, 3, heads, 64).permute(2, 0, 3, 1, 4)
    q, k, v = (t.clone().requires_grad_(True) for t in (x[0], x[1], x[2]))
    mask = (valid[:, None, :] & valid[:, :, None]).float() if masked else torch.ones(B, S, S)
    probs, octx = O.attention_core(q, k, v, mask)  # probs [B,h,S,S], ctx [B,h,S,64]
    rep = {"ctx_rel": rel(ctx.reshape(B, S, heads, 64), octx.permute(0, 2, 1, 3))}
    colsum = torch.zeros(B * S, dtype=torch.float32, device=DEV)
    ops.attention_colsum(qkv_d, lse, colsum, B, S, heads, valid=vd)
    rep["colsum_rel"] = rel(colsum.reshape(B, S), probs.detach().mean(1).sum(1))
    octx.permute(0, 2, 1, 3).backward(dctx.float().reshape(B, S, heads, 64))
    dqkv = torch.empty(B * S, 3 * H, dtype=torch.bfloat16, device=DEV)
    dq_acc = ops.attention_bwd_workspace(B, S, heads, DEV)
    dsum = torch.empty(B, heads, S, dtype=torch.float32, device=DEV)
    ops.attention_bwd(qkv_d, ctx, dctx_d, lse, B, S, heads, dqkv=dqkv, dq_accum=dq_acc, dsum=dsum, valid=vd)
    d3 = dqkv.float().cpu().reshape(B, S, 3, heads, 64).permute(2, 0, 3, 1, 4)
    for i, (name, t) in enumerate((("dq", q), ("dk", k), ("dv", v))):
        rep[f"{name}_rel"] = rel(d3[i], t.grad)
    record(f"cfg5_attention_S3608_{'masked' if masked else 'dense'}", rep)
    assert rep["ctx_rel"] < 5e-3 and rep["colsum_rel"] < 5e-3  # bf16 P and bf16 output rounding
    assert max(rep["dq_rel"], rep["dk_rel"], rep["dv_rel"]) < 1e-2
