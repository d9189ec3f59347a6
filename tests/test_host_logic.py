"""CPU tests of the host-side mirror: config surface, parameter arena, C-ABI export, error behaviour."""
import json
import os

import pytest
import torch

from merlot_b200 import _lib
from merlot_b200.config import NeatConfig, patch_embed_variant
from merlot_b200.params import ParamStore

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def test_library_exports_every_header_symbol():
    lib = _lib.lib()
    names = _lib.exported_symbols_from_header()
    assert len(names) >= 40
    for n in names:
        assert hasattr(lib, n), n
    assert lib.merlot_abi_version() == 1


def test_ctypes_structs_match_the_header_layout(tmp_path):
    """The descriptor structs of include/merlot_b200.h compiled by gcc (sizeof and the offset of the last member) against their
    ctypes mirrors in merlot_b200/_lib.py: a field added on one side only would shift every later argument silently."""
    import ctypes
    import subprocess
    pairs = [("merlot_gemm_t", _lib.GemmDesc), ("merlot_attn_t", _lib.AttnDesc), ("merlot_ln_t", _lib.LnDesc),
             ("merlot_ln_bwd_t", _lib.LnBwdDesc), ("merlot_layer_params_t", _lib.LayerParams), ("merlot_stack_t", _lib.StackDesc),
             ("merlot_mask_t", _lib.MaskDesc), ("merlot_adamw_t", _lib.AdamDesc), ("merlot_ws_item_t", _lib.WsItem)]
    src = tmp_path / "sizes.c"
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "merlot_b200.h"', 'int main(void) {']
    for cname, cls in pairs:
        last = cls._fields_[-1][0]
        lines.append(f'  printf("{cname} %zu %zu\\n", sizeof({cname}), offsetof({cname}, {last}));')
    lines += ['  return 0;', '}']
    src.write_text("\n".join(lines))
    exe = tmp_path / "sizes"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = dict((ln.split()[0], tuple(int(v) for v in ln.split()[1:])) for ln in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for cname, cls in pairs:
        last = cls._fields_[-1][0]
        assert out[cname] == (ctypes.sizeof(cls), getattr(cls, last).offset), (cname, out[cname], ctypes.sizeof(cls), getattr(cls, last).offset)


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours): ONE JSON line on stdout with the contract's keys,
    the oracle port named as such, zero device traffic and no GPU launches."""
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "segments/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["gpu_launches"] == 0
    assert "workload" in d["config"]


def test_bench_dump_outputs_are_float_seeded_and_bounded(tmp_path, tiny_cfg):
    """`bench.py --dump-outputs DIR`: float32/float64 .npy files within 64 MB, identical for identical state, and the parameter
    sample reads the reference-named, name-sorted concatenation at the positions the fixed seed draws."""
    import sys
    from types import SimpleNamespace
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    st = ParamStore(tiny_cfg, device="cpu")
    st.init_reference(seed=0)
    spec = SimpleNamespace(loss_parts=(torch.tensor(2.5), torch.tensor(0.75), torch.tensor(1.25)),
                           metrics={"lang/loss": torch.tensor(2.5), "contr/lang_to_viz": torch.tensor(0.5), "learning_rate": 3e-7},
                           model=SimpleNamespace(encoder_hidden_states={"viz": torch.randn(2, 14, 128), "lang": torch.randn(2, 32, 128)}))
    for d in ("a", "b"):
        bench.write_outputs(str(tmp_path / d), spec, st)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b")) and "params_sample.npy" in names and "loss_parts.npy" in names
    assert "metric_contr_lang_to_viz.npy" in names and "hidden_viz.npy" in names
    total = 0
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), n
        total += a.nbytes
    assert total <= 64 << 20
    assert np.load(tmp_path / "a" / "loss_parts.npy").tolist() == [2.5, 0.75, 1.25]
    params = st.to_tf_dict("p")
    flat = np.concatenate([params[k].reshape(-1).numpy() for k in sorted(params)])
    idx = np.unique(np.random.default_rng(0).integers(0, flat.size, bench.DUMP_PARAM_SAMPLE))
    assert np.array_equal(np.load(tmp_path / "a" / "params_sample.npy"), flat[idx])


def test_pairwise_partner_words_equal_the_reference_mask():
    """disable_pairwise_lang_attn (model/modeling.py:160-168): the attention kernels never see an [S, S] mask -- every row
    derives its partners as two bit ranges per 32-position word (csrc/attention_tcgen05.cu: span_word / pair_lo_of / pair_word).
    The same integer arithmetic restated here must reproduce the reference's segment_idx construction bit for bit, for chunk
    lengths that are not word-aligned, P = 0, single-token chunks, and the 16-bit extraction K3 uses."""
    def span_word(x0, a, b):
        lo, hi = max(a - x0, 0), min(b - x0, 32)
        if hi <= lo:
            return 0
        return (0xFFFFFFFF if hi >= 32 else (1 << hi) - 1) & ((0xFFFFFFFF << lo) & 0xFFFFFFFF)

    def pair_lo_of(t, P, chunk):
        return P + ((t - P) // chunk) * chunk if (chunk > 0 and t >= P) else -1

    def pair_word(x0, lo, P, chunk):
        return 0xFFFFFFFF if lo < 0 else (span_word(x0, 0, P) | span_word(x0, lo, lo + chunk))

    for P, chunk, nch in [(13, 8, 4), (100, 32, 5), (0, 16, 6), (70, 33, 3), (31, 1, 40), (64, 64, 2)]:
        S = P + chunk * nch
        seg = torch.cat([torch.zeros(P, dtype=torch.int64), 1 + torch.arange(chunk * nch) // chunk])  # :162-164
        can = (seg[:, None] == seg[None]) | (seg == 0)[None] | (seg == 0)[:, None]                    # :165-167
        for t in range(S):
            lo = pair_lo_of(t, P, chunk)
            bits = []
            for x0 in range(0, (S + 31) // 32 * 32, 32):
                w = pair_word(x0, lo, P, chunk)
                bits += [(w >> i) & 1 for i in range(32)]
            assert bits[:S] == can[t].int().tolist(), (P, chunk, t)
            for qb in range(0, S, 16):  # K3: 16 queries at a time out of the 32-position word
                aw = (pair_word(qb & ~31, lo, P, chunk) >> (qb & 31)) & 0xFFFF
                n = min(16, S - qb)
                assert [(aw >> i) & 1 for i in range(n)] == can[t, qb:qb + n].int().tolist()


def test_neatconfig_errors_mirror_reference():  # utils/neat_config.py:55-61
    with pytest.raises(ValueError, match="missing model"):
        NeatConfig.from_dict({"data": {}, "optimizer": {}, "device": {"output_dir": "x"}})
    with pytest.raises(ValueError, match="Missing output directory"):
        NeatConfig.from_dict({"data": {}, "model": {}, "optimizer": {}, "device": {}})
    with pytest.raises(ValueError, match="No config file"):
        NeatConfig.from_args(argv=[])


def test_bench_config_equals_reference_yaml():
    """bench.load_config() restates merlot.yaml (the reference tree does not travel to the GPU box); the golden fixture
    generated from the real YAML pins it.  Only resnet_layers differs (patch-embed variant, SURVEY discrepancy 1)."""
    import sys
    sys.path.insert(0, ROOT)
    import bench
    cfg = bench.load_config()
    gold = json.load(open(os.path.join(HERE, "golden", "reference_facts.json")))["configs"]["merlot.yaml"]
    assert cfg.model == patch_embed_variant(gold["model"])
    assert cfg.optimizer == gold["optimizer"]


def test_hybrid_stem_param_arena(tiny_cfg):
    """merlot.yaml as shipped selects the hybrid ResNet-lite stem: the store holds its 164 variables under the reference's
    names (conv kernels flattened [kh*kw*cin, cout]) and round-trips them HWIO against the oracle's independent name walk."""
    from oracle import merlot_oracle as O
    cfg = dict(tiny_cfg, resnet_layers=[1, 2, 1], patch_size=16)
    st = ParamStore(cfg, device="cpu")
    params = O.init_params(cfg, seed=0, perturb=0.1)
    st.load_tf_dict(params)
    back = st.to_tf_dict("p")
    assert set(back) == set(params)
    for k in params:
        assert back[k].shape == params[k].shape and torch.equal(back[k], params[k]), k
    vt = "vision_backbone/vision_transformer"
    assert f"{vt}/conv2d/kernel" not in st.entries and f"{vt}/conv_postresnet_proj/kernel" in st.entries
    assert st.entries[f"{vt}/resnet50lite/block_group2/conv2d_2/kernel"].shape == (9 * 128, 128)
    gn = st.entries[f"{vt}/resnet50lite/stem/GroupNorm_stem0/gamma"]
    assert gn.hyper[1] == 0.0  # "GroupNorm" matches the weight-decay-0 override (optimization.py:125-147)
    gold = json.load(open(os.path.join(HERE, "golden", "reference_facts.json")))["configs"]["merlot.yaml"]
    from merlot_b200.params import stem_variables
    n_stem = sum(int(torch.tensor(s_).prod()) for _, s_ in stem_variables(vt, gold["model"]["resnet_layers"], 64, 768))
    assert n_stem == 11_914_080 + 1024 * 768 + 768  # SURVEY Appendix D: 11.91 M + 0.79 M


def test_param_arena_roundtrip_and_count(tiny_cfg):
    from oracle import merlot_oracle as O
    st = ParamStore(tiny_cfg, device="cpu")
    params = O.init_params(tiny_cfg, seed=0, perturb=0.1)
    st.load_tf_dict(params)
    back = st.to_tf_dict("p")
    assert set(back) == set(params)
    for k in params:
        assert torch.equal(back[k], params[k]), k
    assert st.num_params() == sum(v.numel() for v in params.values())
    # decayed group first, then the LayerNorm/bias group with weight decay 0
    assert [h[1] for h, _, _ in st.groups] == sorted([h[1] for h, _, _ in st.groups], reverse=True)
    for e in st.entries.values():
        assert e.offset % 64 == 0


def test_full_size_param_count():
    import sys
    sys.path.insert(0, ROOT)
    import bench
    st = ParamStore.__new__(ParamStore)
    from merlot_b200.params import _entries
    import math
    n = sum(math.prod(e.shape) if "temporal/logits" not in e.name else math.prod(e.shape) // 2 for e in _entries(bench.load_config().model))
    assert n == 223423946  # SURVEY Appendix A: 223.42 M (pure ViT)


def test_optimizer_factory_errors():  # utils/optimization.py:23-24,178-179
    from merlot_b200.optimization import build_optimizer_from_config
    with pytest.raises(ValueError, match="isn't supported"):
        build_optimizer_from_config(None, {"type": "sgd"}, None, store=None)
    with pytest.raises(ValueError, match="Adafactor"):
        build_optimizer_from_config(None, {"type": "adam_optimizer", "learning_rate": 1, "num_train_steps": 1, "num_warmup_steps": 0,
                                           "adafactor": True}, None, store=None)


def test_no_cpu_fallback():
    from merlot_b200 import ops
    with pytest.raises(_lib.MerlotError):
        ops.gemm(torch.zeros(8, 8, dtype=torch.bfloat16), torch.zeros(8, 8, dtype=torch.bfloat16))


# ---------------------------------------------------------------------------------------------------------------
# batch-level input step (model/dataloader.py:210-272; SURVEY 8(f) next-row 4): integer results bit-exact vs NumPy
# ---------------------------------------------------------------------------------------------------------------
def test_process_example_matches_numpy_restatement():
    import numpy as np
    from merlot_b200 import dataloader as D
    from oracle import oracle_np as N
    b, n, g, L = 3, 8, 4, 5
    gen = torch.Generator().manual_seed(0)
    feats = {
        "images": torch.rand(b, n, 4, 6, 3, generator=gen),
        "input_ids": torch.randint(0, 1000, (b, n, L), generator=gen, dtype=torch.int32),
        "video_src_ids": torch.tensor([[0, 0, 0, 0, 1, 1, 2, 2], [0, 0, 0, 0, 0, 0, 0, 0], [0, 1, 1, 1, 1, 2, 2, 2]], dtype=torch.int32),
        "chunk_num": torch.arange(b * n, dtype=torch.int32).reshape(b, n),
    }
    model_cfg = {"num_chunks_in_group": g, "image_shuffle_prob": 0.4, "transpose_input": True}
    for seed in range(5):
        draws = D.make_draws(b, n, g, 0.4, seed)
        out = D.process_example(feats, {"shuffle_chunks": True}, model_cfg, is_training=True, draws=draws)
        idx, shuf = N.process_example_np(feats["input_ids"].numpy(), feats["video_src_ids"].numpy(), draws["chunk_u"].numpy(),
                                         draws["num_shuffle"].numpy(), draws["pick_u"].numpy(), draws["order_u"].numpy(), g, 0.4, True)
        assert np.array_equal(out["shuffled_idx_img"].numpy(), shuf)
        for r in range(b):
            assert np.array_equal(out["input_ids"][r].numpy(), feats["input_ids"][r].numpy()[idx[r]])
            assert np.array_equal(out["chunk_num"][r].numpy(), feats["chunk_num"][r].numpy()[idx[r]])
            vs = out["video_src_ids"][r].tolist()  # whole videos move together and keep their internal order (:212-213)
            assert all(vs.count(v) == feats["video_src_ids"][r].tolist().count(v) for v in set(vs))
            assert [k for k, _ in __import__("itertools").groupby(vs)] == list(dict.fromkeys(vs))
            for v in set(vs):
                pos = [i for i, q in enumerate(vs) if q == v]
                assert out["chunk_num"][r][pos].tolist() == sorted(out["chunk_num"][r][pos].tolist())
        img = out["images"]
        assert tuple(img.shape) == (4, 6, 3, b * n)  # flattened, then [h, w, 3, N] for the TPU-friendly transpose (:262-264)
        flat = img.permute(3, 0, 1, 2)
        assert torch.equal(flat[1 * n + 2], feats["images"][1][idx[1][2]])
        s = out["shuffled_idx_img"].reshape(b * n // g, g)
        for row, k in zip(s.tolist(), draws["num_shuffle"].tolist()):
            moved = [v for v in row if v >= 16]
            assert len(moved) == k and len(set(moved)) == k and all(16 <= v < 16 + g for v in moved)
            assert all(v == j for j, v in enumerate(row) if v < 16)
    # no shuffling at all: identity ids, images only flattened in eval mode
    out = D.process_example(feats, {}, {"num_chunks_in_group": g, "image_shuffle_prob": 0.0}, is_training=False)
    assert out["shuffled_idx_img"].tolist() == list(range(g)) * (b * n // g) and tuple(out["images"].shape) == (b * n, 4, 6, 3)
    assert torch.equal(out["input_ids"], feats["input_ids"])
    assert D.num_shuffle_probs(4, 0.4)[:2] == [0.6, 1e-6] and abs(D.expected_out_of_place(4, 0.4) - (1.2 + 1e-6)) < 1e-12
    with pytest.raises(ValueError):
        D.process_example({**feats, "input_ids": feats["input_ids"][:, :7]}, {}, model_cfg)


def test_hybrid_stem_orchestration_against_autograd():
    """tools/stem_cpu_emulation.py: the stem's forward tape and backward walk (merlot_b200/modeling.py) driven with fp32
    emulations of the K13 / K1 calls must reproduce the oracle's forward and torch-autograd parameter gradients (< 1e-3; it
    reaches ~2e-6).  Runs in a subprocess because it swaps merlot_b200.ops entry points."""
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "stem_cpu_emulation.py")], cwd=ROOT, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "parameter gradients, worst rel err" in r.stdout


def test_sort_story_scoring_matches_loop_restatement():
    """downstream/sort_story/score_permutations.py:15-71 restated with explicit loops (as the reference writes it) vs the
    vectorised merlot_b200.sort_story; closed-form metric values."""
    import itertools
    import numpy as np
    from scipy import stats
    from merlot_b200 import sort_story as S
    rng = np.random.default_rng(0)
    for n in (3, 5):
        for _ in range(4):
            p = rng.dirichlet(np.ones(3), size=(n, n))
            best, best_score = None, -np.inf
            for perm in itertools.permutations(range(n)):
                eq, gtlt = np.ones((n, n)), np.ones((n, n))
                for i in range(n):
                    for j, pj in enumerate(perm):
                        if i == pj:
                            eq[i, j] = p[i, j, 0]
                        elif i < pj:
                            gtlt[i, j] = p[i, j, 1]
                        else:
                            gtlt[i, j] = p[i, j, 2]
                sc = np.log(eq).sum() + np.log(gtlt).sum()
                if sc > best_score:  # strict: the first maximum in itertools order, like the reference's stable sort
                    best, best_score = perm, sc
            got, got_score = S.best_permutation(p)
            assert got == best and abs(got_score - best_score) < 1e-9
    n = 5  # a model that is certain of the true order recovers it; the reversed story gets the reversed permutation
    sure = np.full((n, n, 3), 1e-6)
    for i in range(n):
        for j in range(n):
            sure[i, j, 0 if i == j else (1 if i < j else 2)] = 1.0
    assert S.best_permutation(sure)[0] == (0, 1, 2, 3, 4)
    assert S.best_permutation(sure[:, ::-1])[0] == (4, 3, 2, 1, 0)
    assert S.pairwise_acc([0, 1, 2, 3, 4]) == 1.0 and S.pairwise_acc([4, 3, 2, 1, 0]) == 0.0 and S.pairwise_acc([1, 0, 2, 3, 4]) == 0.9
    assert S.absolute_distance([4, 3, 2, 1, 0]) == 2.4 and S.absolute_distance([0, 1, 2, 3, 4]) == 0.0
    for story in ([0, 1, 2, 3, 4], [4, 3, 2, 1, 0], [1, 0, 2, 4, 3], [2, 0, 1, 4, 3]):
        assert abs(S.spearman_acc(story) - stats.spearmanr(story, [0, 1, 2, 3, 4])[0]) < 1e-12
    ev = S.evaluate([sure, sure[:, ::-1]])
    assert ev["stories"] == [(0, 1, 2, 3, 4), (4, 3, 2, 1, 0)] and ev["pairwise"] == 0.5 and abs(ev["spearman"]) < 1e-12
    with pytest.raises(ValueError):
        S.permutation_scores(np.ones((5, 4, 3)))


def test_vit_gradient_buckets_partition_the_vit_ranges():
    """train.py's bucketed all-reduce: the buckets are disjoint, ordered top-down and cover exactly the ViT part of the arena."""
    import sys, os
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    from merlot_b200.params import ParamStore
    cfg = bench.load_config()
    st = ParamStore(cfg.model, device="cpu", optimizer_cfg=cfg.optimizer)
    for n in (1, 3, 4, 12):
        groups, ranges = st.vit_buckets(n)
        assert groups[0][1] == 12 and groups[-1][0] == 0 and all(groups[i][0] == groups[i + 1][1] for i in range(len(groups) - 1))
        flat = sorted(r for rs in ranges for r in rs)
        assert all(flat[i][1] <= flat[i + 1][0] for i in range(len(flat) - 1))                      # disjoint
        assert sum(b - a for a, b in flat) == sum(b - a for a, b in st.vit_ranges)                   # complete
        for (lo, hi), rs in zip(groups[:-1], ranges[:-1]):                                           # a bucket holds exactly its layers' kernels
            names = [e.name for e in st.entries.values() if any(a <= e.offset < b for a, b in rs)]
            assert names and all(lo <= int(nm.split("/layer")[1][:2]) < hi and nm.endswith("/kernel") for nm in names)


def test_multi_replica_contrastive_restatement_reduces_to_single_replica():
    """oracle.contrastive_loss_replicas with one replica == MerlotOracle.contrastive_loss; with two, labels are shifted by
    rank * N (model/modeling.py:519) and each replica sees the other's features as extra negatives."""
    import torch
    from oracle import merlot_oracle as O
    from tests.test_gpu_model import synth
    cfg = dict(use_bfloat16=True, hidden_size=64, vocab_size=500, patch_size=16, spatial_pool_size=2, num_attention_heads=1,
               num_hidden_layers=1, num_vision_transformer_hidden_layers=1, num_lang_transformer_hidden_layers=1, intermediate_size=128,
               initializer_range=0.02, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0, max_position_embeddings=64,
               num_chunks_in_group=2, do_projection=True, do_bias=True, contrastive_size=64, contrast_coef=0.25, contrast_temp=0.05,
               image_shuffle_prob=0.4, masking_rate=0.2, resnet_layers=[])
    params = O.init_params(cfg, seed=1, perturb=0.05)
    data = [synth(cfg, 2, 2, 16, 32, 48, 10 + r) for r in range(2)]
    oms = [O.MerlotOracle(cfg, params, d[0], d[1], mask_input=True, shuffled_idx_img=d[2], mask_draws=O.make_mask_draws(2, 32, 6, 500, seed=3)) for d in data]
    single, _ = oms[0].contrastive_loss()
    one, _ = O.contrastive_loss_replicas([oms[0]], 0)
    assert float(single) == float(one)
    two0, _ = O.contrastive_loss_replicas(oms, 0)
    two1, _ = O.contrastive_loss_replicas(oms, 1)
    assert float(two0) > float(single)  # more negatives, same positives => larger cross entropy
    # replica 1's positives sit at columns N..2N-1 of the gathered matrix
    lx, vx = oms[1]._ctr_feats
    all_v = torch.cat([oms[0]._ctr_feats[1], vx], 0)
    logits = lx @ all_v.t() / 0.05
    n = lx.shape[0]
    assert torch.allclose(O.raw_cross_entropy_with_logits(logits, torch.arange(n) + n).mean() * 0.125 +
                          O.raw_cross_entropy_with_logits(vx @ torch.cat([oms[0]._ctr_feats[0], lx], 0).t() / 0.05, torch.arange(n) + n).mean() * 0.125,
                          two1)


def test_sort_story_logit_container_round_trip(tmp_path):
    """write_logits_npz / read_logits_npz carry the records of get_zero_shot_logits.py:105-119 (h5py is not in this image; the
    HDF5 writer raises ImportError instead of silently writing something else) and feed the scorer unchanged."""
    import numpy as np
    import pytest
    from merlot_b200 import sort_story as ss
    rng = np.random.RandomState(0)
    preds = []
    for sid in (7, 9, 7):  # a duplicate story id is skipped, like the reference's `except ValueError: continue`
        p = rng.dirichlet(np.ones(3), size=(5, 5))
        preds.append({"story_id": sid, "permutation_identity_encode": rng.permutation(5), "sentences": rng.randint(0, 100, (5, 32)),
                      "lang_viz_probs": p, "viz_viz_probs": p[::-1].copy(), "images": rng.rand(5, 4, 4, 3)})
    path = str(tmp_path / "logits_val.npz")
    assert ss.write_logits_npz(path, preds, include_images=True) == 2
    back = ss.read_logits_npz(path)
    assert sorted(back) == ["7", "9"] and back["7"]["images"].dtype == np.uint8
    assert np.array_equal(back["9"]["lang_viz_probs"], preds[1]["lang_viz_probs"])
    perms, scores = ss.permutation_scores(back["7"]["lang_viz_probs"])
    assert perms.shape == (120, 5) and np.isfinite(scores).all()
    try:
        import h5py  # noqa: F401
    except ImportError:
        with pytest.raises(ImportError):
            ss.write_logits_h5(str(tmp_path / "x.h5"), preds)
    idx = ss.fixed_shuffle_index(3, 5)
    assert idx.shape == (3, 5) and all(sorted(r - 64) == list(range(5)) for r in idx) and np.array_equal(idx, ss.fixed_shuffle_index(3, 5))
