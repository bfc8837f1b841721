"""The oracle restatement vs. the golden outputs of the UNMODIFIED reference (CPU, no GPU)."""
import os
import subprocess
import sys

import torch
import pytest

from oracle import fourm_oracle as O
from oracle import vq_oracle as V
from tests import helpers as H


@pytest.fixture(scope="module")
def tiny():
    gold = H.load_golden("fourm_tiny_golden.pt")
    specs = O.mod7_specs()
    sd = H.fill_fourm_buffers(H.golden_state_dict(gold), specs, 384)
    for k, c in gold["weight_checksums"].items():
        assert abs(float(sd[k].double().sum()) - c) <= 1e-6 * max(1.0, abs(c)), f"fixture weight drift in {k}"
    return gold, specs, sd


def test_static_known_answers():
    st = H.load_golden("static_golden.pt")
    for m, i in st["mod_ids"].items():
        assert O.modality_id(m) == i
    assert O.modality_id("rgb@224") == 20716 and O.modality_id("caption") == 32652      # SURVEY.md 4
    assert torch.equal(O.sincos_1d(8, 16), st["sincos1d_8x16"])
    assert torch.equal(O.sincos_2d(3, 5, 8), st["sincos2d_3x5x8"])
    assert torch.equal(O.sincos_2d(14, 14, 384).double().sum(-1), st["sincos2d_14x14x384_sum"])


@pytest.mark.parametrize("tag", ["fp32_128", "bf16_128", "fp32_trunc", "fp32_pad"])
def test_fourm_forward_matches_reference(tiny, tag):
    gold, specs, sd = tiny
    c = gold["cases"][tag]
    batch = O.synthetic_mod7_batch(2, seed=c["batch_seed"], extra_valid=c["extra_valid"])
    order = H.decoder_order(c["py_seed"], [m for m in batch if specs[m]["kind"] != "img"])
    assert order == c["decoder_order"]
    cfg = O.PRESETS[gold["model"]]
    with torch.autocast("cpu", dtype=torch.bfloat16, enabled=c["amp"]):
        loss, mod_loss, it = O.fourm_forward(sd, cfg, specs, batch, c["N"], c["M"], order, "mod", return_intermediates=True)
        tl, _ = O.fourm_forward(sd, cfg, specs, batch, c["N"], c["M"], order, "token")
        logits = O.fourm_forward(sd, cfg, specs, batch, c["N"], c["M"], order, return_logits=True)
    # integer / bool parts: exact
    assert torch.equal(it["enc_mask"], c["enc_mask"]) and torch.equal(it["dec_mask"], c["dec_mask"])
    assert torch.equal(it["enc_mod"], c["enc_mod"]) and torch.equal(it["dec_mod"], c["dec_mod"])
    assert torch.equal(it["target_ids"], c["target_ids"]) and it["target_ids"].dtype == c["target_ids"].dtype
    assert torch.equal(it["dec_attn_mask"], c["dec_attn_mask"])
    if not c["amp"]:   # the golden intermediates were taken outside autocast
        assert torch.equal(it["enc_x0"].double().sum(-1), c["enc_x0_sum"])
        assert torch.equal(it["dec_y0"].double().sum(-1), c["dec_y0_sum"])
    # floating point: same ops in the same order -> tight
    tol = 2e-3 if c["amp"] else 1e-5
    assert abs(float(loss) - float(c["loss"])) <= tol
    assert abs(float(tl) - float(c["token_loss"])) <= tol
    for m, v in c["mod_loss"].items():
        assert abs(float(mod_loss[m]) - float(v)) <= tol, m
    for m, v in c["logits_slices"].items():
        torch.testing.assert_close(logits[m][:, :4, :32].float(), v, rtol=tol * 10, atol=tol * 10)


def test_fourm_backward_matches_reference(tiny):
    gold, specs, sd = tiny
    c = gold["cases"]["fp32_128"]
    names = set(gold["param_names"])
    sdg = {k: (v.clone().requires_grad_(True) if k in names else v) for k, v in sd.items()}
    # shared parameters (fm.py:176-180, decoder_embeddings.py:89-91): same tensor object under both names
    for m, s in specs.items():
        e, d = f"encoder_embeddings.{m}.mod_emb", f"decoder_embeddings.{m}.mod_emb"
        if e in sdg and d in sdg:
            sdg[d] = sdg[e]
        t, l = f"decoder_embeddings.{m}.token_emb.weight", f"decoder_embeddings.{m}.to_logits.weight"
        if t in sdg:
            sdg[l] = sdg[t]
    batch = O.synthetic_mod7_batch(2, seed=c["batch_seed"])
    loss, _ = O.fourm_forward(sdg, O.PRESETS[gold["model"]], specs, batch, c["N"], c["M"], c["decoder_order"])
    loss.backward()
    for k, ref_norm in c["grads"]["norm"].items():
        g = sdg[k].grad
        assert g is not None, k
        assert abs(float(g.norm()) - ref_norm) <= 1e-4 * max(ref_norm, 1e-3), k
    for k, sl in c["grads"]["slices"].items():
        torch.testing.assert_close(sdg[k].grad.flatten()[:64], sl, rtol=1e-3, atol=1e-6)


def test_stable_keep_equals_argsort_trick():
    g = torch.Generator().manual_seed(0)
    for L in (7, 196, 2204, 3000):
        mask = torch.rand(4, L, generator=g) < 0.6
        ref = torch.argsort(mask + torch.arange(L)[None] * 1e-6, dim=1)        # fm.py:364-365
        assert torch.equal(O.stable_keep_indices(mask, L), ref)


def test_decoder_mask_semantics():
    # SURVEY.md v3
    dam = torch.tensor([[3, 0, 0, 1, 1, 0]], dtype=torch.int32)
    mod = torch.tensor([[7, 7, 7, 9, 9, 9]], dtype=torch.int16)
    allow = ~O.decoder_attention_mask(dam, mod)[0]
    assert allow[0].tolist() == [True, True, True, False, False, False]
    assert allow[3].tolist() == [False, False, False, True, False, False]
    assert allow[4].tolist() == [False, False, False, True, True, False]
    assert allow[5].tolist() == [False, False, False, True, True, False]


def test_fully_masked_row_is_uniform():
    q = torch.randn(1, 1, 2, 8); k = torch.randn(1, 1, 8, 8); v = torch.randn(1, 1, 8, 8)
    mask = torch.ones(1, 1, 1, 8, dtype=torch.bool)
    out = O._sdpa(q, k, v, mask, 1.0)
    torch.testing.assert_close(out[0, 0, 0], v[0, 0].mean(0))


def _vq_encode_case(tag, out):
    """The oracle's VQ.encode of a golden case on the fixture weights -> torch.save((quant, tokens, latents), out)."""
    torch.set_num_threads(1)
    c = H.load_golden("vq_golden.pt")["cases"][tag]
    kw = c["kw"]
    sd = {}
    for k, shape in c["shapes"].items():
        if k.endswith("pos_emb"):
            side = kw["image_size"] // 16
            sd[k] = V.sincos_2d_grid(side, side, shape[1])
        elif k.endswith("initted"):
            sd[k] = torch.ones(shape)
        elif k.endswith("cluster_size"):
            sd[k] = torch.zeros(shape)
        elif k.endswith("_codebook.embed") or k.endswith("embed_avg"):
            e = O.deterministic_tensor("quantize._codebook.embed", shape, 1.0)
            sd[k] = torch.nn.functional.normalize(e, dim=-1) if kw["norm_codes"] else e * 0.3
        else:
            sd[k] = O.deterministic_tensor(k, shape, 0.05 if len(shape) > 1 else 0.02)
        assert abs(float(sd[k].double().sum()) - c["weight_checksums"][k]) <= 1e-5 * max(1.0, abs(c["weight_checksums"][k])), k
    x = torch.randn(3, 3, 64, 64, generator=torch.Generator().manual_seed(5))
    torch.save(V.vq_encode(x, sd, kw["enc_type"], 16, kw["norm_codes"], kw["post_mlp"]), out)


@pytest.mark.parametrize("tag", ["vit_s_cos", "vit_s_l2"])
def test_vq_encode_matches_reference(tag, tmp_path):
    """Both sides run in fp32 under helpers.REPRODUCIBLE_CPU_ENV (the reference's: make_golden.py), so the comparison does not depend
    on the host's BLAS code path or thread count."""
    c = H.load_golden("vq_golden.pt")["cases"][tag]
    out = tmp_path / "vq_encode.pt"
    subprocess.run([sys.executable, "-c", f"from tests.test_oracle_golden import _vq_encode_case; _vq_encode_case({tag!r}, {str(out)!r})"],
                   cwd=H.ROOT, env={**os.environ, **H.REPRODUCIBLE_CPU_ENV, "PYTHONPATH": os.pathsep.join([H.ROOT, os.path.join(H.ROOT, "ml-4m_b200")])},
                   check=True)
    quant, tokens, lat = torch.load(out)
    torch.testing.assert_close(lat, c["latents"], rtol=1e-4, atol=1e-5)
    assert torch.equal(tokens, c["tokens"])
    torch.testing.assert_close(quant, c["quant"])


def test_scan_kats_torch_and_c():
    s = H.load_golden("vq_golden.pt")["scan"]
    z = s["z"]
    assert torch.equal(V.cosine_scan(z, s["cos_embed"]), s["cos_idx"])
    assert torch.equal(V.euclidean_scan(z, s["l2_embed"]), s["l2_idx"])
    lib = H.load_c_oracle()
    zn = torch.nn.functional.normalize(z, dim=-1).contiguous()
    en = torch.nn.functional.normalize(s["cos_embed"], dim=-1).contiguous()
    idx = torch.empty(z.shape[0], dtype=torch.int64)
    lib.vq_cosine_argmax_oracle(zn.data_ptr(), en.data_ptr(), z.shape[0], en.shape[0], 32, idx.data_ptr(), None)
    sc = V.scan_scores(z, s["cos_embed"], True)
    bad = idx != s["cos_idx"]
    # summation order differs from the BLAS kernel: any mismatch must be a genuine fp32 near-tie
    assert float((sc.gather(1, idx[:, None]) - sc.gather(1, s["cos_idx"][:, None])).abs()[bad].max() if bad.any() else 0.0) <= 1e-6
    assert bad.sum() <= 2
    e2 = s["l2_embed"].contiguous(); zc = z.contiguous()
    lib.vq_euclid_argmax_oracle(zc.data_ptr(), e2.data_ptr(), z.shape[0], e2.shape[0], 32, idx.data_ptr(), None)
    bad = idx != s["l2_idx"]
    sc = V.scan_scores(z, s["l2_embed"], False)
    assert float((sc.gather(1, idx[:, None]) - sc.gather(1, s["l2_idx"][:, None])).abs()[bad].max() if bad.any() else 0.0) <= 1e-4
    assert bad.sum() <= 2


# ---- qk_norm presets (a13: NormAttention / NormCrossAttention, fm_utils.py:222-307) ---------------------------------------------
@pytest.fixture(scope="module")
def tiny_qknorm():
    gold = H.load_golden("fourm_tiny_qknorm_golden.pt")
    specs = O.mod7_specs()
    sd = H.fill_fourm_buffers(H.golden_state_dict(gold), specs, 384)
    for k, c in gold["weight_checksums"].items():
        assert abs(float(sd[k].double().sum()) - c) <= 1e-6 * max(1.0, abs(c)), f"fixture weight drift in {k}"
    assert "encoder.0.attn.q_norm.weight" in sd and "decoder.0.cross_attn.k_norm.weight" in sd
    return gold, specs, sd


@pytest.mark.parametrize("tag", ["fp32_128", "bf16_128"])
def test_fourm_qknorm_forward_matches_reference(tiny_qknorm, tag):
    gold, specs, sd = tiny_qknorm
    c = gold["cases"][tag]
    batch = O.synthetic_mod7_batch(2, seed=c["batch_seed"], extra_valid=c["extra_valid"])
    cfg = O.PRESETS[gold["model"]]
    with torch.autocast("cpu", dtype=torch.bfloat16, enabled=c["amp"]):
        loss, mod_loss = O.fourm_forward(sd, cfg, specs, batch, c["N"], c["M"], c["decoder_order"], "mod")
        logits = O.fourm_forward(sd, cfg, specs, batch, c["N"], c["M"], c["decoder_order"], return_logits=True)
    tol = 2e-3 if c["amp"] else 1e-5
    assert abs(float(loss) - float(c["loss"])) <= tol
    for m, v in c["mod_loss"].items():
        assert abs(float(mod_loss[m]) - float(v)) <= tol, m
    for m, v in c["logits_slices"].items():
        torch.testing.assert_close(logits[m][:, :4, :32].float(), v, rtol=tol * 10, atol=tol * 10)


def test_fourm_qknorm_backward_matches_reference(tiny_qknorm):
    gold, specs, sd = tiny_qknorm
    c = gold["cases"]["fp32_128"]
    names = set(gold["param_names"])
    sdg = {k: (v.clone().requires_grad_(True) if k in names else v) for k, v in sd.items()}
    for m in specs:
        e, d = f"encoder_embeddings.{m}.mod_emb", f"decoder_embeddings.{m}.mod_emb"
        if e in sdg and d in sdg:
            sdg[d] = sdg[e]
        t, l = f"decoder_embeddings.{m}.token_emb.weight", f"decoder_embeddings.{m}.to_logits.weight"
        if t in sdg:
            sdg[l] = sdg[t]
    batch = O.synthetic_mod7_batch(2, seed=c["batch_seed"])
    loss, _ = O.fourm_forward(sdg, O.PRESETS[gold["model"]], specs, batch, c["N"], c["M"], c["decoder_order"])
    loss.backward()
    for k in ("encoder.0.attn.q_norm.weight", "encoder.3.attn.k_norm.weight", "decoder.0.cross_attn.q_norm.weight",
              "decoder.2.self_attn.q_norm.weight", "encoder.0.attn.qkv.weight"):
        ref_norm = c["grads"]["norm"][k]
        assert abs(float(sdg[k].grad.norm()) - ref_norm) <= 1e-4 * max(ref_norm, 1e-3), k
        torch.testing.assert_close(sdg[k].grad.flatten()[:64], c["grads"]["slices"][k], rtol=1e-3, atol=1e-6)


# ---- VQ-VAE training side (a25): codebook EMA update + one VQVAE training step -------------------------------------------------
def test_codebook_ema_updates_match_reference():
    gold = H.load_golden("vq_train_golden.pt")
    c = gold["cosine"]
    embed, cs = c["embed0"].clone(), torch.zeros(512)
    for z, st in zip(c["z"], c["steps"]):
        q, idx, embed, cs = V.cosine_codebook_train_step(z, embed, cs, 0.9)
        assert torch.equal(idx, st["idx"])
        torch.testing.assert_close(q.double().sum(-1), st["quant_sum"], rtol=1e-6, atol=1e-6)
        torch.testing.assert_close(embed, st["embed"], rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(cs, st["cluster_size"], rtol=1e-6, atol=1e-6)
    e = gold["euclid"]
    embed, avg, cs = e["embed0"].clone(), e["embed0"].clone(), torch.zeros(300)
    for z, st in zip(c["z"], e["steps"]):
        q, idx, embed, avg, cs = V.euclid_codebook_train_step(z, embed, avg, cs, 0.8)
        assert torch.equal(idx, st["idx"])
        torch.testing.assert_close(embed, st["embed"], rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(avg, st["embed_avg"], rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(cs, st["cluster_size"], rtol=1e-6, atol=1e-6)


def _vqvae_fixture():
    gold = H.load_golden("vq_train_golden.pt")["vqvae"]
    sd = {}
    for k, shape in gold["shapes"].items():
        if k.endswith("pos_emb"):
            sd[k] = V.sincos_2d_grid(shape[2], shape[3], shape[1])
        elif k.endswith("initted"):
            sd[k] = torch.ones(shape)
        elif k.endswith("cluster_size"):
            sd[k] = torch.zeros(shape)
        elif k.endswith("_codebook.embed"):
            sd[k] = torch.nn.functional.normalize(O.deterministic_tensor("quantize._codebook.embed", shape, 1.0), dim=-1)
        else:
            sd[k] = O.deterministic_tensor(k, shape, 0.05 if len(shape) > 1 else 0.02)
    for k, c in gold["weight_checksums"].items():
        assert abs(float(sd[k].double().sum()) - c) <= 1e-5 * max(1.0, abs(c)), f"fixture weight drift in {k}"
    x = torch.randn(4, 3, 64, 64, generator=torch.Generator().manual_seed(7))
    return gold, sd, x


def test_vqvae_training_step_matches_reference():
    gold, sd, x = _vqvae_fixture()
    names = set(gold["param_names"])
    sdg = {k: (v.clone().requires_grad_(True) if k in names else v) for k, v in sd.items()}
    dec, code_loss, idx, new_embed, new_cs = V.vqvae_forward_train(x, sdg, gold["kw"])
    rec = torch.nn.functional.mse_loss(dec, x)
    (rec + code_loss.sum()).backward()
    assert abs(float(rec) - float(gold["rec_loss"])) <= 1e-4 * float(gold["rec_loss"])
    assert abs(float(code_loss) - float(gold["code_loss"])) <= 1e-4 * float(gold["code_loss"])
    torch.testing.assert_close(dec[:, :, :8, :8].detach(), gold["dec_slice"], rtol=1e-3, atol=1e-3)
    torch.testing.assert_close(new_embed.detach(), gold["embed_after"], rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(new_cs.detach(), gold["cluster_size_after"], rtol=1e-6, atol=1e-6)
    for k, ref in gold["grad_norm"].items():
        assert abs(float(sdg[k].grad.norm()) - ref) <= 2e-3 * max(ref, 1e-3), k
    for k, sl in gold["grad_slices"].items():
        torch.testing.assert_close(sdg[k].grad.flatten()[:64], sl, rtol=5e-3, atol=1e-4 * float(sl.abs().max()) + 1e-7)


# ---- a6: SequenceEmbEncoderEmbedding (T5-XXL features, 4M-21) ----------------------------------------------------------------
def _seqemb_case(tag):
    c = H.load_golden("seqemb_golden.pt")["cases"][tag]
    g = torch.Generator().manual_seed(41)                        # == make_golden_seqemb.inputs()
    feats = torch.randn(3, 77, 4096, generator=g)
    mask = torch.rand(3, 77, generator=g) < 0.35
    mask[0] = False
    mask[1, 5:] = True
    wx = torch.randn(3, 77, 384, generator=g)
    we = torch.randn(3, 77, 384, generator=g)
    sd = {k: (O.sincos_1d(512, 384) if k == "pos_emb" else O.deterministic_tensor("seqemb." + k, shape, 0.02)) for k, shape in c["shapes"].items()}
    return c, sd, feats, mask, wx, we


@pytest.mark.parametrize("tag", ["plain", "bottleneck"])
def test_sequence_feature_embedding_matches_reference(tag):
    c, sd, feats, mask, wx, we = _seqemb_case(tag)
    proj = [(sd["emb_proj.weight"], sd["emb_proj.bias"])] if tag == "plain" else \
        [(sd["emb_proj.0.weight"], sd["emb_proj.0.bias"]), (sd["emb_proj.1.weight"], sd["emb_proj.1.bias"])]
    x, emb = O.embed_sequence_features(feats, mask, proj, sd["pos_emb"], sd["mod_emb"])
    torch.testing.assert_close(x[:, :6, :48], c["x_slice"], rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(x.double().sum(-1), c["x_sum"], rtol=1e-4, atol=1e-3)
    assert torch.equal(emb[:, :6, :48], c["emb_slice"])
    assert torch.equal(emb.double().sum(-1), c["emb_sum"])
