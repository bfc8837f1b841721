"""Generate the committed golden fixtures by running the UNMODIFIED reference (apple/ml-4m @ /root/reference).

Run in the authoring container only:   python tests/golden/make_golden.py
Writes tests/golden/{fourm_tiny_golden,static_golden,vq_golden}.pt (small).
Weights are not stored: they are regenerated from `oracle.fourm_oracle.deterministic_tensor(name, shape)`
and a checksum of every tensor is stored so a torch RNG change would be detected.  Inputs are regenerated
from `oracle.fourm_oracle.synthetic_mod7_batch` (seeded).  The torch version is recorded in every file.
"""
import os
import random
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)

import ref_import  # noqa: E402
from oracle import fourm_oracle as O  # noqa: E402


def det_state_dict(model):
    """Deterministic weights for every parameter; constant buffers (sincos pos_emb, the zero `bias`
    buffers of bias-free LayerNorms) keep the values the reference constructed."""
    params = dict(model.named_parameters(remove_duplicate=False))
    full = model.state_dict()
    sd = {}
    for k, v in full.items():
        if k in params:
            sd[k] = O.deterministic_tensor(O.canonical_param_name(k, full), v.shape).to(v.dtype)
        else:
            sd[k] = v.clone()
    return sd


def build_reference_fourm(model_name, specs, MODALITY_INFO, **kw):
    from fourm.utils import create_model
    enc, dec = {}, {}
    for name in specs:
        info = MODALITY_INFO[name]
        is_img = info["type"] == "img"
        if info.get("encoder_embedding") is not None:
            enc[name] = info["encoder_embedding"](patch_size=16, image_size=224) if is_img else info["encoder_embedding"]()
        if info.get("decoder_embedding") is not None:
            dec[name] = info["decoder_embedding"](patch_size=16, image_size=224) if is_img else info["decoder_embedding"]()
    return create_model(model_name, encoder_embeddings=enc, decoder_embeddings=dec,
                        modality_info={m: MODALITY_INFO[m] for m in specs}, **kw)


def clone_batch(b):
    return {m: {k: v.clone() for k, v in d.items()} for m, d in b.items()}


def run_fourm_case(model, batch, N, M, seed, amp):
    def ctx():
        return torch.autocast("cpu", dtype=torch.bfloat16, enabled=amp)
    random.seed(seed)
    model.zero_grad(set_to_none=True)
    with ctx():
        loss, mod_loss = model(clone_batch(batch), num_encoder_tokens=N, num_decoder_tokens=M, loss_type="mod")
    loss.backward()
    grads = {k: p.grad.detach().clone() for k, p in model.named_parameters() if p.grad is not None}
    random.seed(seed)
    with torch.no_grad(), ctx():
        logits = model(clone_batch(batch), num_encoder_tokens=N, num_decoder_tokens=M, return_logits=True)
    random.seed(seed)
    with torch.no_grad(), ctx():
        tl, _ = model(clone_batch(batch), num_encoder_tokens=N, num_decoder_tokens=M, loss_type="token")
    return loss.detach(), {k: v.detach().reshape(()) for k, v in mod_loss.items()}, grads, logits, tl.detach()


def grad_summary(grads, keys):
    return {"norm": {k: g.float().norm().item() for k, g in grads.items()},
            "slices": {k: grads[k].flatten()[:64].clone() for k in keys if k in grads}}


SLICE_KEYS = ["mask_token", "encoder.0.attn.qkv.weight", "encoder.5.mlp.fc2.weight", "decoder.0.cross_attn.kv.weight",
              "decoder.5.mlp.fc1.weight", "decoder_proj_context.weight", "decoder_proj_context.bias",
              "encoder_embeddings.rgb@224.proj.weight", "encoder_embeddings.caption.mod_emb",
              "encoder_norm.weight", "decoder.3.query_norm.weight"]

FOURM_CASES = {   # tag: (amp, N, M, python-random seed, batch seed, extra valid targets per tok_img modality)
    "fp32_128": (False, 128, 128, 0, 1234, 0),
    "bf16_128": (True, 128, 128, 0, 1234, 0),
    "fp32_trunc": (False, 96, 100, 3, 77, 6),     # more valid tokens than budget: truncation depends on shuffle
    "fp32_pad": (False, 160, 150, 5, 99, 0),      # fewer valid tokens than budget: padded rows
}


def main():
    fm, fm_utils, MODALITY_INFO = ref_import.import_reference_models()
    torch.manual_seed(0)
    specs = O.mod7_specs()
    meta = dict(torch=torch.__version__, reference_commit="cda590f")

    # ---- 4M-Tiny mod7 (BASELINE.json configs[0]), B=2 ----
    model = build_reference_fourm("fm_tiny_6e_6d_swiglu_nobias", specs, MODALITY_INFO)
    sd = det_state_dict(model)
    model.load_state_dict(sd)
    gold = dict(meta=meta, model="fm_tiny_6e_6d_swiglu_nobias",
                weight_checksums={k: float(v.double().sum()) for k, v in sd.items()},
                shapes={k: tuple(v.shape) for k, v in sd.items()},
                param_names=[k for k, _ in model.named_parameters(remove_duplicate=False)], cases={})
    for tag, (amp, N, M, seed, bseed, extra) in FOURM_CASES.items():
        b = O.synthetic_mod7_batch(2, seed=bseed, extra_valid=extra)
        loss, mod_loss, grads, logits, tl = run_fourm_case(model, b, N, M, seed, amp)
        random.seed(seed)
        dec_names = [m for m in b if m in model.decoder_embeddings]
        order = random.sample(dec_names, len(dec_names))
        random.seed(seed)
        with torch.no_grad():
            bb = clone_batch(b)
            enc_d = {m: model.encoder_embeddings[m](d) for m, d in bb.items() if m in model.encoder_embeddings}
            et, ee, em, emod = model.forward_mask_encoder(enc_d, N)
            dec_d = {m: model.decoder_embeddings[m].forward_embed(d) for m, d in bb.items() if m in model.decoder_embeddings}
            dt, de, dm, tgt, damask, dmod = model.forward_mask_decoder(dec_d, M)
        gold["cases"][tag] = dict(
            amp=amp, N=N, M=M, py_seed=seed, batch_seed=bseed, extra_valid=extra, decoder_order=order,
            loss=loss, mod_loss=mod_loss, token_loss=tl, grads=grad_summary(grads, SLICE_KEYS),
            logits_slices={m: v[:, :4, :32].float().clone() for m, v in logits.items()},
            logits_norm={m: v.float().norm().item() for m, v in logits.items()},
            enc_mask=em.clone(), enc_mod=emod.clone(), dec_mask=dm.clone(), dec_mod=dmod.clone(), target_ids=tgt.clone(),
            dec_attn_mask=damask.clone(), enc_x0_sum=(et + ee).double().sum(-1), dec_y0_sum=(dt + de).double().sum(-1))
        print(tag, float(loss), {k: round(float(v), 5) for k, v in mod_loss.items()}, "order", order)
    torch.save(gold, os.path.join(HERE, "fourm_tiny_golden.pt"))

    # ---- static known answers ----
    static = dict(meta=meta,
                  mod_ids={m: MODALITY_INFO[m]["id"] for m in specs},
                  sincos1d_8x16=fm_utils.build_1d_sincos_posemb(8, 16),
                  sincos2d_3x5x8=fm_utils.build_2d_sincos_posemb(3, 5, 8),
                  sincos2d_14x14x384_sum=fm_utils.build_2d_sincos_posemb(14, 14, 384).double().sum(-1))
    torch.save(static, os.path.join(HERE, "static_golden.pt"))

    # ---- VQ tokenizer forward (a20-a24): in a subprocess under REPRODUCIBLE_CPU_ENV, like the test that compares against it ----
    import subprocess
    import tempfile
    from tests.helpers import REPRODUCIBLE_CPU_ENV
    with tempfile.TemporaryDirectory() as tmp:
        subprocess.run([sys.executable, os.path.abspath(__file__), "vq_encode_cases", os.path.join(tmp, "cases.pt")], check=True,
                       env={**os.environ, **REPRODUCIBLE_CPU_ENV})
        vgold = dict(meta=meta, cases=torch.load(os.path.join(tmp, "cases.pt"), weights_only=False))
    import fourm.vq as vq  # noqa: F401
    # stand-alone codebook scan KATs (a23/a24) straight through the reference codebook classes
    from fourm.vq.quantizers.quantize_lucid import CosineSimCodebook, EuclideanCodebook
    g = torch.Generator().manual_seed(11)
    z = torch.randn(1, 777, 32, generator=g)
    cb = CosineSimCodebook(dim=32, codebook_size=2048).eval()
    cb.embed.copy_(torch.nn.functional.normalize(torch.randn(2048, 32, generator=g), dim=-1))
    eb = EuclideanCodebook(dim=32, codebook_size=1000).eval()
    eb.embed.copy_(torch.randn(1000, 32, generator=g))
    with torch.no_grad():
        qc, ic = cb(z)
        qe, ie = eb(z)
    vgold["scan"] = dict(z=z[0].clone(), cos_embed=cb.embed.clone(), cos_idx=ic[0].clone(), cos_quant=qc[0].clone(),
                         l2_embed=eb.embed.clone(), l2_idx=ie[0].clone(), l2_quant=qe[0].clone())
    torch.save(vgold, os.path.join(HERE, "vq_golden.pt"))
    for f in ("fourm_tiny_golden.pt", "static_golden.pt", "vq_golden.pt"):
        print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, "KiB")


def vq_encode_cases():
    """VQ.encode of the reference tokenizer on deterministic weights, for the two tokenizer cases of vq_golden.pt."""
    torch.set_num_threads(1)
    ref_import.install()
    import fourm.vq as vq
    cases = {}
    for tag, kw in {
        "vit_s_cos": dict(enc_type="vit_s_enc", image_size=64, codebook_size=1024, latent_dim=32, norm_codes=True, post_mlp=True),
        "vit_s_l2": dict(enc_type="vit_s_enc", image_size=64, codebook_size=512, latent_dim=32, norm_codes=False, post_mlp=False),
    }.items():
        m = vq.VQ(patch_size=16, sync_codebook=False, **kw).eval()
        vsd = {}
        for k, v in m.state_dict().items():
            if k.endswith("pos_emb") or k.endswith("initted") or k.endswith("cluster_size"):
                vsd[k] = v.clone()
            elif k.endswith("_codebook.embed") or k.endswith("embed_avg"):
                e = O.deterministic_tensor("quantize._codebook.embed", v.shape, 1.0)
                vsd[k] = torch.nn.functional.normalize(e, dim=-1) if kw["norm_codes"] else e * 0.3
            else:
                vsd[k] = O.deterministic_tensor(k, v.shape, 0.05 if v.ndim > 1 else 0.02)
        m.load_state_dict(vsd)
        g = torch.Generator().manual_seed(5)
        x = torch.randn(3, 3, 64, 64, generator=g)
        with torch.no_grad():
            quant, code_loss, tokens = m.encode(x)
            h = m.quant_proj(m.encoder(x))
        cases[tag] = dict(kw=kw, shapes={k: tuple(v.shape) for k, v in vsd.items()},
                          weight_checksums={k: float(v.double().sum()) for k, v in vsd.items()},
                          tokens=tokens.clone(), latents=h.clone(), quant=quant.clone())
        print(tag, tokens.flatten()[:8].tolist())
    return cases


if __name__ == "__main__":
    if sys.argv[1:2] == ["vq_encode_cases"]:
        torch.save(vq_encode_cases(), sys.argv[2])
    else:
        main()
