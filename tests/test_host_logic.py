"""Host-side logic that needs no GPU: model registry / state_dict contract / parameter sharing of the overlay, the synthetic
wire-format batches, segment construction, the loud no-fallback behaviour, and the N>1 launch contract of bench.py
(world_size 2 under torchrun on CPU)."""
import json
import os
import subprocess
import sys

import pytest
import torch

from oracle import fourm_oracle as O
from tests import helpers as H

ROOT = H.ROOT


@pytest.fixture(scope="module")
def tiny_cpu():
    from b200fm.compat import build_mod7_embeddings, create_model
    enc, dec, info = build_mod7_embeddings()
    return create_model("fm_tiny_6e_6d_swiglu_nobias", encoder_embeddings=enc, decoder_embeddings=dec, modality_info=info)


def test_registry_has_the_13_reference_names():
    import fourm.models.fm as fm
    from b200fm import compat
    names = ['fm_tiny_6e_6d_gelu', 'fm_small_8e_8d_gelu', 'fm_base_12e_12d_gelu', 'fm_large_24e_24d_gelu', 'fm_xlarge_24e_24d_gelu',
             'fm_tiny_6e_6d_swiglu_nobias', 'fm_small_8e_8d_swiglu_nobias', 'fm_base_12e_12d_swiglu_nobias',
             'fm_large_24e_24d_swiglu_nobias', 'fm_xlarge_24e_24d_swiglu_nobias', 'fm_base_12e_12d_swiglu_qknorm_nobias',
             'fm_large_24e_24d_swiglu_qknorm_nobias', 'fm_xlarge_24e_24d_swiglu_qknorm_nobias']      # reference fm.py:33-50
    assert sorted(fm.__all__) == sorted(names)
    for n in names:
        assert callable(getattr(fm, n)) and n in compat._local_entrypoints


def test_state_dict_matches_reference_golden_shapes(tiny_cpu):
    gold = H.load_golden("fourm_tiny_golden.pt")
    sd = tiny_cpu.state_dict()
    assert list(sd.keys()) == list(gold["shapes"].keys())
    assert all(tuple(v.shape) == gold["shapes"][k] and v.dtype == torch.float32 for k, v in sd.items())
    assert [k for k, _ in tiny_cpu.named_parameters(remove_duplicate=False)] == gold["param_names"]
    # sincos buffers are bit-identical to the reference's tables (same construction)
    assert torch.equal(sd["encoder_embeddings.tok_rgb@224.pos_emb"], O.sincos_2d(14, 14, 384))
    assert torch.equal(sd["encoder_embeddings.caption.pos_emb"], O.sincos_1d(512, 384))


def test_parameter_sharing_and_weight_decay_groups(tiny_cpu):
    from b200fm.optim import param_groups_like_reference
    m = tiny_cpu
    for mod in ("caption", "tok_rgb@224"):
        assert m.decoder_embeddings[mod].mod_emb is m.encoder_embeddings[mod].mod_emb
        assert m.decoder_embeddings[mod].to_logits.weight is m.decoder_embeddings[mod].token_emb.weight
    groups = param_groups_like_reference(m, 0.05)
    decay, no_decay = groups
    ids_no = {id(p) for p in no_decay["params"]}
    assert id(m.encoder[0].norm1.weight) in ids_no and id(m.decoder_proj_context.bias) in ids_no
    assert id(m.encoder[0].attn.qkv.weight) not in ids_no and decay["weight_decay"] == 0.05
    n = sum(p.numel() for g in groups for p in g["params"])
    assert n == sum(p.numel() for p in m.parameters())


def test_forward_refuses_cpu_tensors(tiny_cpu):
    from b200fm import lib
    batch = O.synthetic_mod7_batch(1)
    with pytest.raises(lib.B200FMError):
        tiny_cpu(batch, num_encoder_tokens=128, num_decoder_tokens=128)


def test_invalid_loss_type_raises_like_reference(tiny_cpu):
    with pytest.raises(ValueError, match="Invalid loss type"):
        tiny_cpu(O.synthetic_mod7_batch(1), 128, 128, loss_type="nope")


def test_synthetic_batches_have_exact_budgets():
    from b200fm.synthetic import budgets_for, mod7_batch
    for n_tok in (128, 256):
        a, b, c, d = budgets_for(n_tok)
        batch = mod7_batch(3, a, b, c, d, seed=7)
        n_in = sum((~v["input_mask"]).sum(1) for v in batch.values())
        n_tgt = 0
        for name, v in batch.items():
            if name == "rgb@224":
                continue
            tm = v["target_mask"]
            if v["tensor"].dim() == 2 and v["tensor"].dtype == torch.int32:      # sequences lose one row to the shift
                tm = tm[:, 1:] | tm[:, :-1]
            n_tgt = n_tgt + (~tm).sum(1)
        assert n_in.tolist() == [n_tok] * 3 and n_tgt.tolist() == [n_tok] * 3
        assert batch["caption"]["tensor"].shape == (3, 514) and batch["tok_rgb@224"]["tensor"].dtype == torch.int64


def test_segment_struct_layout_matches_header():
    import ctypes
    import re
    from b200fm import lib
    text = open(os.path.join(ROOT, "include", "b200fm.h")).read()
    body = text[text.index("typedef struct b200fm_segment {"):text.index("} b200fm_segment;")]
    fields = re.findall(r"\b(\w+);\s*(?:/\*|$)", body, flags=re.M)
    assert fields == [f[0] for f in lib.Segment._fields_]
    assert ctypes.sizeof(lib.Segment) == 10 * 8 + 8 + 6 * 4 + 8
    assert int(re.search(r"#define B200FM_MAX_SEGMENTS (\d+)", text).group(1)) == lib.MAX_SEGMENTS


def test_bench_reference_arm_contract_under_torchrun_world2():
    """`bench.py --impl reference` launched like the driver does for N=2 (gloo-free: rank 0 runs the CPU oracle, rank 1 exits 0)."""
    env = dict(os.environ, OMP_NUM_THREADS="4")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29731", os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["metric"] == "tokens_per_sec" and j["value"] > 0 and j["n_gpus"] == 2
    assert j["cpu_baseline"]["kind"] in ("port", "reference") and j["e2e"]["h2d_bytes_per_step"] == 0


def test_device_prefetcher_order_cpu_fallback_refused():
    """DevicePrefetcher is CUDA-only plumbing: constructing it without a GPU must fail loudly (no silent CPU path)."""
    import pytest
    import torch
    from b200fm.data import DevicePrefetcher
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    with pytest.raises(Exception):
        DevicePrefetcher([], "cuda")


def _sample_worker(rank, world, port, q):
    import os
    import sys
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "ml-4m_b200"))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from fourm.vq.quantizers.quantize_lucid import CosineSimCodebook
    cb = CosineSimCodebook(dim=8, codebook_size=16, use_ddp=True)
    torch.manual_seed(100 + rank)
    samples = torch.nn.functional.normalize(torch.randn(5 + 7 * rank, 8), dim=-1) + 10.0 * rank     # rank is recognisable
    out = cb._sample(samples, 9)
    allsamp = [torch.empty(5 + 7 * r, 8) for r in range(world)]
    for r in range(world):
        t = samples if r == rank else allsamp[r]
        dist.broadcast(t, src=r)
        allsamp[r] = t
    q.put((rank, out, torch.cat(allsamp)))
    dist.destroy_process_group()


def test_dead_code_resampling_is_identical_on_all_ranks_gloo():
    """sync_codebook dead-code re-seeding (quantize_lucid.py:100-113): every rank must end up with the SAME replacement vectors,
    drawn from the union of the ranks' latents (world_size 2, gloo, CPU tensors: pure host logic, no kernel involved)."""
    import torch
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29650
    procs = [ctx.Process(target=_sample_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=120) for _ in procs], key=lambda t: t[0])
    for p in procs:
        p.join(60)
    (_, o0, pool), (_, o1, _) = res
    assert o0.shape == (9, 8) and torch.equal(o0, o1)
    d = (o0[:, None, :] - pool[None]).abs().sum(-1).min(dim=1).values
    assert float(d.max()) == 0.0                                  # every row is one of the pooled latents


def test_param_groups_match_reference_optim_factory():
    """a18: the decay / no-decay split of `b200fm.optim.param_groups_like_reference` equals what the unmodified reference's
    `get_parameter_groups` (optim_factory.py:111-168) produced for the same model (fixture: tests/golden/make_golden_param_groups.py)."""
    import json
    import os
    from b200fm.compat import build_mod7_embeddings, create_model
    from b200fm.optim import param_groups_like_reference
    gold = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "param_groups_golden.json")))
    for tag, kw in {"tiny": {}, "tiny_qknorm": dict(qk_norm=True)}.items():
        enc, dec, info = build_mod7_embeddings()
        model = create_model("fm_tiny_6e_6d_swiglu_nobias", encoder_embeddings=enc, decoder_embeddings=dec, modality_info=info, **kw)
        names = {id(p): n for n, p in model.named_parameters()}
        groups = param_groups_like_reference(model, 0.05)
        got = {("decay" if g["weight_decay"] > 0 else "no_decay"): sorted(names[id(p)] for p in g["params"]) for g in groups}
        assert got["decay"] == gold[tag]["decay"], tag
        assert got["no_decay"] == gold[tag]["no_decay"], tag
        assert sorted(model.no_weight_decay()) == gold[tag]["skip_list"]


def test_all_13_presets_match_reference_state_dict_contract():
    """Every registered model name builds the same state_dict (keys, order, shapes, dtypes: compared as a digest) and the same number of
    parameters as the unmodified reference constructor (fixture: tests/golden/make_golden_presets.py; initialisation patched out so the
    2.8 B parameter XL presets build in seconds from untouched memory)."""
    import hashlib
    import importlib.util
    import json
    import os
    here = os.path.dirname(os.path.abspath(__file__))
    spec = importlib.util.spec_from_file_location("_mgp", os.path.join(here, "golden", "make_golden_presets.py"))
    mgp = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mgp)
    from b200fm.compat import build_mod7_embeddings, create_model
    gold = json.load(open(os.path.join(here, "golden", "presets_golden.json")))
    assert len(gold) == 13
    for name, ref in gold.items():
        with mgp.no_init():
            enc, dec, info = build_mod7_embeddings()
            model = create_model(name, encoder_embeddings=enc, decoder_embeddings=dec, modality_info=info)
        got = mgp.digest(model)
        assert got == ref, (name, got, ref)
        del model


def test_tokenizer_constructors_match_reference_state_dict_contract():
    """`fourm.vq.VQ` / `VQVAE` of the overlay build the reference's state_dict (digest of keys, order, shapes, dtypes) for the ViT-S/B/L
    encoders / decoders, patch 8 / 16, cosine and Euclidean codebooks, class-label inputs (fixture: make_golden_vq_presets.py)."""
    import importlib.util
    import json
    import os
    here = os.path.dirname(os.path.abspath(__file__))

    def load(name):
        spec = importlib.util.spec_from_file_location("_" + name, os.path.join(here, "golden", name + ".py"))
        mod = importlib.util.module_from_spec(spec)
        sys.path.insert(0, os.path.join(here, "golden"))
        try:
            spec.loader.exec_module(mod)
        finally:
            sys.path.remove(os.path.join(here, "golden"))
        return mod
    cases = load("make_golden_vq_presets")
    mgp = load("make_golden_presets")
    import fourm.vq as vq
    gold = json.load(open(os.path.join(here, "golden", "vq_presets_golden.json")))
    for tag, (cls, kw) in cases.CASES.items():
        with mgp.no_init():
            m = getattr(vq, cls)(sync_codebook=False, **kw)
        assert mgp.digest(m) == gold[tag], (tag, mgp.digest(m), gold[tag])


# the parts of the reference the overlay talks to, restated minimally for the stand-in tree: the timm-style model registry and the
# `create_model` that looks names up in it, and MODALITY_INFO rebuilt from the recorded embedding factories
_STANDIN = {
    "fourm/utils/timm/registry.py": '''
_model_entrypoints = {{}}


def register_model(fn):
    _model_entrypoints[fn.__name__] = fn
    return fn


def model_entrypoint(model_name):
    return _model_entrypoints[model_name]
''',
    "fourm/utils/__init__.py": '''
from .timm.registry import model_entrypoint, register_model


def create_model(model_name, **kwargs):
    return model_entrypoint(model_name)(**kwargs)
''',
    "fourm/data/modality_info.py": '''
import importlib
import json
from functools import partial

with open({golden!r}) as f:
    _entries = json.load(f)["modality_info"]


def _factory(spec):
    return None if spec is None else partial(getattr(importlib.import_module(spec["module"]), spec["name"]), **spec["kwargs"])


MODALITY_INFO = {{m: {{k: _factory(v) if k.endswith("_embedding") else v for k, v in e.items()}} for m, e in _entries.items()}}
''',
}


def test_overlay_resolves_ahead_of_reference_tree(tmp_path):
    """INTEGRATION.md level 1: with `ml-4m_b200/` ahead of the reference on sys.path, exactly the hot-path modules resolve to the overlay
    (fourm.models.fm / fm_utils / *_embeddings / generate, fourm.vq) while fourm.utils and fourm.data stay the reference's; the
    reference's registry-based `create_model` + `MODALITY_INFO` factories then build the overlay classes and `GenerationSampler` wraps
    them.  The reference is a stand-in tree with the unmodified reference's package layout (every module empty except the registry,
    `create_model` and MODALITY_INFO); the layout, the resolution and the built class were recorded from the unmodified reference
    (fixture: tests/golden/make_golden_overlay.py)."""
    golden_path = os.path.join(ROOT, "tests", "golden", "overlay_golden.json")
    gold = json.load(open(golden_path))
    ref = tmp_path / "reference"
    for rel in gold["layout"]:
        (ref / rel).parent.mkdir(parents=True, exist_ok=True)
        (ref / rel).write_text(_STANDIN.get(rel, "").format(golden=golden_path))
    assert set(_STANDIN) <= set(gold["layout"])
    code = r'''
import json, sys
ov, ref = {ov!r}, {ref!r}
sys.path[:0] = [ov, ref]
gold = json.load(open({golden!r}))
import importlib
where = lambda f: "overlay" if f.startswith(ov + "/") else "reference" if f.startswith(ref + "/") else f
assert {{m: where(importlib.import_module(m).__file__) for m in gold["resolved"]}} == gold["resolved"]
import fourm.utils as utils, fourm.models.generate as gen
from fourm.data.modality_info import MODALITY_INFO
mods = list(gold["modality_info"])
mk = lambda m, side: MODALITY_INFO[m][side]() if MODALITY_INFO[m]["type"] != "img" else MODALITY_INFO[m][side](patch_size=16, image_size=224)
enc = {{m: mk(m, "encoder_embedding") for m in mods}}
dec = {{m: mk(m, "decoder_embedding") for m in mods[1:]}}
model = utils.create_model("fm_tiny_6e_6d_swiglu_nobias", encoder_embeddings=enc, decoder_embeddings=dec, modality_info={{m: MODALITY_INFO[m] for m in mods}})
assert [type(model).__module__, type(model).__name__] == gold["model_class"]
assert where(sys.modules[type(model).__module__].__file__) == "overlay"
assert hasattr(model.encoder[0], "forward_pending")            # the overlay's block, not the reference's
gen.GenerationSampler(model)
print("OK")
'''.format(ov=os.path.join(ROOT, "ml-4m_b200"), ref=str(ref), golden=golden_path)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=tmp_path,
                         env={**os.environ, "PYTHONPATH": ""})
    assert out.returncode == 0 and "OK" in out.stdout, out.stderr[-2000:]


def test_hub_wrapper_fm_config_matches_reference():
    """`fourm.models.fm.FM(config)` (the class Demo4MSampler / from_pretrained instantiate, fm.py:783-831) builds the reference's
    state_dict for a 4M-7-style config (untied decoder heads) and a small GELU / bias config (fixture: make_golden_fm_config.py)."""
    import importlib.util
    import json
    here = os.path.dirname(os.path.abspath(__file__))
    sys.path.insert(0, os.path.join(here, "golden"))
    try:
        spec = importlib.util.spec_from_file_location("_mgfc", os.path.join(here, "golden", "make_golden_fm_config.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        sys.path.remove(os.path.join(here, "golden"))
    from fourm.models.fm import FM
    gold = json.load(open(os.path.join(here, "golden", "fm_config_golden.json")))
    for tag, cfg in mod.CONFIGS.items():
        with mod.MGP.no_init():
            m = FM(cfg)
        assert mod.MGP.digest(m) == gold[tag], (tag, mod.MGP.digest(m), gold[tag])


def test_model_ema_rule_matches_reference_golden():
    """The EMA rule the GPU kernel implements -- decay * ema + (1 - decay) * model, each product and the sum rounded to fp32, 1 - decay
    formed in double -- replayed with torch on the CPU reproduces the UNMODIFIED reference's ModelEmaV2 (tests/golden/ema_golden.pt) bit
    for bit; and FusedModelEma refuses the configurations it does not implement instead of silently averaging elsewhere."""
    import copy
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import make_golden_ema as G
    import torch
    gold = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ema_golden.pt"), weights_only=False)
    model = G.build_model()
    ema = copy.deepcopy(model).eval()
    decay = gold["decay"]
    for step in range(3):
        with torch.no_grad():
            for p, d in zip(model.parameters(), G.perturbations(model, step)):
                p.add_(d)
            model[1].running_mean.add_(0.5)
            model[1].num_batches_tracked.add_(1)
            for e, m in zip(ema.state_dict().values(), model.state_dict().values()):
                if e.dtype == torch.float32:
                    e.copy_(torch.tensor(decay, dtype=torch.float32) * e + torch.tensor(1. - decay, dtype=torch.float32) * m)
                else:
                    e.copy_(decay * e + (1. - decay) * m)
        for k, v in ema.state_dict().items():
            assert torch.equal(v, gold["states"][step][k]), (step, k)
    from b200fm.optim import FusedModelEma
    import pytest as _pt
    with _pt.raises(NotImplementedError):
        FusedModelEma(model, device="cpu")
    with _pt.raises(NotImplementedError):
        FusedModelEma(model, resume="ckpt.pth")
