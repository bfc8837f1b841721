"""Shared helpers for the tests (fixtures, deterministic weights, golden loading)."""
import ctypes
import os
import random

import torch

from oracle import fourm_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden")

# fp32 CPU results that do not depend on the host: MKL's reproducible code path, ATen and oneDNN kernels at the baseline ISA, one
# thread.  Deep fp32 networks otherwise differ by more than their tolerance between BLAS code paths and thread counts.  MKL reads
# these at start-up, so a computation that needs them runs in a subprocess with this environment.
REPRODUCIBLE_CPU_ENV = dict(MKL_CBWR="COMPATIBLE", ATEN_CPU_CAPABILITY="default", ONEDNN_MAX_CPU_ISA="SSE41", OMP_NUM_THREADS="1",
                            MKL_NUM_THREADS="1")


def load_golden(name):
    return torch.load(os.path.join(GOLDEN, name), weights_only=False)


def golden_state_dict(gold):
    """Rebuild the fixture weights from names+shapes and verify their checksums."""
    params = set(gold.get("param_names", []))
    sd = {}
    for k, shape in gold["shapes"].items():
        if k in params:
            sd[k] = O.deterministic_tensor(O.canonical_param_name(k, gold['shapes']), shape)
        elif k.endswith("pos_emb"):
            sd[k] = None    # filled by caller (sincos tables)
        else:
            sd[k] = torch.zeros(shape)
    return sd


def fill_fourm_buffers(sd, specs, dim):
    for name, s in specs.items():
        for side in ("encoder_embeddings", "decoder_embeddings"):
            k = f"{side}.{name}.pos_emb"
            if k in sd and sd[k] is None:
                if s["kind"] == "seq":
                    sd[k] = O.sincos_1d(512, dim)       # quirk: [1,512,D] (slice hits the batch dim)
                else:
                    side_len = s["image_size"] // s["patch_size"]
                    sd[k] = O.sincos_2d(side_len, side_len, dim)
    return sd


def decoder_order(seed, names):
    random.seed(seed)
    return random.sample(list(names), len(names))


def load_c_oracle():
    so = os.path.join(ROOT, "oracle", "_build", "libvq_argmax_oracle.so")
    if not os.path.exists(so):
        import subprocess
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")])
    lib = ctypes.CDLL(so)
    for fn in (lib.vq_cosine_argmax_oracle, lib.vq_euclid_argmax_oracle):
        fn.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64,
                       ctypes.c_void_p, ctypes.c_void_p]
        fn.restype = None
    return lib


class StubTextTokenizer:
    """Stand-in for the reference's WordPiece tokenizer (fourm/utils/tokenizer/trained/text_tokenizer_4m_wordpiece_30k.json, which
    cannot travel to the GPU box): only what the generation code touches -- the special-token ids the reference's helpers hard-code
    ([PAD] 0, [EOS] 3, [S_1] 5: generate.py:39, 119) and 100 sentinels."""

    def __init__(self):
        self.vocab = {"[PAD]": 0, "[UNK]": 1, "[SOS]": 2, "[EOS]": 3}
        for i in range(100):
            self.vocab[f"[S_{i}]"] = 4 + i

    def get_vocab(self):
        return dict(self.vocab)

    def token_to_id(self, tok):
        return self.vocab.get(tok)


GEN_TARGETS = ['tok_depth@224', 'tok_normal@224', 'caption']


def generation_case(modality_info, device="cpu", B=2, seed=3):
    """The sample + schedule of the generation parity fixture (tests/golden/make_golden_gen.py): RGB -> depth (MaskGIT, cosine, 4 steps,
    temperature 1, guided), -> normals (ROAR, 3 steps, temperature 0, guided), -> caption (autoregressive, temperature 0, guided)."""
    from fourm.models import generate as G
    g = torch.Generator().manual_seed(seed)
    sample = {'rgb@224': {'tensor': torch.randn(B, 3, 224, 224, generator=g).to(device)}}
    sample = G.init_full_input_modality(sample, modality_info, 'rgb@224', device)
    for mod, n in zip(GEN_TARGETS, (196, 196, 256)):
        sample = G.init_empty_target_modality(sample, modality_info, mod, B, n, device)
    schedule = G.build_chained_generation_schedules(
        cond_domains=['rgb@224'], target_domains=GEN_TARGETS, tokens_per_target=[196, 196, 256],
        autoregression_schemes=['maskgit', 'roar', 'autoregressive'], decoding_steps=[4, 3, None],
        token_decoding_schedules=['cosine', 'linear', None], temps=[1.0, 0.0, 0.0], temp_schedules=['constant', 'constant', 'constant'],
        cfg_scales=[2.0, 1.5, 2.0], cfg_schedules=['constant', 'constant', 'constant'], cfg_grow_conditioning=True, modality_info=modality_info)
    return sample, schedule
