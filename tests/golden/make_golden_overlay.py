"""Golden fixture for the overlay import test (INTEGRATION.md level 1): the UNMODIFIED reference imported with `ml-4m_b200/`
ahead of it on sys.path, recorded as data so that tests/test_host_logic.py can rebuild a stand-in of the reference tree:
  * layout:        every .py file of the reference's `fourm` package (which directories are packages, which are namespaces);
  * resolved:      which tree each hot-path / glue module resolved to ("overlay" or "reference");
  * modality_info: the MODALITY_INFO entries the test uses, with each embedding factory as (module, class, keywords);
  * model_class:   module and class of what the reference's `fourm.utils.create_model` built.

Run in the authoring container only:   python tests/golden/make_golden_overlay.py   -> tests/golden/overlay_golden.json
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OVERLAY = os.path.join(ROOT, "ml-4m_b200")
sys.path.insert(0, HERE)

import ref_import  # noqa: E402

MODULES = ["fourm.models.fm", "fourm.models.fm_utils", "fourm.models.encoder_embeddings", "fourm.models.decoder_embeddings",
           "fourm.models.generate", "fourm.vq", "fourm.utils", "fourm.data.modality_info"]
MODS = ["rgb@224", "caption", "tok_depth@224"]


def main():
    ref = ref_import.REFERENCE_ROOT
    layout = sorted(os.path.relpath(os.path.join(d, f), ref) for d, _, fs in os.walk(os.path.join(ref, "fourm"))
                    for f in fs if f.endswith(".py"))
    ref_import.install(extra_first_paths=[OVERLAY])
    import importlib
    for m in MODULES:
        importlib.import_module(m)

    def where(m):
        f = sys.modules[m].__file__
        return "overlay" if f.startswith(OVERLAY + os.sep) else "reference" if f.startswith(ref.rstrip(os.sep) + os.sep) else f
    import fourm.utils as utils
    from fourm.data.modality_info import MODALITY_INFO

    def factory(p):
        return None if p is None else dict(module=p.func.__module__, name=p.func.__qualname__, kwargs=p.keywords)
    info = {m: {k: factory(v) if k.endswith("_embedding") else v for k, v in MODALITY_INFO[m].items()} for m in MODS}
    mk = lambda m, side: MODALITY_INFO[m][side]() if MODALITY_INFO[m]["type"] != "img" else MODALITY_INFO[m][side](patch_size=16, image_size=224)
    model = utils.create_model("fm_tiny_6e_6d_swiglu_nobias", encoder_embeddings={m: mk(m, "encoder_embedding") for m in MODS},
                               decoder_embeddings={m: mk(m, "decoder_embedding") for m in MODS[1:]},
                               modality_info={m: MODALITY_INFO[m] for m in MODS})
    out = dict(layout=layout, resolved={m: where(m) for m in MODULES}, modality_info=info,
               model_class=[type(model).__module__, type(model).__name__])
    print(out["resolved"], out["model_class"])
    json.dump(out, open(os.path.join(HERE, "overlay_golden.json"), "w"), indent=0)


if __name__ == "__main__":
    main()
