"""Generate tests/golden/seams.json and tests/golden/seams.npz from the ORIGINAL Flash-VStream checkout (unmodified,
imported on CPU), for the tests that used to import it at test time:

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden_seams.py <path to the Flash-VStream checkout>

seams.json: the parameter lists (name, repr of the default) of every function and method the drop-in mirrors replace, the
NeuralTuringMachine(64, 32) state-dict shapes, and which of the names install() / install_qwen() rebind each original
module defines.  seams.npz: reshape_2x2_image_features of the LLaVA variant on an index-coded input (the function only
moves elements, so the stored gather map is its output on any input of that shape), and the outputs and RNG draws of the
Qwen variant's weighted_kmeans_ordered_feature and fast_weighted_kmeans_ordered_feature on the same case and seed.
"""
from __future__ import annotations

import contextlib
import importlib
import inspect
import io
import json
import os
import random
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from tests import qwen_inputs as QI  # noqa: E402

LLAVA_CF = ("weighted_kmeans_feature", "attention_feature", "drop_feature", "merge_feature", "kmeans_feature",
            "k_drop_feature", "k_merge_feature")
LLAVA_ARCH = ("encode_images", "attention", "compress_spatial_features", "compress_temporal_features", "embed_video_streaming")
QWEN_MODEL = ("__init__", "temporal_pool", "cat_spa_tem", "calc_am_rope", "temporal_compress", "spatial_enhance", "forward")
QWEN_RT = ("embed_new_video_clip", "prepare_realtime_inference", "get_video_embedding_memory_cuda_list")
FAST_CASE, FAST_SEED = "ko_scene_bf16", 5


@contextlib.contextmanager
def recorded_draws():
    """log what torch.randperm / random.randint return while the original code runs (the draws the oracle replays)"""
    rec = types.SimpleNamespace(perms=[], ints=[])
    rp, ri = torch.randperm, random.randint

    def randperm(*a, **k):
        r = rp(*a, **k)
        rec.perms.append(r.clone())
        return r

    def randint(a, b):
        r = ri(a, b)
        rec.ints.append(r)
        return r

    torch.randperm, random.randint = randperm, randint
    try:
        yield rec
    finally:
        torch.randperm, random.randint = rp, ri


def params(f):
    """[name, repr(default) or None] of every parameter that is not keyword-only"""
    return [[p.name, None if p.default is p.empty else repr(p.default)]
            for p in inspect.signature(f).parameters.values() if p.kind is not p.KEYWORD_ONLY]


def present(mod, names):
    return sorted(n for n in names if hasattr(mod, n))


def llava(ref_root, out, arrays):
    sys.path.insert(0, os.path.join(ref_root, "Flash-VStream-LLaVA"))
    rcf = importlib.import_module("flash_vstream.model.compress_functions")
    rarch = importlib.import_module("flash_vstream.model.vstream_arch")
    rclip = importlib.import_module("flash_vstream.model.multimodal_encoder.clip_encoder")
    rbuilder = importlib.import_module("flash_vstream.model.multimodal_encoder.builder")
    rproj = importlib.import_module("flash_vstream.model.multimodal_projector.builder")
    Ref = rarch.VStreamMetaForCausalLM
    out["llava"] = {
        "compress_functions": {n: params(getattr(rcf, n)) for n in LLAVA_CF},
        "VStreamMetaForCausalLM": {n: params(getattr(Ref, n)) for n in LLAVA_ARCH},
        "CLIPVisionTower": {n: params(getattr(rclip.CLIPVisionTower, n)) for n in ("__init__", "forward")},
        "ntm_64_32_state_dict": {k: list(v.shape) for k, v in rarch.NeuralTuringMachine(64, 32).state_dict().items()},
        "modules": {
            "flash_vstream.model.compress_functions": present(rcf, LLAVA_CF),
            "flash_vstream.model.vstream_arch": present(rarch, LLAVA_CF + ("build_vision_projector",)),
            "flash_vstream.model.multimodal_encoder.clip_encoder": present(rclip, ("CLIPVisionTower",)),
            "flash_vstream.model.multimodal_encoder.builder": present(rbuilder, ("CLIPVisionTower",)),
            "flash_vstream.model.multimodal_projector.builder": present(rproj, ("build_vision_projector",)),
        },
        "VStreamMetaForCausalLM_methods": sorted(n for n, v in vars(Ref).items() if callable(v)),
    }
    B, P, D = 2, 576, 32
    coded = torch.arange(B * P * D, dtype=torch.float32).reshape(B, P, D)
    got = Ref.reshape_2x2_image_features(None, coded)
    assert got.dtype == torch.float32 and torch.equal(got, got.round()), "not a pure rearrangement"
    gather = got.to(torch.int64)
    x = torch.randn(B, P, D, generator=torch.Generator().manual_seed(5))
    assert torch.equal(Ref.reshape_2x2_image_features(None, x), x.reshape(-1)[gather])
    arrays["reshape_2x2_gather"] = gather.numpy().astype(np.int32)


def qwen(ref_root, out, arrays):
    # the import shim of tests/golden/make_golden_qwen.py: a symbol of an older transformers that only the original LLM
    # forward uses, and the `models` package registered by path so its relative imports resolve
    import transformers.models.qwen2_vl.modeling_qwen2_vl as hf
    if not hasattr(hf, "_prepare_4d_causal_attention_mask_with_cache_position"):
        hf._prepare_4d_causal_attention_mask_with_cache_position = None
    pkg = types.ModuleType("models")
    pkg.__path__ = [os.path.join(ref_root, "Flash-VStream-Qwen", "models")]
    sys.modules["models"] = pkg
    ref_model = importlib.import_module("models.vstream_qwen2vl_model")
    ref_rt = importlib.import_module("models.vstream_qwen2vl_realtime")
    ref_cf = importlib.import_module("models.compress_functions")
    seam = ("FlashMemory", "weighted_kmeans_ordered_feature")
    out["qwen"] = {
        "FlashMemory": {n: params(getattr(ref_model.FlashMemory, n)) for n in QWEN_MODEL},
        "realtime_FlashMemory": {"temporal_compress": params(ref_rt.FlashMemory.temporal_compress)},
        "weighted_kmeans_ordered_feature": params(ref_cf.weighted_kmeans_ordered_feature),
        "FlashVStreamQwen2VLModel": {n: params(getattr(ref_rt.FlashVStreamQwen2VLModel, n)) for n in QWEN_RT},
        "modules": {
            "models.compress_functions": present(ref_cf, ("weighted_kmeans_ordered_feature",)),
            "models.vstream_qwen2vl_model": present(ref_model, seam),
            "models.vstream_qwen2vl_realtime": present(ref_rt, seam),
        },
    }
    c = QI.KMEANS_CASES[FAST_CASE]
    x, w = QI.kmeans_input(c)
    for tag, fn in (("slow", ref_cf.weighted_kmeans_ordered_feature), ("fast", ref_cf.fast_weighted_kmeans_ordered_feature)):
        torch.manual_seed(FAST_SEED)
        random.seed(FAST_SEED)
        with recorded_draws() as rec, contextlib.redirect_stdout(io.StringIO()):
            feat, weights, ts, idx = fn(x.clone(), c["K"], None if w is None else w.clone())
        arrays[f"{tag}_feat"] = QI.to_bits(feat)
        arrays[f"{tag}_weights"] = weights.float().numpy()
        arrays[f"{tag}_ts"] = ts.float().numpy()
        arrays[f"{tag}_members"] = np.array([len(m) for m in idx], np.int32)
        arrays[f"{tag}_members_flat"] = np.array([j for m in idx for j in m], np.int32)
        arrays[f"{tag}_init"] = rec.perms[0][: c["K"]].numpy().astype(np.int32) if rec.perms else np.zeros(0, np.int32)
        arrays[f"{tag}_refill"] = np.array(rec.ints, np.int32)
    arrays["fast_chk"] = QI.checksum(x)
    out["qwen"]["fast_kmeans"] = {"case": FAST_CASE, "seed": FAST_SEED}


def main():
    ref_root = os.path.abspath(sys.argv[1])
    out, arrays = {}, {}
    llava(ref_root, out, arrays)
    qwen(ref_root, out, arrays)
    with open(os.path.join(HERE, "seams.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    np.savez_compressed(os.path.join(HERE, "seams.npz"), **arrays)
    print("seams.json", sorted(out), "seams.npz", sorted(arrays))


if __name__ == "__main__":
    main()
