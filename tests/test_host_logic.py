"""CPU tests of the host side: the C-ABI library loads and exports every symbol include/fvs_b200.h declares (no compute
calls — there is no GPU here), the Python mirror has the reference's signatures, the multi-GPU host logic works over
gloo with world_size 2, and the product refuses to run without CUDA."""
import inspect
import json
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    src = open(os.path.join(ROOT, "include", "fvs_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(fvs_[a-z0-9_]+)\s*\(", src)))


def test_library_builds_loads_and_exports_every_declared_symbol():
    from flash_vstream_b200 import _build, _lib
    _build.build()  # cross-compiles for sm_100a without a GPU; no-op when fresh
    lib = _lib.load()
    declared = header_functions()
    assert len(declared) >= 15
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/fvs_b200.h but not exported"
        assert name in _lib.SIGNATURES, f"{name} has no ctypes signature"
    assert set(_lib.SIGNATURES) == set(declared)
    assert lib.fvs_version() >= 100
    # a freshly loaded library has launched nothing (its own process: earlier tests of this one may have run kernels)
    fresh = subprocess.run([sys.executable, "-c", "from flash_vstream_b200 import _lib; print(_lib.load().fvs_launch_count())"],
                           cwd=ROOT, capture_output=True, text=True)
    assert fresh.returncode == 0, fresh.stderr
    assert fresh.stdout.strip() == "0"


def test_sass_contains_blackwell_tensor_and_tma_instructions():
    from flash_vstream_b200 import _build
    exe = "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([exe, "-sass", str(_build.LIB_PATH)], capture_output=True, text=True).stdout
    assert "UTCHMMA" in sass, "tcgen05.mma not found in SASS"
    assert "UTMALDG" in sass and "UTMASTG" in sass, "TMA load/store not found in SASS"
    assert "LDTM" in sass, "tcgen05.ld not found in SASS"
    assert "HMMA" not in sass.replace("UTCHMMA", ""), "legacy mma.sync path present"


def test_errors_map_to_python_exceptions_and_no_cpu_fallback():
    from flash_vstream_b200 import _lib, ops
    with pytest.raises(_lib.FvsError):
        ops.spatial_pool(torch.zeros(2, 576, 64, dtype=torch.float16), 8)   # CPU tensor: refused, never computed
    with pytest.raises(_lib.FvsError):
        ops.VitEncoder({"class_emb": torch.zeros(1024), "layers": []}, device="cpu")
    lib = _lib.load()
    rc = lib.fvs_linear(None, None, None, None, None, 1, 64, 64, 64, 64, 0, 0, 0, None)
    assert rc == _lib.FVS_EINVAL and b"null" in lib.fvs_last_error()
    with pytest.raises(ValueError):
        _lib.check(rc, "fvs_linear")
    rc = lib.fvs_weighted_kmeans(1, None, 1, 1, 10, 5, 1000, 10, 1e-4, 1, 1, 1, 1, 1, 1 << 30, 0, None)
    assert rc == _lib.FVS_EINVAL and b"multiple of 1024" in lib.fvs_last_error()
    assert lib.fvs_kmeans_workspace_bytes(26, 25, 16384) > 2 * 25 * 16384 * 2


def test_unknown_sample_type_raises_like_reference():
    from flash_vstream_b200.vstream_arch import FlashVStreamB200, NeuralTuringMachine
    m = FlashVStreamB200(None, NeuralTuringMachine(64, 32), video_sample_type="center")
    with pytest.raises(NotImplementedError):          # vstream_arch.py:235
        m.compress_temporal_features([torch.zeros(3, 64, 64)])
    m2 = FlashVStreamB200(None, NeuralTuringMachine(64, 32), compress_type="conv")
    with pytest.raises(NotImplementedError):          # vstream_arch.py:211
        m2.compress_spatial_features(torch.zeros(1, 64, 64), 4)
    with pytest.raises(AssertionError):               # vstream_arch.py:196
        m.compress_spatial_features(torch.zeros(1, 60, 64), 4)


def _seams():
    """tests/golden/seams.json: what the original Flash-VStream modules define (tests/golden/make_golden_seams.py)"""
    with open(os.path.join(ROOT, "tests", "golden", "seams.json")) as f:
        return json.load(f)


def _params(f):
    """[name, repr(default) or None] of every parameter that is not keyword-only (the format of seams.json)"""
    return [[p.name, None if p.default is p.empty else repr(p.default)]
            for p in inspect.signature(f).parameters.values() if p.kind is not p.KEYWORD_ONLY]


def _stand_in_modules(monkeypatch, names_by_module, classes=None):
    """register, for the duration of a test, module objects under the original modules' import names that define the
    names each original module defines (values are placeholders), so install() rebinds attributes on modules of the
    original layout; returns {module name: module}"""
    import types
    mods = {}
    for full, names in names_by_module.items():
        parts = full.split(".")
        for i in range(1, len(parts) + 1):
            name = ".".join(parts[:i])
            if name not in mods:
                mod = types.ModuleType(name)
                mod.__path__ = []
                mods[name] = mod
                monkeypatch.setitem(sys.modules, name, mod)
                if i > 1:
                    setattr(mods[".".join(parts[:i - 1])], parts[i - 1], mod)
        for n in names:
            setattr(mods[full], n, object())
    for (full, cls_name), methods in (classes or {}).items():
        setattr(mods[full], cls_name, type(cls_name, (), {m: object() for m in methods}))
    return mods


def test_mirror_signatures_match_reference():
    from flash_vstream_b200 import clip_encoder as mclip
    from flash_vstream_b200 import compress_functions as mcf
    from flash_vstream_b200 import vstream_arch as march
    ref = _seams()["llava"]
    for name, want in ref["compress_functions"].items():
        assert _params(getattr(mcf, name)) == want, name
    for name in ("encode_images", "attention", "compress_spatial_features"):
        assert _params(getattr(march.VStreamMetaForCausalLM, name)) == ref["VStreamMetaForCausalLM"][name], name
    for name in ("compress_temporal_features", "embed_video_streaming"):   # ours add an optional trailing `draws=None`
        mine = _params(getattr(march.VStreamMetaForCausalLM, name))
        assert mine[:-1] == ref["VStreamMetaForCausalLM"][name] and mine[-1] == ["draws", "None"], name
    assert _params(mclip.CLIPVisionTower.__init__) == ref["CLIPVisionTower"]["__init__"]
    assert _params(mclip.CLIPVisionTower.forward) == ref["CLIPVisionTower"]["forward"]
    ntm_mine = march.NeuralTuringMachine(64, 32).state_dict()
    assert {k: list(v.shape) for k, v in ntm_mine.items()} == ref["ntm_64_32_state_dict"]


def test_install_rebinds_reference_seam(monkeypatch):
    import flash_vstream_b200
    from flash_vstream_b200 import clip_encoder as mclip
    from flash_vstream_b200 import compress_functions as mcf
    from flash_vstream_b200 import multimodal_projector as mproj
    from flash_vstream_b200 import vstream_arch as march
    ref = _seams()["llava"]
    arch = "flash_vstream.model.vstream_arch"
    mods = _stand_in_modules(monkeypatch, ref["modules"],
                             {(arch, "VStreamMetaForCausalLM"): ref["VStreamMetaForCausalLM_methods"]})
    rcf, rarch = mods["flash_vstream.model.compress_functions"], mods[arch]
    Ref = rarch.VStreamMetaForCausalLM
    keep = Ref.embed_video_streaming
    patched = flash_vstream_b200.install()
    assert rcf.weighted_kmeans_feature is mcf.weighted_kmeans_feature
    assert rarch.weighted_kmeans_feature is mcf.weighted_kmeans_feature
    assert "VStreamMetaForCausalLM.embed_video_streaming" in patched
    assert Ref.embed_video_streaming is not keep
    for name in ref["modules"]["flash_vstream.model.compress_functions"]:
        assert getattr(rcf, name) is getattr(mcf, name), name
    assert rarch.build_vision_projector is mproj.build_vision_projector
    assert mods["flash_vstream.model.multimodal_projector.builder"].build_vision_projector is mproj.build_vision_projector
    for mod in ("flash_vstream.model.multimodal_encoder.clip_encoder", "flash_vstream.model.multimodal_encoder.builder"):
        assert mods[mod].CLIPVisionTower is mclip.CLIPVisionTower, mod
    for name in ("encode_images", "attention", "compress_spatial_features", "compress_temporal_features", "cat_proj",
                 "reshape_2x2_image_features"):        # methods the original class defines and the mirror replaces
        assert name in ref["VStreamMetaForCausalLM_methods"], name
        assert getattr(Ref, name) is getattr(march.VStreamMetaForCausalLM, name), name


def test_install_qwen_rebinds_reference_seam_and_signatures(monkeypatch):
    """the Qwen-side seam: FlashMemory (offline + streaming) and weighted_kmeans_ordered_feature on modules laid out like
    the original `models.*` ones, same constructor / method signatures as the original's"""
    import flash_vstream_b200.qwen as mine
    from flash_vstream_b200.qwen import vstream_qwen2vl_realtime as mine_rt
    ref = _seams()["qwen"]
    assert _params(mine.FlashMemory.__init__) == ref["FlashMemory"]["__init__"]
    for name in ("temporal_pool", "cat_spa_tem", "calc_am_rope"):
        assert _params(getattr(mine.FlashMemory, name)) == ref["FlashMemory"][name], name
    for name in ("temporal_compress", "spatial_enhance", "forward"):        # ours add one optional trailing `draws=None`
        got = _params(getattr(mine.FlashMemory, name))
        assert got[:-1] == ref["FlashMemory"][name] and got[-1] == ["draws", "None"], name
    got = _params(mine_rt.FlashMemory.temporal_compress)
    assert got[:-1] == ref["realtime_FlashMemory"]["temporal_compress"] and got[-1] == ["draws", "None"]
    assert _params(mine.weighted_kmeans_ordered_feature) == ref["weighted_kmeans_ordered_feature"]
    for name, want in ref["FlashVStreamQwen2VLModel"].items():
        got = _params(getattr(mine_rt.RealtimeStreamingMixin, name))
        assert got[: len(want)] == want, name
    mods = _stand_in_modules(monkeypatch, ref["modules"])
    ref_model, ref_rt = mods["models.vstream_qwen2vl_model"], mods["models.vstream_qwen2vl_realtime"]
    ref_cf = mods["models.compress_functions"]
    from flash_vstream_b200.install import install_qwen
    patched = install_qwen()
    assert ref_model.FlashMemory is mine.FlashMemory and ref_rt.FlashMemory is mine_rt.FlashMemory
    assert ref_cf.weighted_kmeans_ordered_feature is mine.weighted_kmeans_ordered_feature
    assert ref_model.weighted_kmeans_ordered_feature is mine.weighted_kmeans_ordered_feature
    assert ref_rt.weighted_kmeans_ordered_feature is mine.weighted_kmeans_ordered_feature
    assert len(patched) == 3


def test_shard_streams():
    from flash_vstream_b200.distributed import shard_streams
    for n, w in ((8, 8), (10, 4), (3, 8), (1000, 7)):
        owned = [shard_streams(n, r, w) for r in range(w)]
        flat = [s for o in owned for s in o]
        assert flat == list(range(n))
        assert max(len(o) for o in owned) - min(len(o) for o in owned) <= 1


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    from flash_vstream_b200.distributed import allgather_prefix, unpack_prefixes
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        rows = 681 if rank == 0 else 3 + 2 * 16 + 2 * 64   # rank 1 is still warming up (fewer rows)
        g = torch.Generator().manual_seed(rank)
        prefix = torch.randn(rows, 32, generator=g).half()
        stacked, nrows = allgather_prefix(prefix, 681)
        parts = unpack_prefixes(stacked, nrows)
        ok = stacked.shape == (world, 681, 32) and nrows.tolist() == [681, 163]
        for r in range(world):
            exp = torch.randn(int(nrows[r]), 32, generator=torch.Generator().manual_seed(r)).half()
            ok = ok and torch.equal(parts[r], exp) and bool((stacked[r, int(nrows[r]):] == 0).all())
        # Qwen variant of the same exchange: each rank's merged video embeddings [<= 6480, hidden] in bf16 plus its AM-RoPE
        # position ids; rank 1's stream is still short
        qrows = 6480 if rank == 0 else 1440
        emb = torch.randn(qrows, 48, generator=g).bfloat16()
        qs, qn = allgather_prefix(emb, 6480)
        ok = ok and qs.shape == (world, 6480, 48) and qn.tolist() == [6480, 1440] and torch.equal(qs[rank, :qrows], emb)
        pos = torch.arange(3 * qrows, dtype=torch.int64).view(qrows, 3) + rank
        ps, pn = allgather_prefix(pos, 6480)
        ok = ok and ps.dtype == torch.int64 and torch.equal(unpack_prefixes(ps, pn)[rank], pos)
        q.put((rank, bool(ok)))
    finally:
        dist.destroy_process_group()


def test_prefix_allgather_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert res == [(0, True), (1, True)]


def test_rng_contract_never_rewinds_python_random():
    """ADVICE r1: the refill candidates come from a private clone of `random`; the global generator is only ever ADVANCED
    by the number of draws the device consumed (0 in the common case), never rewound over what the user did in between"""
    import random
    from flash_vstream_b200 import compress_functions as cf

    class Ev:
        def synchronize(self):
            pass

    cf._unsettled.clear()
    random.seed(5)
    cf._unsettled.append([26, torch.tensor([1, 0, 1, 0], dtype=torch.int32), Ev()])      # nothing consumed
    random.seed(7)                                                                        # the user reseeds in between
    cf.sync_rng()
    probe = random.random()
    random.seed(7)
    assert probe == random.random(), "global RNG state was touched although no refill was consumed"
    cf._unsettled.append([26, torch.tensor([1, 2, 1, 0], dtype=torch.int32), Ev()])      # two refills consumed
    random.seed(11)
    cf.sync_rng()
    probe = random.random()
    random.seed(11)
    random.randint(0, 25), random.randint(0, 25)
    assert probe == random.random(), "the global RNG must be advanced by exactly the consumed draws"
    assert not cf._unsettled


def test_inference_only_guard_and_metric_meter():
    from types import SimpleNamespace
    from flash_vstream_b200 import multimodal_projector as mp
    from flash_vstream_b200.serve import MetricMeter
    from flash_vstream_b200.vstream_arch import _is_manager_proxy
    proj = mp.build_vision_projector(SimpleNamespace(mm_projector_type="mlp2x_gelu", hidden_size=64), 64)
    with torch.enable_grad(), pytest.raises(RuntimeError, match="inference-only"):
        proj(torch.zeros(2, 64))                       # parameters require grad and grad mode is on: refuse, do not detach
    m = MetricMeter()
    with pytest.raises(KeyError):
        m["memory_latency"]
    m.add("memory_latency", 0.5)
    m.add("memory_latency", 0.25)
    assert m["memory_latency"] == "0.250000 (0.375000, 0.500000)"      # cli_video_stream.py:59-63 format
    assert m.val("memory_latency") == 0.25 and m.max("memory_latency") == 0.5
    import multiprocessing as mproc
    assert not _is_manager_proxy([])
    with mproc.Manager() as mgr:
        assert _is_manager_proxy(mgr.list())


def test_stale_library_is_not_loaded_silently(tmp_path, monkeypatch):
    from flash_vstream_b200 import _build, _lib
    monkeypatch.setattr(_build, "is_fresh", lambda: False)
    monkeypatch.setattr(_build, "can_build", lambda: False)
    monkeypatch.setattr(_lib, "_lib", None)
    with pytest.raises(_lib.FvsError, match="stale"):
        _lib.load(build_if_missing=False)


def test_qwen_lazy_members_materialise_on_demand():
    """qwen/compress_functions.LazyMembers: the member lists of the ordered k-means are built from (labels, cluster order)
    only when somebody reads them"""
    from flash_vstream_b200.qwen.compress_functions import LazyMembers
    labels = torch.tensor([2, 0, 2, 1, 0], dtype=torch.int32)
    order = torch.tensor([1, 2, 0], dtype=torch.int64)
    m = LazyMembers(labels, order)
    assert m._lists is None
    assert len(m) == 3 and m[0] == [3] and list(m) == [[3], [0, 2], [1, 4]] and m == [[3], [0, 2], [1, 4]]
    assert m._labels is None            # the device tensors are released once materialised


def test_qwen_stream_state_fill_phase_on_host_tensors():
    """qwen/stream_state.QwenStreamState while the memory is filling (pass-through branches only: no kernel is reached, so
    the bookkeeping runs on CPU tensors): banks grow in place, the CSM is the concatenation of the half-resolution frames,
    the DAM is the whole bank, the 13-item list has the reference's layout with host thw triples."""
    from flash_vstream_b200.qwen.stream_state import QwenStreamState
    from flash_vstream_b200.qwen.vstream_qwen2vl_realtime import FlashMemory
    flash = FlashMemory(flash_memory_temporal_length=12, flash_memory_spatial_length=8)      # 6 CSM / 4 DAM frames
    st = QwenStreamState(flash, merger=None)
    g = torch.Generator().manual_seed(0)
    t, h, w, D = 2, 4, 4, 64
    xs, smalls = [], []
    for s in range(2):
        x = torch.randn(t * h * w, D, generator=g).bfloat16()
        small = torch.randn(t * 4, D, generator=g).bfloat16()
        xs.append(x)
        smalls.append(small)
        st.step(x, small, t, (h, w), (2, 2), s * t)
        (tem_x, tem_thw, tem_w, tem_ts, spa_x, spa_thw, spa_pos, bank, thw, small_bank, small_thw, embeds, shape) = st.as_list()
        n = t * (s + 1)
        assert thw.tolist() == [n, h, w] and small_thw.tolist() == [n, 2, 2] and tem_thw.tolist() == [n, 2, 2]
        assert spa_thw.tolist() == [n, h, w] and spa_pos.tolist() == list(range(n))
        assert torch.equal(bank, torch.cat(xs)) and torch.equal(small_bank, torch.cat(smalls))
        assert torch.equal(tem_x, torch.cat(smalls)) and torch.equal(spa_x.reshape(-1, D), torch.cat(xs))
        assert tem_w.tolist() == [1.0] * n and tem_ts.tolist() == list(range(n)) and tem_ts.dtype == torch.int32
        assert embeds is None and shape is None and st.n_tem == n and st.n_frames == n
    assert st.fast_steps == 0 and st.redone_steps == 0
    with pytest.raises(AssertionError):                                   # merge_thw of the reference: grids must agree
        st.step(xs[0][: 2 * 4], smalls[0][:2], 1, (2, 4), (1, 2), 4)


def test_bench_gemm_breakdown_groups_launches_by_position():
    import importlib.util
    spec = importlib.util.spec_from_file_location("_bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    M = 18464
    w = [2.0 * M * 1024 * 640] + [2.0 * M * n * k for _ in range(23) for (n, k) in ((3072, 1024), (1024, 1024), (4096, 1024), (1024, 4096))]
    ms = [0.05] + [t for _ in range(23) for t in (0.080, 0.040, 0.112, 0.100)]
    out = bench.gemm_breakdown(ms, w)
    assert abs(out["qkv"] - 2.0 * M * 3072 * 1024 / 0.080e-3 / 1e12) < 1e-6
    assert abs(out["fc2_residual"] - 2.0 * M * 1024 * 4096 / 0.100e-3 / 1e12) < 1e-6
    assert abs(out["ms"]["out_proj_residual"] - 23 * 0.040) < 1e-9
    plain = (w[0] + 23 * 2.0 * M * (3072 + 4096) * 1024) / ((0.05 + 23 * 0.192) * 1e-3) / 1e12
    assert abs(out["without_residual_epilogue"] - plain) < 1e-6
    assert bench.gemm_breakdown(ms[:-1], w[:-1]) is None


def test_bench_dump_outputs_writes_float32_memory_and_a_fixed_buffer_sample(tmp_path):
    import importlib.util
    import numpy as np
    spec = importlib.util.spec_from_file_location("_bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    g = torch.Generator().manual_seed(0)
    cur, lng, tur = (torch.randn(*s, generator=g).half() for s in ((4, 64, 32), (25, 16, 32), (25, 1, 32)))
    buf = torch.arange(100, dtype=torch.float16).view(100, 1, 1).expand(100, 64, 32).contiguous()
    names = bench.dump_outputs(str(tmp_path / "a"), [cur, lng, tur, buf], buffer_frames=8)
    bench.dump_outputs(str(tmp_path / "b"), [cur, lng, tur, buf], buffer_frames=8)
    assert names == ["memory_buffer_sample", "memory_current", "memory_long", "memory_turing"]
    for name, want in (("memory_current", cur), ("memory_long", lng), ("memory_turing", tur)):
        got = np.load(tmp_path / "a" / f"{name}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, want.float().numpy()), name
    sample = np.load(tmp_path / "a" / "memory_buffer_sample.npy")
    frames = sample[:, 0, 0]
    assert sample.shape == (8, 64, 32) and sample.dtype == np.float32
    assert len(set(frames)) == 8 and (np.diff(frames) > 0).all()          # distinct frames, in stream order
    assert np.array_equal(sample, np.load(tmp_path / "b" / "memory_buffer_sample.npy"))   # the same frames every run
