#!/usr/bin/env python
"""bench.py — frames/s encoded + consolidated into the Flash memory (BASELINE.json metric).

One "step" = one embed_video_streaming call on a clip of CHUNK synthetic 336x336 frames: ViT-L/14 encode (23 layers,
f16 with fp32 residual stream; the layer stack replays as one CUDA graph) with the three STAR levels pooled in the
encoder's tail, + ONE fused consolidation kernel on the persistent per-GPU bank (weighted k-means over 25+CHUNK rows,
abstract-memory update, key retrieval, write-back of the [Turing|long|key|current] prefix).  31 steps x 32 frames ~ the
1k-frame stream of BASELINE config[1].  Multi-GPU (torchrun): one stream-shard per GPU (weak scaling), NO collective on the
per-frame path; the NCCL all-gather of the [681,1024] memory prefix happens once per QUERY (end of the stream), is inside
the timed region once, and is also timed alone (`allgather_us`).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--chunk 32] [--microbatch 32]
    ablations: --gather-every-step  --no-sampler  --no-graph  --op-by-op
    --dump-outputs DIR: after the timed steps, the memory they left as DIR/<name>.npy (seeded inputs: two builds compare
    output for output)

Prints ONE JSON line (rank 0).  `value` = frames/s with inputs resident in HBM; `e2e` = the same through the public
API from pinned HOST frames (H2D inside the timed region, D2H of the memory prefix every step).
`--impl reference` times the reference's CPU path (transformers CLIPVisionModel — the library the reference calls —
plus the oracle port of the consolidation) on a bounded sample of the same workload (same clip length).
"""
from __future__ import annotations

import argparse
import datetime
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GFLOP_PER_FRAME = 366.0          # SURVEY.md §8d: 23 layers x 15.884 + 0.694 patch embed (N=577, D=1024, F=4096)
GEMM_GFLOP_PER_FRAME = 334.65    # the 93 GEMMs alone (23 x 14.52 + 0.69)
CONSOLIDATION_BYTES_PER_FRAME = 4.17e6  # SURVEY.md §8d streaming, default 681-token bank, f16 (2.99e6 with the pooled tail)
METRIC = "frames/sec into memory (336px, ViT-L/14)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=31)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--chunk", type=int, default=32, help="frames per embed_video_streaming call")
    ap.add_argument("--microbatch", type=int, default=32, help="frames per ViT micro-batch")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-prof", action="store_true", help="disable the per-launch CUDA events (roofline becomes null)")
    ap.add_argument("--steady-s", type=float, default=3.0, help="seconds of the steady-state pass (0 = skip)")
    ap.add_argument("--no-extras", action="store_true", help="skip the chunk=1 / bank=256 / offline / torch_gpu rows (N=1 only)")
    # ablations of the round-1 scaling collapse (SCALE_r01: 0.51 at N=8)
    ap.add_argument("--gather-every-step", action="store_true", help="all-gather the prefix after EVERY step (round-1 behaviour)")
    ap.add_argument("--no-sampler", action="store_true", help="no nvidia-smi clock sampling")
    ap.add_argument("--no-graph", action="store_true", help="launch the ViT layer stack eagerly (FVS_VIT_GRAPH=0)")
    ap.add_argument("--op-by-op", action="store_true", help="op-by-op consolidation instead of fvs_stream_step")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the memory the last timed step left (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return args


def dump_outputs(out_dir, memory, buffer_frames=64):
    """Write `video_embedding_memory` = [current, long, Turing, frame buffer], what a caller of embed_video_streaming
    reads, as float32 DIR/<name>.npy.  The frame buffer holds one 8x8 map per frame of the stream (285 MB in float32 for
    the default run), so only `buffer_frames` of its frames are written, picked by a fixed seed and kept in stream order."""
    import numpy as np
    cur, lng, tur, buf = memory
    rows = np.sort(np.random.default_rng(0).choice(buf.shape[0], size=min(buf.shape[0], buffer_frames), replace=False))
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"memory_current": cur, "memory_long": lng, "memory_turing": tur, "memory_buffer_sample": buf[rows.tolist()]}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())
    return sorted(arrays)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"tensor": d.get("bf16_tflops_sustained", 1421.6), "tensor_burst": d.get("bf16_tflops", 1679.2),
                "hbm": d.get("hbm_gbs", 6571.9), "source": "measured",
                "sustained_clock_mhz": (d.get("clocks_under_load") or {}).get("sm_mhz_median")}
    return {"tensor": 1400.0, "tensor_burst": 1590.0, "hbm": 6650.0, "source": "fallback", "sustained_clock_mhz": 1300.0}


class ClockSampler:
    """ONE nvidia-smi process for the whole node (rank 0 starts it, seconds before the first timed region, -lms 200 like the
    recipe's clocks line in B200_PROFILING.md); rows carry a timestamp, so every timed region picks its own samples."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, enabled=True):
        self.p, self.f, self.rows = None, None, None
        if not enabled:
            return
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
            self.t_start = time.time()
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = []
        for line in open(self.f.name):
            r = [c.strip() for c in line.strip().split(",")]
            if len(r) < 10:
                continue
            try:
                ts = datetime.datetime.strptime(r[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, int(r[1]), float(r[2]), float(r[3]), float(r[4]),
                             [n for n, v in zip(self.NAMES, r[6:10]) if v.lower().startswith("active")]))
            except Exception:
                pass
        os.unlink(self.f.name)
        self.rows = rows
        self.p = None

    def window(self, t0, t1, gpu=None, n_gpus=None):
        """median SM clock etc. of the samples taken in [t0, t1] (wall clock) on `gpu` (None = GPUs 0..n_gpus-1: the ranks' GPUs,
        not the idle ones of a bigger box)"""
        if gpu is None and n_gpus is not None and self.rows is not None:
            rows_all, self.rows = self.rows, [r for r in self.rows if r[1] < n_gpus]
            try:
                return self.window(t0, t1)
            finally:
                self.rows = rows_all
        if self.rows is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable" if self.f is None else "no samples"]}
        pad = 0.0
        sel = [r for r in self.rows if t0 - pad <= r[0] <= t1 + pad and (gpu is None or r[1] == gpu)]
        if not sel:   # a region shorter than the sampling period: take the nearest sample on either side
            near = sorted((r for r in self.rows if gpu is None or r[1] == gpu), key=lambda r: min(abs(r[0] - t0), abs(r[0] - t1)))
            sel = near[:2]
        if not sel:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(r[2] for r in sel)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(r[3] for r in sel), "power_w_max": max(r[4] for r in sel),
                "samples": len(sel), "reasons": sorted({n for r in sel for n in r[5]})}


# ------------------------------------------------------------------------------------------------ reference CPU arm
_cpu_threads = None


def pick_cpu_threads():
    """Thread count that runs the reference's dominant CPU op (a [577,1024]x[1024,4096] fp32 matmul) fastest on this
    host: cgroup quotas / SMT make `os.cpu_count()` threads far slower than fewer on some boxes, and the CPU arm is
    supposed to be the reference at its best."""
    global _cpu_threads
    if _cpu_threads is not None:
        return _cpu_threads
    import torch
    total = os.cpu_count() or 1
    cands = {total, 96, 64, 48, 32, 24, 16, 8}
    try:
        cands.add(len(os.sched_getaffinity(0)))
        q = open("/sys/fs/cgroup/cpu.max").read().split()
        if q[0] != "max":
            cands.add(max(1, int(int(q[0]) / int(q[1]))))
    except Exception:
        pass
    a, w = torch.randn(577 * 4, 1024), torch.randn(4096, 1024)
    best = (None, 1e9)
    for c in sorted(c for c in cands if 1 <= c <= total):
        torch.set_num_threads(c)
        torch.matmul(a, w.t())
        t0 = time.perf_counter()
        for _ in range(3):
            torch.matmul(a, w.t())
        dt = time.perf_counter() - t0
        if dt < best[1]:
            best = (c, dt)
    _cpu_threads = best[0]
    return _cpu_threads


class CpuReference:
    """The reference's CPU path: CLIPVisionTower semantics over transformers' CLIPVisionModel (24 layers,
    output_hidden_states=True, hidden_states[-2][:,1:], clip_encoder.py:41-53), fp32, all host threads that help; then the
    consolidation in f16 torch-CPU ops (oracle/fast_cpu.py, pinned to the oracle by tests), clips of `clip` frames per
    embed_video_streaming call exactly like the GPU arm."""

    def __init__(self):
        import torch
        from oracle import fast_cpu as FC
        from oracle import fvs_oracle as O
        from tests import golden_inputs as GI
        self.torch, self.FC, self.GI = torch, FC, GI
        self.cores = pick_cpu_threads()
        torch.set_num_threads(self.cores)
        cfg = O.VitConfig()
        w = O.random_vit_weights(cfg, 0)
        self.kind_vit = "transformers.CLIPVisionModel"
        try:
            from transformers import CLIPVisionConfig, CLIPVisionModel
            hf_cfg = CLIPVisionConfig(hidden_size=cfg.hidden, intermediate_size=cfg.mlp, num_hidden_layers=cfg.layers,
                                      num_attention_heads=cfg.heads, image_size=cfg.image_size, patch_size=cfg.patch_size)
            model = CLIPVisionModel(hf_cfg).eval()
            model.load_state_dict(O.hf_state_dict(w, cfg), strict=False)

            def encode(p):
                with torch.no_grad():
                    return model(p, output_hidden_states=True).hidden_states[-2][:, 1:]
        except Exception:  # transformers unavailable: the oracle's own restatement (runs 23 layers)
            self.kind_vit = "oracle.vit_forward"

            def encode(p):
                with torch.no_grad():
                    return O.vit_forward(p, w, cfg)
        self.encode = encode
        wn = GI.ntm_weights(1024, 32, 0)
        self.ntm = (wn["q_w"], wn["q_b"], wn["k_w"], wn["k_b"])
        # pre-fill the bank (not timed) so the sample pays the steady-state k-means (25 + clip rows -> 25)
        self.state = FC.State()
        warm = GI.scene_features(26, 64, 1024, 3)
        for s in range(26):
            dn = GI.kmeans_draws(26, 25, s) if s >= 25 else (None, None)
            self.state = FC.stream_step(self.state, warm[s:s + 1], self.ntm, dn[0], dn[1])
        self.g = torch.Generator().manual_seed(1234)
        encode(torch.randn(1, 3, 336, 336, generator=self.g))  # one untimed warm-up frame (thread pool, allocator)
        self.k = 0

    def clip(self, n_frames: int, sub: int = 8):
        """one embed_video_streaming call on an n_frames clip; returns (seconds, seconds in the ViT)"""
        torch, FC, GI = self.torch, self.FC, self.GI
        pix = torch.randn(n_frames, 3, 336, 336, generator=self.g)
        t0 = time.perf_counter()
        feats = [self.encode(pix[i:i + sub]).to(torch.float16) for i in range(0, n_frames, sub)]   # encode_images, :643
        t_vit = time.perf_counter() - t0
        f64 = FC.pool(torch.cat(feats), 8)                                                          # compress_spatial_features, :644
        self.k += 1
        dn = GI.kmeans_draws(25 + n_frames, 25, 100 + self.k)
        self.state = FC.stream_step(self.state, f64, self.ntm, dn[0], dn[1])
        return time.perf_counter() - t0, t_vit


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t_all = time.perf_counter()
    ref = CpuReference()
    probe_s, _ = ref.clip(2)                      # untimed probe: seconds per frame on this host
    per_frame = probe_s / 2
    budget_s = 150.0
    clip = args.chunk
    same_clip = True
    if clip * per_frame > budget_s:               # even one full clip does not fit: bounded sample of the clip
        clip = max(1, int(budget_s / per_frame))
        same_clip = False
    n_clips = max(1, min(args.steps, int(budget_s / (clip * per_frame))))
    secs = vit_secs = 0.0
    for _ in range(n_clips):
        a, b = ref.clip(clip)
        secs += a
        vit_secs += b
    frames = n_clips * clip
    fps = frames / secs
    sample = (f"{n_clips} clip(s) of {clip} frames ({frames} frames, {secs:.1f} s of which ViT {vit_secs:.1f} s): 24-layer "
              f"{ref.kind_vit} fp32 + f16 torch-CPU consolidation, {ref.cores} threads")
    line = {
        "metric": METRIC, "impl": "reference", "value": fps, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * clip / fps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"1k-frame 336x336 stream in {args.chunk}-frame clips, ViT-L/14 + STAR Flash memory (681-token "
                               f"bank); reference CPU path, 1 process", "chunk_frames": clip, "sample": sample},
        "same_config": {"chunk_frames": same_clip, "bank": True, "dtype": "fp32 on the CPU (the reference's CPU dtype) vs f16 on the GPU",
                        "layers": "24 executed (the reference runs and discards the last layer), 23 needed",
                        "steps": f"{n_clips} timed clip(s) instead of {args.steps} (bounded to ~150 s of CPU work)"},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": ref.cores, "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t_all,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ B200 arm
def gemm_breakdown(mss, works):
    """per-GEMM-kind TFLOP/s of one micro-batch's tensor-core launches, in launch order: patch GEMM, then per layer QKV,
    out-proj, fc1, fc2 (vit_engine.cu stack_launches).  mss / works: sequences of milliseconds and FLOP of the linear
    launches.  Returns None unless the count is 1 + 4 * layers."""
    n = len(mss)
    if n < 5 or (n - 1) % 4:
        return None
    kinds = ("qkv", "out_proj_residual", "fc1", "fc2_residual")
    acc = {k: [0.0, 0.0] for k in ("patch",) + kinds}
    acc["patch"] = [float(works[0]), float(mss[0])]
    for i in range(1, n):
        k = kinds[(i - 1) % 4]
        acc[k][0] += float(works[i])
        acc[k][1] += float(mss[i])
    out = {k: (w / (t * 1e-3) / 1e12 if t > 0 else None) for k, (w, t) in acc.items()}
    plain_w = sum(acc[k][0] for k in ("patch", "qkv", "fc1"))
    plain_t = sum(acc[k][1] for k in ("patch", "qkv", "fc1"))
    out["without_residual_epilogue"] = plain_w / (plain_t * 1e-3) / 1e12 if plain_t > 0 else None
    out["ms"] = {k: t for k, (w, t) in acc.items()}
    return out


def run_b200(args):
    if args.no_graph:
        os.environ["FVS_VIT_GRAPH"] = "0"
    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert torch.cuda.is_available(), "bench.py --impl b200 needs a GPU (there is no CPU fallback)"
    torch.set_grad_enabled(False)     # inference, like every caller of this path in the reference (torch.inference_mode())
    # ONE sampler for the node, started now: model build + warm-up put >= 2 s between its start and the first timed region
    sampler = ClockSampler(enabled=(rank == 0 and not args.no_sampler))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from flash_vstream_b200 import _lib
    from flash_vstream_b200.clip_encoder import CLIPVisionTower
    from flash_vstream_b200.distributed import PrefixGather
    from flash_vstream_b200.vstream_arch import FlashVStreamB200, NeuralTuringMachine
    from oracle import fvs_oracle as O          # only for the seeded synthetic WEIGHTS generator and the cpu_baseline leg
    from tests import golden_inputs as GI

    lib = _lib.load(build_if_missing=False)
    cfg = O.VitConfig()
    w = O.random_vit_weights(cfg, 0)     # random-init ViT-L/14-336, all 24 layers (no checkpoints offline)
    tower = CLIPVisionTower.from_weights(w, select_layer=-2, max_batch=args.microbatch, device=dev)
    del w
    # hidden_states[-2] of a 24-layer tower = 23 executed layers = the 366 GFLOP/frame of SURVEY.md §8d.  (Rounds 1's bench
    # handed the tower a 23-layer weight dict, for which select_layer=-2 means 22 layers: its numbers were one layer short.)
    assert tower.engine.layers_run == 23, tower.engine.layers_run
    ntm = NeuralTuringMachine(1024, 32)
    GI.load_ntm(ntm, 0)
    model = FlashVStreamB200(tower, ntm.half().to(dev))
    model.fvs_fused_stream = not args.op_by_op
    model.fvs_chunk_cap = max(args.chunk, 1)
    chunk, K, W = args.chunk, args.steps, args.warmup

    # synthetic stream: a pool of distinct clips is cycled so no step re-reads a hot input
    # (SURVEY.md §8d: piecewise-stationary frames — scene_k + 0.1 randn, a new scene every 16-64 frames — so that the k-means
    # has structure; the ViT's cost does not depend on the data)
    n_clips = 4
    stream_px = GI.scene_pixels(n_clips * chunk, 1234 + rank)
    host_clips = [stream_px[i * chunk:(i + 1) * chunk].half().pin_memory() for i in range(n_clips)]
    del stream_px
    dev_clips = [c.to(dev) for c in host_clips]

    # RNG draws of every step, prepared up front (device resident) so the timed region has no host RNG work; the working-set
    # size of step s of a fresh stream is host-known: chunk, then min(long, 25) + chunk
    def stream_draws(n_steps, seed0):
        out, n_long = [], 0
        for s in range(n_steps):
            T = n_long + chunk
            if s > 0 and T > 25:
                di, dr = GI.kmeans_draws(T, 25, seed0 + s)
                out.append((torch.from_numpy(di).to(dev), torch.from_numpy(dr).to(dev)))
                n_long = 25
            else:
                out.append(None)
                n_long = T
        return out

    gather = PrefixGather(681, 1024, torch.float16, dev) if world > 1 else None
    prefix_host = torch.empty(681, 1024, dtype=torch.float16).pin_memory()

    def query():
        """what a query costs on top of the stream: one all-gather of every rank's finished prefix (north_star: "NCCL
        all-gather only to assemble the final memory prefix for the single LLM decode")"""
        if gather is not None:
            gather(model.memory_prefix())

    # e2e: frames start in pinned HOST memory.  The H2D copy of clip s+1 is issued on a copy stream while clip s is being
    # encoded (double-buffered device staging), so every step's 21.7 MB upload happens inside the timed region but
    # overlaps compute, as a real frame-ingest loop would; the step's result (the memory prefix) is read back to the host.
    copy_stream = torch.cuda.Stream(device=dev)
    stage = [torch.empty(chunk, 3, 336, 336, dtype=torch.float16, device=dev) for _ in range(2)]
    copied = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    e2e_state = {"next": None}

    def issue_copy(s):
        b = s % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[b])                       # the encoder has finished reading this buffer
            stage[b].copy_(host_clips[s % n_clips], non_blocking=True)  # H2D of step s' inputs
            copied[b].record(copy_stream)
        e2e_state["next"] = s + 1

    def make_steps(draws):
        def step_resident(s):
            model.embed_video_streaming(dev_clips[s % n_clips].unsqueeze(0), draws=draws[s])
            if args.gather_every_step:
                query()

        def step_e2e(s):
            b = s % 2
            if e2e_state["next"] != s + 1 and e2e_state["next"] != s + 2:
                issue_copy(s)                                               # first step of a run: nothing prefetched yet
            cur = torch.cuda.current_stream()
            cur.wait_event(copied[b])
            if e2e_state["next"] == s + 1:
                issue_copy(s + 1)                                           # prefetch the next clip during this step's compute
            model.embed_video_streaming(stage[b].unsqueeze(0), draws=draws[s])
            consumed[b].record(cur)
            if args.gather_every_step:
                query()
            pre = model.memory_prefix()                                     # a view of the bank: no concatenation
            prefix_host[:pre.shape[0]].copy_(pre, non_blocking=True)        # D2H of the step's result
        return step_resident, step_e2e

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step_fn, n_steps, n_warm, profile, prof_every=4):
        """fresh stream; n_warm untimed + n_steps timed steps (+ one query at the end, inside the timed region).
        profile: every prof_every-th timed step replays the encoder's PROFILED graph (an event-record node before and after
        each tensor-core kernel, captured during the warm-up); the collect afterwards returns the last such step."""
        model.reset_video_stream()
        e2e_state["next"] = None
        n_rec = ((n_steps + prof_every - 1) // prof_every + 1) * ((chunk + args.microbatch - 1) // args.microbatch) * 100 + 64
        if profile:
            _lib.check(lib.fvs_prof_enable(n_rec))
            lib.fvs_prof_pause(1)
        for s in range(n_warm):
            if profile:
                lib.fvs_prof_pause(0 if s == n_warm - 1 else 1)     # the last warm-up step captures the profiled graph
            step_fn(s)
        if profile:
            lib.fvs_prof_pause(1)
        barrier()
        if profile:
            import ctypes as C0
            dump = ((C0.c_int32 * n_rec)(), (C0.c_float * n_rec)(), (C0.c_double * n_rec)())
            lib.fvs_prof_collect(*dump, n_rec)                          # drop the warm-up's records
        launches0 = lib.fvs_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_wall0 = time.time()
        e0.record()
        for s in range(n_steps):
            if profile:
                lib.fvs_prof_pause(0 if s % prof_every == prof_every // 2 else 1)
            step_fn(n_warm + s)
        if profile:
            lib.fvs_prof_pause(1)
        if not args.gather_every_step:
            query()
        e1.record()
        barrier()
        t_wall1 = time.time()
        ms = e0.elapsed_time(e1)
        launches = lib.fvs_launch_count() - launches0
        prof = None
        if profile:
            import ctypes as C
            kinds, mss, works = (C.c_int32 * n_rec)(), (C.c_float * n_rec)(), (C.c_double * n_rec)()
            got = lib.fvs_prof_collect(kinds, mss, works, n_rec)
            prof = (np.frombuffer(kinds, np.int32)[:got].copy(), np.frombuffer(mss, np.float32)[:got].copy(),
                    np.frombuffer(works, np.float64)[:got].copy())
            lib.fvs_prof_enable(0)
        per_rank = None
        if world > 1:
            # per-rank view (a slow or throttled GPU in the node shows up here; the reported time is the max over ranks)
            t = torch.tensor([ms], device=dev)
            allt = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(allt, t)
            per_rank = [float(x.item()) / n_steps for x in allt]
            ms = max(float(x.item()) for x in allt)
        return {"ms": ms, "launches": launches, "prof": prof, "wall": (t_wall0, t_wall1), "per_rank_ms": per_rank,
                "profiled_steps": len([s for s in range(n_steps) if s % prof_every == prof_every // 2])}

    prof_every = 4
    n_total = K + W
    draws = stream_draws(n_total, 9000)
    step_resident, step_e2e = make_steps(draws)
    res = timed(step_resident, K, W, profile=not args.no_prof, prof_every=prof_every)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model.video_embedding_memory)
    res_e2e = timed(step_e2e, K, W, profile=False)

    # ---- the all-gather alone (once per query): microseconds per call, events around 20 back-to-back calls
    allgather_us = None
    if gather is not None:
        for _ in range(3):
            query()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(20):
            query()
        b.record()
        barrier()
        t = torch.tensor([a.elapsed_time(b) / 20 * 1e3], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        allgather_us = float(t.item())

    # ---- steady state: the same step for >= steady_s seconds (power-capped clocks: the regime MEASURED_PEAKS.json's
    # bf16_tflops_sustained was taken in), per-launch events on every 8th step
    steady = None
    if args.steady_s > 0:
        n_st = max(K, int(args.steady_s * 1e3 / (res["ms"] / K)) + 1)
        d2 = stream_draws(n_st + 2, 17000)
        sr, _ = make_steps(d2)
        steady = timed(sr, n_st, 2, profile=not args.no_prof, prof_every=8)
        steady["n_steps"] = n_st

    sampler.stop()

    def clocks_of(r, gpu):
        return sampler.window(r["wall"][0], r["wall"][1], gpu, n_gpus=world)

    qwen_row = None
    if world > 1 and not args.no_extras:
        # BASELINE config 5 in its own shape: one Qwen stream-shard per GPU, nothing shared between ranks (weak scaling);
        # measured by EVERY rank after and outside the headline region, aggregated as N x frames per step / slowest rank's
        # median step
        try:
            from tests.gpu_qwen_stream_timing import measure as measure_qwen
            qwen_row = measure_qwen(depth=32, t_clip=8, steps=16, breakdown=False)
            ms = torch.tensor([qwen_row["ms_per_step_full_memory"]], device=dev, dtype=torch.float64)
        except Exception as e:
            qwen_row = {"error": repr(e)[:300]}
            ms = torch.tensor([float("inf")], device=dev, dtype=torch.float64)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        if "error" not in qwen_row:
            qwen_row["ms_per_step_full_memory_max_over_ranks"] = float(ms.item())
            qwen_row["frames_per_s_full_memory_all_ranks"] = world * 2 * 8 / float(ms.item()) * 1e3
            qwen_row["note"] = (f"Flash-VStream-Qwen streaming step on {world} independent stream-shards (no collective), "
                                f"bf16, 16-frame clips")

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk = peaks()

    def roofline_of(r, n_steps):
        if r["prof"] is None or not len(r["prof"][0]):
            return None, None
        kinds, mss, works = r["prof"]
        ok = mss >= 0
        lin, att = (kinds == 1) & ok, (kinds == 2) & ok
        step_ms = r["ms"] / n_steps
        # records = the LAST profiled step (a graph replay re-records its events); 23 attention launches per micro-batch
        sampled = max(1.0, float(att.sum()) / (23.0 * ((chunk + args.microbatch - 1) // args.microbatch)))
        roof = att_d = None
        if lin.any():
            ach = works[lin].sum() / (mss[lin].sum() * 1e-3) / 1e12
            roof = {"achieved": ach, "launches_timed": int(lin.sum()), "sampled_steps": sampled,
                    "profiled_steps_in_region": r["profiled_steps"],
                    "share_of_step": float(mss[lin].sum() / (step_ms * sampled))}
            try:
                roof["by_gemm"] = gemm_breakdown(list(mss[lin]), list(works[lin])) if sampled == 1.0 else None
            except Exception:
                roof["by_gemm"] = None
        if att.any():
            att_d = {"achieved_tflops": works[att].sum() / (mss[att].sum() * 1e-3) / 1e12,
                     "share_of_step": float(mss[att].sum() / (step_ms * sampled)), "launches_timed": int(att.sum())}
        return roof, att_d

    frames = chunk * K * world
    value = frames / (res["ms"] / 1e3)
    e2e_v = frames / (res_e2e["ms"] / 1e3)
    clocks = clocks_of(res, 0 if world == 1 else None)
    roof, att_d = roofline_of(res, K)
    extra = {}
    traffic = None
    tp = os.path.join(ROOT, "profiles", "linear_kernel_traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    if roof is not None:
        # the timed region is short (K steps): it runs at burst clocks, so the burst cuBLAS figure is the honest denominator;
        # the sustained one is quoted beside it and used for the steady-state pass below
        roof = {"bound": "tensor", "kernel": "fvs::gemm::linear_kernel (all 93 GEMMs/micro-batch)", "achieved": roof["achieved"],
                "peak": pk["tensor_burst"], "unit": "TFLOP/s", "frac": roof["achieved"] / pk["tensor_burst"], "traffic": traffic,
                "peak_source": f"MEASURED_PEAKS.json bf16_tflops (burst; {pk['source']}); timed region {res['ms'] / 1e3:.2f} s at "
                               f"{clocks.get('sm_mhz')} MHz",
                "frac_of_sustained": roof["achieved"] / pk["tensor"], "peak_sustained": pk["tensor"],
                "sustained_peak_clock_mhz": pk["sustained_clock_mhz"],
                "launches_timed": roof["launches_timed"], "sampled_steps": roof["sampled_steps"],
                "profiled_steps_in_region": roof["profiled_steps_in_region"],
                "how": "CUDA events as external event-record nodes of the encoder's graph (no eager launches in the timed region)",
                "share_of_step": roof["share_of_step"],
                # TFLOP/s per GEMM kind of the profiled step: the out-proj / fc2 launches also read-modify-write the fp32
                # residual stream (151 MB each, TMA reduce-add epilogue), so their time buys more than their 2MNK
                "by_gemm_tflops": roof.get("by_gemm")}
    whole = value / world * GFLOP_PER_FRAME / 1e3      # TFLOP/s of the whole path per GPU
    extra["whole_path"] = {"tflops_per_gpu": whole, "frac_of_burst": whole / pk["tensor_burst"], "frac_of_sustained": whole / pk["tensor"]}
    if att_d is not None:
        extra["attention"] = att_d
    if steady is not None:
        s_roof, s_att = roofline_of(steady, steady["n_steps"])
        s_val = chunk * steady["n_steps"] * world / (steady["ms"] / 1e3)
        s_whole = s_val / world * GFLOP_PER_FRAME / 1e3
        extra["steady_state"] = {
            "seconds": steady["ms"] / 1e3, "steps": steady["n_steps"], "value": s_val, "ms_per_step": steady["ms"] / steady["n_steps"],
            "clocks": clocks_of(steady, 0 if world == 1 else None),
            "gemm_tflops": s_roof and s_roof["achieved"], "gemm_frac_of_sustained": s_roof and s_roof["achieved"] / pk["tensor"],
            "gemm_share_of_step": s_roof and s_roof["share_of_step"], "attention": s_att,
            "whole_path_tflops_per_gpu": s_whole, "whole_path_frac_of_sustained": s_whole / pk["tensor"],
            **({"per_rank_ms": steady["per_rank_ms"]} if steady["per_rank_ms"] else {})}

    line = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world,
        "steps": K, "warmup": W, "ms_per_step": res["ms"] / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic",
        "config": {"workload": f"1k-frame 336x336 stream per GPU in {chunk}-frame clips, ViT-L/14 (23 layers run) + "
                               f"STAR Flash memory (681-token bank: 25 abstract + 25x16 long + 4x64 key/current)",
                   "chunk_frames": chunk, "vit_microbatch": args.microbatch, "vit_layers_run": int(tower.engine.layers_run),
                   "parallelism": f"stream-shard x{world}",
                   "step": "embed_video_streaming(pixels): ViT layer stack as one CUDA graph, STAR levels pooled in the encoder tail, "
                           "one fused consolidation kernel on the persistent bank" if not args.op_by_op else "op-by-op consolidation",
                   "collective": ("all-gather after every step (ablation)" if args.gather_every_step else
                                  "none per step; one prefix all-gather per query, inside the timed region once") if world > 1 else "none",
                   "residual_stream": "fp32", "l2": "per-step working set (579 MB weights + activations) exceeds the "
                                                    "126 MB L2; inputs rotate over 4 clips; no explicit flush",
                   "ablations": {"gather_every_step": args.gather_every_step, "sampler": not args.no_sampler,
                                 "vit_graph": not args.no_graph, "fused_consolidation": not args.op_by_op}},
        "clocks": clocks,
        "e2e": {"value": e2e_v, "unit": "frames/s", "ms_per_step": res_e2e["ms"] / K,
                "h2d_bytes_per_step": int(chunk * 3 * 336 * 336 * 2), "d2h_bytes_per_step": int(681 * 1024 * 2)},
        "gpu_launches": int(res["launches"]),
        "roofline": roof,
    }
    if world > 1:
        line["per_rank"] = [{"rank": r, "ms_per_step": res["per_rank_ms"][r], "e2e_ms_per_step": res_e2e["per_rank_ms"][r],
                             **{k: v for k, v in clocks_of(res, r).items() if k in ("sm_mhz", "reasons")}} for r in range(world)]
        line["allgather_us"] = allgather_us
    line.update(extra)

    if world == 1 and not args.no_extras:
        line["rows"] = extra_rows(args, model, tower, dev, pk, lib, GI, torch)
    if qwen_row is not None:
        line["rows"] = {"qwen_stream": qwen_row}
    if not args.no_cpu_baseline and world == 1:
        try:
            ref = CpuReference()
            n = 16
            secs, vit_secs = ref.clip(n)
            line["cpu_baseline"] = {"value": n / secs, "unit": "frames/s", "cores": ref.cores, "kind": "port",
                                    "sample": f"one {n}-frame clip: 24-layer {ref.kind_vit} fp32 + f16 torch-CPU consolidation, "
                                              f"{secs:.1f} s of which ViT {vit_secs:.1f} s"}
        except Exception as e:
            line["cpu_baseline"] = {"error": repr(e)[:200]}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def extra_rows(args, model, tower, dev, pk, lib, GI, torch):
    """Other shapes of the same path at N=1, measured after and outside the headline region (never fatal for the line):
    chunk=1 (the reference's realtime loop feeds single frames, cli_video_stream.py:180-192), the 256-token bank of SURVEY.md
    §8d(2), the offline 1k-frame consolidation, and the library path (torch fp16 on this GPU) as an informational baseline."""
    rows = {}

    def ev_time(fn, n, warm=3):
        for i in range(warm):
            fn(i)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = lib.fvs_launch_count()
        a.record()
        for i in range(n):
            fn(warm + i)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n, (lib.fvs_launch_count() - n0) / n

    frames = GI.scene_pixels(64, 77).half().to(dev)
    # ---- chunk = 1: per-frame latency of the whole step, and of the consolidation alone
    try:
        draws1 = [None] * 25 + [tuple(torch.from_numpy(d).to(dev) for d in GI.kmeans_draws(26, 25, 500 + s)) for s in range(400)]
        model.reset_video_stream()
        ms1, l1 = ev_time(lambda i: model.embed_video_streaming(frames[i % 64:i % 64 + 1].unsqueeze(0), draws=draws1[min(i, 425)]), 200, warm=30)
        info1 = model._fvs_bank.info()[1].cpu().tolist()
        # consolidation alone on structured features (SURVEY.md §8d: piecewise-stationary, unit scale — the k-means converges in
        # 2-3 Lloyd iterations like on real video); the random-weight ViT's own features overflow the f16 distance sums
        # (-> inf, ties) and run all 10 iterations with refills, which is the worst case and is what the pixel rows above pay
        sf = GI.scene_features(232, 576, 1024, 5, scene_len=(16, 64)).to(dev)      # no frame repeats: 30 warm-up + 200 timed steps
        model.reset_video_stream()
        msc, lc = ev_time(lambda i: model.consolidate_streaming(sf[i:i + 1], draws=draws1[min(i, 425)]), 200, warm=30)
        infoc = model._fvs_bank.info()[1].cpu().tolist()
        feats = tower(frames[:8])
        model.reset_video_stream()
        msw, _ = ev_time(lambda i: model.consolidate_streaming(feats[i % 8:i % 8 + 1], draws=draws1[min(i, 425)]), 200, warm=30)
        per = CONSOLIDATION_BYTES_PER_FRAME
        rows["chunk1"] = {"frames_per_s": 1e3 / ms1, "ms_per_frame": ms1, "launches_per_frame": l1,
                          "whole_path_tflops": GFLOP_PER_FRAME / ms1 / 1e3, "kmeans_exit_step_refills": info1[:2],
                          "consolidation_ms": msc, "consolidation_launches": lc, "consolidation_gbps": per / msc / 1e6,
                          "consolidation_hbm_frac": per / msc / 1e6 / pk["hbm"], "consolidation_kmeans_exit_step_refills": infoc[:2],
                          "consolidation_ms_worst_case_10_iterations": msw,
                          "note": "single-frame steps (M = 577 rows): weight streaming (579 MB/frame) and launch latency bound; "
                                  "consolidation = pool3 + ONE fused kernel (2 launches)"}
    except Exception as e:
        rows["chunk1"] = {"error": repr(e)[:300]}
    # ---- consolidation alone at the headline clip length
    try:
        chunk = args.chunk
        feats = GI.scene_features(chunk, 576, 1024, 6, scene_len=(16, 64)).to(dev)
        drawsC = [None, None] + [tuple(torch.from_numpy(d).to(dev) for d in GI.kmeans_draws(25 + chunk, 25, 900 + s)) for s in range(40)]
        drawsC[1] = tuple(torch.from_numpy(d).to(dev) for d in GI.kmeans_draws(2 * chunk, 25, 899)) if 2 * chunk > 25 else None
        model.reset_video_stream()
        msc, lc = ev_time(lambda i: model.consolidate_streaming(feats, draws=drawsC[min(i, 41)]), 20, warm=4)
        b = CONSOLIDATION_BYTES_PER_FRAME * chunk
        rows["consolidation"] = {"chunk_frames": chunk, "ms_per_step": msc, "launches_per_step": lc, "achieved_gbps": b / msc / 1e6,
                                 "peak_gbps": pk["hbm"], "frac": b / msc / 1e6 / pk["hbm"],
                                 "note": "pool3 + one fused kernel (k-means over 25+chunk rows, abstract, retrieve, write-back)"}
    except Exception as e:
        rows["consolidation"] = {"error": repr(e)[:300]}
    # ---- 256-token bank (3 current frames @8x8 + 64 abstract tokens, no long memory), chunk 32
    try:
        from flash_vstream_b200.vstream_arch import FlashVStreamB200
        m256 = FlashVStreamB200(tower, model.get_model().attention_model, video_long_memory_length=0,
                                video_Turing_memory_length=64, video_current_memory_length=3)
        ms256, l256 = ev_time(lambda i: m256.embed_video_streaming(frames[(i % 2) * 32:(i % 2) * 32 + 32].unsqueeze(0)), 10, warm=3)
        rows["bank256"] = {"frames_per_s": 32e3 / ms256, "ms_per_step": ms256, "launches_per_step": l256,
                           "prefix_rows": int(m256.memory_prefix().shape[0]),
                           "config": "video_long_memory_length=0, video_Turing_memory_length=64, video_current_memory_length=3"}
    except Exception as e:
        rows["bank256"] = {"error": repr(e)[:300]}
    # ---- offline: one 1000-frame video through compress_temporal_features (the shape §8d quotes the HBM fraction on)
    try:
        from tests.gpu_offline_timing import measure as measure_offline
        rows["offline_1k_frames"] = measure_offline(pk["hbm"])
    except Exception as e:
        rows["offline_1k_frames"] = {"error": repr(e)[:300]}
    # ---- BASELINE config 5's shape on one GPU (one stream-shard of the Qwen variant): 336 px stream, 8-patch (16-frame) clips
    # through embed_new_video_clip = temporal_pool + 32-layer head_dim-80 tower + CSM k-means + DAM retrieval + PatchMerger
    try:
        from tests.gpu_qwen_stream_timing import measure as measure_qwen
        q = measure_qwen(depth=32, t_clip=8, steps=20, breakdown=False)
        q["note"] = ("Flash-VStream-Qwen streaming step, bf16, pixels from pinned host memory, memory full (60 CSM + 30 DAM frames -> "
                     "6480 merged tokens); a 20-step stream (the DAM retrieval reads the whole low-resolution bank, which grows by "
                     "368 KB per temporal patch: see qwen_stream_10k_frames)")
        rows["qwen_stream"] = q
    except Exception as e:
        rows["qwen_stream"] = {"error": repr(e)[:300]}
    try:
        # the same step 10 k frames into the stream (BASELINE config 5's length): the banks are pre-filled with synthetic
        # features (5000 temporal patches = 14 GB), so the DAM retrieval sweeps a 1.8 GB half-resolution bank per step
        q = measure_qwen(depth=32, t_clip=8, steps=20, breakdown=False, prefill_patches=4992)
        q["note"] = "as qwen_stream, with the feature banks of a stream that is 10 k frames long (pre-filled with synthetic features)"
        rows["qwen_stream_10k_frames"] = q
    except Exception as e:
        rows["qwen_stream_10k_frames"] = {"error": repr(e)[:300]}
    # ---- the library path on this GPU: HF CLIPVisionModel fp16 (SDPA) + the consolidation in plain torch ops
    try:
        rows["torch_gpu"] = torch_gpu_row(args, dev, frames, GI, torch)
    except Exception as e:
        rows["torch_gpu"] = {"error": repr(e)[:300]}
    return rows


def torch_gpu_row(args, dev, frames, GI, torch):
    """Informational: what the reference's own PyTorch code path reaches on this B200 (SURVEY.md §2.2) — transformers'
    CLIPVisionModel in fp16 through the clip_encoder.py:41-53 call shape (24 layers, output_hidden_states=True) and the
    consolidation as whole-tensor torch ops on the GPU (the op granularity of vstream_arch.py:644-697).  Library kernels
    (cuBLAS, SDPA); never a substitute for the --impl reference CPU arm."""
    from transformers import CLIPVisionConfig, CLIPVisionModel
    from oracle import fast_cpu as FC
    from oracle import fvs_oracle as O
    cfg = O.VitConfig()
    w = O.random_vit_weights(cfg, 0)
    hf_cfg = CLIPVisionConfig(hidden_size=cfg.hidden, intermediate_size=cfg.mlp, num_hidden_layers=cfg.layers,
                              num_attention_heads=cfg.heads, image_size=cfg.image_size, patch_size=cfg.patch_size)
    hf = CLIPVisionModel(hf_cfg).eval()
    hf.load_state_dict(O.hf_state_dict(w, cfg), strict=False)
    hf = hf.half().to(dev)
    wn = GI.ntm_weights(1024, 32, 0)
    ntm = tuple(wn[k].to(dev) for k in ("q_w", "q_b", "k_w", "k_b"))
    chunk = args.chunk
    state = FC.State()
    clip = frames[:chunk]

    def step(i):
        nonlocal state
        with torch.no_grad():
            f = hf(clip, output_hidden_states=True).hidden_states[-2][:, 1:]
        dn = GI.kmeans_draws(25 + chunk, 25, 300 + i) if state.buf is not None else (None, None)
        state = FC.stream_step(state, FC.pool(f, 8), ntm, dn[0], dn[1])

    def enc(i):
        with torch.no_grad():
            hf(clip, output_hidden_states=True).hidden_states[-2][:, 1:]

    def timeit(fn, n, warm):
        for i in range(warm):
            fn(i)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(n):
            fn(warm + i)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n

    ms_enc = timeit(enc, 8, 3)
    ms_step = timeit(step, 8, 3)
    return {"frames_per_s": chunk * 1e3 / ms_step, "ms_per_step": ms_step, "encode_only_ms": ms_enc,
            "encode_only_frames_per_s": chunk * 1e3 / ms_enc, "chunk_frames": chunk,
            "what": "transformers CLIPVisionModel fp16 (24 layers, attn via the installed transformers' default = SDPA) + "
                    "torch-op consolidation on the GPU with per-step host RNG draws; library kernels, same 32-frame clips"}


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
