#!/usr/bin/env python
"""Benchmark of the B200-native 4M hot path (contract: see the task statement / DESIGN.md "Measurement").

    python bench.py --gpus 1 --steps 20 --warmup 5                     # one GPU
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W                      # N GPUs, one rank each (data parallel, NCCL)
    python bench.py --impl reference --steps 2 --warmup 1              # the reference algorithm on the host CPU cores
    python bench.py --steps 20 --warmup 5 --dump-outputs DIR          # also writes the last timed step's outputs as DIR/*.npy

A step = one full training step of 4M-B mod7 (BASELINE.json configs[1]): forward + backward + gradient all-reduce (DDP)
+ AdamW, per-GPU batch 128, 128 encoder + 128 decoder tokens per sample, synthetic data, random-init weights.
Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "ml-4m_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402

MODEL = "fm_base_12e_12d_swiglu_nobias"
# driver-measurable workloads (BASELINE.json configs[1], [2], [4]; configs[3] = `gen`): per-GPU batch and token budget are the
# reference configs' (cfgs/default/4m/models/main/4m-{b,l}_mod7_500b.yaml:28)
WORKLOADS = {
    "4m-b": dict(model="fm_base_12e_12d_swiglu_nobias", batch=128, tokens=128, D=768, Le=12, Ld=12, H=2048,
                 name="4M-B mod7 full train step (fwd+bwd+gradient all-reduce+AdamW), BASELINE.json configs[1]"),
    "4m-l": dict(model="fm_large_24e_24d_swiglu_nobias", batch=64, tokens=256, D=1024, Le=24, Ld=24, H=2730,
                 name="4M-L mod7 full train step (fwd+bwd+gradient all-reduce+AdamW), 256+256 tokens, BASELINE.json configs[2]"),
}


def vbar(n_tok):
    """token-weighted mean target vocabulary of the synthetic mod-7 batch (SURVEY.md 8d)."""
    from b200fm.synthetic import budgets_for
    _, _, n_img, n_seq = budgets_for(n_tok)
    return ((16384 + 8192 + 8192 + 4096 + 8192) * n_img + 2 * 30000 * (n_seq - 1)) / n_tok


def flops_per_sample_fwd(N, M, D=768, Le=12, Ld=12, H=2048):
    """SURVEY.md 8d algorithmic FLOPs (multiply-add = 2)."""
    enc = 8 * N * D * D + 4 * N * N * D + 6 * N * D * H
    dec = (8 * M * D * D + 4 * M * M * D) + (4 * M * D * D + 4 * N * D * D + 4 * M * N * D) + 6 * M * D * H
    blocks = Le * enc + Ld * dec
    extras = 2 * N * D * D + 2 * M * D * vbar(M) + 2 * 196 * 768 * D
    return blocks, blocks + extras


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(bf16=float(p.get("bf16_tflops_sustained", p.get("bf16_tflops", 1590.0))), hbm=float(p.get("hbm_gbs", 6650.0)), src="measured")
    return dict(bf16=1400.0, hbm=6650.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md clocks line)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        mx = max((int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()), default=None)
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


# ----------------------------------------------------------------------------------------------------------------------
# the reference algorithm on the host CPU (oracle port): cpu_baseline leg and `--impl reference`
# ----------------------------------------------------------------------------------------------------------------------
def cpu_threads():
    """Thread count for the CPU arm when not auto-tuned (B200FM_CPU_THREADS overrides)."""
    env = os.environ.get("B200FM_CPU_THREADS")
    return int(env) if env else min(os.cpu_count() or 1, 16)


def gemm_traffic_per_launch():
    """DRAM bytes (read + write) per GEMM launch of a 4M-B step, from the committed ncu capture (never measured in this process)."""
    for name in ("r2_step_traffic.json", "r1_step_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                return float(json.load(f)["gemm"]["dram_bytes_per_launch"]), name
        except (OSError, KeyError, ValueError):
            continue
    return None, None


def reference_tree():
    """Path of the unmodified apple/ml-4m tree when it is present (authoring container), else None (GPU box)."""
    root = os.environ.get("ML4M_REFERENCE", "/root/reference")
    return root if os.path.isdir(os.path.join(root, "fourm", "models")) else None


def _import_real_reference():
    """Make `fourm` resolve to the unmodified tree (drop the overlay from sys.path / sys.modules) and import it with the shims of
    tests/golden/ref_import.py.  Only the `--impl reference` arm calls this; it never runs in the same process as the B200 arm."""
    from b200fm.synthetic import budgets_for  # noqa: F401  (pure python; imported before the overlay directory leaves sys.path)
    pkg = os.path.join(ROOT, "ml-4m_b200")
    sys.path[:] = [p for p in sys.path if os.path.abspath(p) != pkg]
    for k in [k for k in sys.modules if k == "fourm" or k.startswith("fourm.")]:
        del sys.modules[k]
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import ref_import
    return ref_import.import_reference_models()


def cpu_real_reference_steps(steps, warmup, sample_B, n_tok, model_name):
    """Times fwd+bwd of the UNMODIFIED reference `FourM.forward` (fm.py:640-691) on the host CPU, fp32 -- only where the
    reference tree exists (it cannot travel to the GPU box); `kind: "reference"`."""
    import random
    from b200fm.synthetic import budgets_for
    fm, fm_utils, MODALITY_INFO = _import_real_reference()
    from make_golden import build_reference_fourm, clone_batch
    from oracle import fourm_oracle as O
    torch.set_num_threads(cpu_threads())
    torch.manual_seed(0)
    model = build_reference_fourm(model_name, O.mod7_specs(), MODALITY_INFO)
    batch = O.synthetic_mod7_batch(sample_B, *budgets_for(n_tok), seed=1234)
    times = []
    for it in range(warmup + steps):
        random.seed(it)
        t0 = time.perf_counter()
        loss, _ = model(clone_batch(batch), num_encoder_tokens=n_tok, num_decoder_tokens=n_tok, loss_type="mod")
        loss.backward()
        dt = time.perf_counter() - t0
        model.zero_grad(set_to_none=True)
        if it >= warmup:
            times.append(dt)
    sec = sum(times) / len(times)
    return sample_B * 2 * n_tok / sec, sec, torch.get_num_threads()


def cpu_reference_steps(steps, warmup, sample_B, n_tok, threads=None, model_name=MODEL):
    """Times fwd+bwd of the oracle restatement of FourM.forward (mod7, fp32, host threads per cpu_threads())."""
    import random
    from oracle import fourm_oracle as O
    torch.set_num_threads(threads or cpu_threads())
    specs = O.mod7_specs()
    cfg = O.PRESETS[model_name]
    g = torch.Generator().manual_seed(0)
    sd = {}
    D = cfg["dim"]

    def w(*shape, std=0.02):
        return (torch.randn(*shape, generator=g) * std).requires_grad_(True)
    for name, s in specs.items():
        for side in ("encoder_embeddings", "decoder_embeddings"):
            if side == "decoder_embeddings" and s["kind"] == "img":
                continue
            p = f"{side}.{name}."
            sd[p + "mod_emb"] = w(1, 1, D) if side == "encoder_embeddings" else sd[f"encoder_embeddings.{name}.mod_emb"]
            sd[p + "pos_emb"] = O.sincos_1d(512, D) if s["kind"] == "seq" else O.sincos_2d(14, 14, D)
            if s["kind"] == "img":
                sd[p + "proj.weight"] = w(D, 768)
            else:
                sd[p + "token_emb.weight"] = w(s["vocab"], D)
                if side == "decoder_embeddings":
                    sd[p + "to_logits.weight"] = sd[p + "token_emb.weight"]
    H = int(2 * 4 * D / 3)
    for i in range(cfg["enc_depth"]):
        p = f"encoder.{i}."
        for n in ("norm1", "norm2"):
            sd[p + n + ".weight"] = torch.ones(D, requires_grad=True); sd[p + n + ".bias"] = torch.zeros(D)
        sd[p + "attn.qkv.weight"] = w(3 * D, D); sd[p + "attn.proj.weight"] = w(D, D)
        sd[p + "mlp.fc1.weight"] = w(H, D); sd[p + "mlp.fc3.weight"] = w(H, D); sd[p + "mlp.fc2.weight"] = w(D, H)
    for i in range(cfg["dec_depth"]):
        p = f"decoder.{i}."
        for n in ("norm1", "norm2", "query_norm", "context_norm"):
            sd[p + n + ".weight"] = torch.ones(D, requires_grad=True); sd[p + n + ".bias"] = torch.zeros(D)
        sd[p + "self_attn.qkv.weight"] = w(3 * D, D); sd[p + "self_attn.proj.weight"] = w(D, D)
        sd[p + "cross_attn.q.weight"] = w(D, D); sd[p + "cross_attn.kv.weight"] = w(2 * D, D); sd[p + "cross_attn.proj.weight"] = w(D, D)
        sd[p + "mlp.fc1.weight"] = w(H, D); sd[p + "mlp.fc3.weight"] = w(H, D); sd[p + "mlp.fc2.weight"] = w(D, H)
    for n in ("encoder_norm", "decoder_norm"):
        sd[n + ".weight"] = torch.ones(D, requires_grad=True); sd[n + ".bias"] = torch.zeros(D)
    sd["decoder_proj_context.weight"] = w(D, D); sd["decoder_proj_context.bias"] = torch.zeros(D, requires_grad=True)
    sd["mask_token"] = w(1, 1, D)
    from b200fm.synthetic import budgets_for
    a, b, c, d = budgets_for(n_tok)
    batch = O.synthetic_mod7_batch(sample_B, a, b, c, d, seed=1234)
    dec_names = [m for m, s in specs.items() if s["kind"] != "img"]
    leaves = [t for t in {id(v): v for v in sd.values()}.values() if t.requires_grad]

    def one(it):
        random.seed(it)
        order = random.sample(dec_names, len(dec_names))
        t0 = time.perf_counter()
        loss, _ = O.fourm_forward(sd, cfg, specs, batch, n_tok, n_tok, order)
        loss.backward()
        dt = time.perf_counter() - t0
        for t in leaves:
            t.grad = None
        return dt

    if threads is None and not os.environ.get("B200FM_CPU_THREADS"):
        # the reference gets the thread count that serves it best on this host: on the GPU box (128 hardware threads) 16 torch
        # threads are ~3x faster than 64 and ~25x faster than 128 for these fp32 sizes (measured, profiles/README.md)
        ncpu = os.cpu_count() or 1
        best = None
        one(0)                                           # first-touch / allocator warm-up
        for cand in sorted({min(ncpu, c) for c in (8, 16, 32, 64)}):
            torch.set_num_threads(cand)
            dt = one(0)
            if best is None or dt < best[0]:
                best = (dt, cand)
        torch.set_num_threads(best[1])
    times = []
    for it in range(warmup + steps):
        random.seed(it)
        order = random.sample(dec_names, len(dec_names))
        t0 = time.perf_counter()
        loss, _ = O.fourm_forward(sd, cfg, specs, batch, n_tok, n_tok, order)
        loss.backward()
        dt = time.perf_counter() - t0
        for t in leaves:
            t.grad = None
        if it >= warmup:
            times.append(dt)
    tok = sample_B * 2 * n_tok
    return tok / (sum(times) / len(times)), sum(times) / len(times), torch.get_num_threads()


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload in ("vq-tokenize", "vqvae-train"):
        return run_vq_reference_arm(args)
    if args.workload == "gen":
        return run_gen_reference_arm(args)
    wl = WORKLOADS[args.workload]
    n_tok = wl["tokens"]
    B = 8 if args.workload == "4m-b" else 2
    if reference_tree() is not None and not os.environ.get("B200FM_CPU_PORT"):
        tps, sec, cores = cpu_real_reference_steps(args.steps, args.warmup, B, n_tok, wl["model"])
        kind, what = "reference", "the unmodified reference FourM.forward (fourm/models/fm.py:640-691)"
    else:
        tps, sec, cores = cpu_reference_steps(args.steps, args.warmup, B, n_tok, model_name=wl["model"])
        kind, what = "port", "oracle port of FourM.forward"
    line = dict(metric="tokens_per_sec", value=tps, unit="tokens/s", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=sec * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                impl="reference",
                config=dict(workload=f"{wl['name'].split(' (')[0]} fwd+bwd ({what} on host CPU, fp32)", model=wl["model"],
                            global_batch=B, seq_len=2 * n_tok, parallelism="cpu"),
                cpu_baseline=dict(value=tps, unit="tokens/s", cores=cores, kind=kind,
                                  sample=f"fwd+bwd of B={B} samples x {2 * n_tok} tokens per step, fp32, torch CPU {cores} threads of {os.cpu_count()}"),
                e2e=dict(value=tps, unit="tokens/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------------------
# B200 arm
# ----------------------------------------------------------------------------------------------------------------------
PARAM_SAMPLE = 1 << 21          # parameter values written by --dump-outputs (8 MB of float32)


def dump_outputs(out_dir, loss, mod_loss, gnorm, model):
    """Writes what one train step returns (loss, per-modality losses, gradient norm) and a fixed, seeded sample of the parameters it
    updated to out_dir/<name>.npy as float32, so that two builds run with the same arguments can be compared array by array."""
    import numpy as np
    arrays = {"loss": loss, "grad_norm": gnorm, **{f"mod_loss.{m}": v for m, v in mod_loss.items()}}
    flat = torch.cat([p.detach().reshape(-1).float() for p in model.parameters()])
    idx = torch.randint(0, flat.numel(), (min(PARAM_SAMPLE, flat.numel()),), generator=torch.Generator().manual_seed(0)).sort().values
    arrays["params_sample"] = flat[idx.to(flat.device)]
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def run_b200_arm(args):
    import torch.distributed as dist
    from b200fm import lib, ops
    from b200fm.compat import build_mod7_embeddings, create_model
    from b200fm.data import DevicePrefetcher
    from b200fm.optim import FusedAdamW, param_groups_like_reference
    from b200fm.synthetic import batch_bytes, budgets_for, mod7_batch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py (B200 arm) needs a GPU; there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib.load()

    wl = WORKLOADS[args.workload]
    B = args.batch or wl["batch"]
    n_tok = args.tokens or wl["tokens"]
    args.model = args.model or wl["model"]
    torch.manual_seed(0)
    enc, dec, info = build_mod7_embeddings()
    model = create_model(args.model, encoder_embeddings=enc, decoder_embeddings=dec, modality_info=info).to(dev)
    n_params = sum(p.numel() for p in model.parameters())
    lr = 1e-4 * B * world / 256                                 # run_training_4m.py:496-503 scaling rule
    groups = param_groups_like_reference(model, 0.05)
    net, gsync, comm = model, None, "none"
    if world > 1:
        comm = os.environ.get("B200FM_COMM", "p2p")
        if comm == "ddp":            # round-1 path, kept for A/B: torch DDP buckets + NCCL all-reduce
            net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local], find_unused_parameters=False,
                                                            gradient_as_bucket_view=True, broadcast_buffers=False,
                                                            bucket_cap_mb=int(os.environ.get("B200FM_DDP_BUCKET_MB", "25")))
        else:                        # gradient arena + NVLink peer-memory all-reduce kernel (b200fm.parallel / csrc/comm.cu)
            from b200fm.parallel import GradSync
            try:
                net = gsync = GradSync(model, transport=comm, wait_at_end=False)
            except Exception as exc:      # e.g. CUDA IPC not permitted between the ranks' containers: NCCL on the arena chunks instead
                print(f"[bench] GradSync transport '{comm}' unavailable ({exc!r}); falling back to 'collective'", file=sys.stderr)
                comm = "collective"
                net = gsync = GradSync(model, transport=comm, wait_at_end=False)
            groups = gsync.split_param_groups(groups)
    # whole-step CUDA graph (b200fm.graph): the step is captured once and replayed; B200FM_GRAPH=0 issues every launch from Python
    use_graph = os.environ.get("B200FM_GRAPH", "1") != "0" and comm != "ddp"
    opt = FusedAdamW(groups, lr=lr, betas=(0.9, 0.95), eps=1e-8, capturable=use_graph)
    if gsync is not None:
        opt.pre_group_hook = gsync.wait
    gstep = None
    if use_graph:
        from b200fm.graph import GraphedTrainStep
        gstep = GraphedTrainStep(net, opt, n_tok, n_tok, loss_type="mod")
    import random
    random.seed(rank)
    a, b, c, d = budgets_for(n_tok)
    host_batches = [mod7_batch(B, a, b, c, d, seed=1234 + rank + 17 * i, pin_memory=True) for i in range(2)]
    dev_batches = [{m: {k: v.to(dev) for k, v in dd.items()} for m, dd in hb.items()} for hb in host_batches]
    h2d = batch_bytes(host_batches[0])

    def step(batch):
        return gstep(batch) if gstep is not None else eager_step(batch)

    def eager_step(batch):
        if opt.capturable:
            opt.prepare_step()
        loss, mod_loss = net(batch, num_encoder_tokens=n_tok, num_decoder_tokens=n_tok, loss_type="mod")
        loss.backward()
        # AdamW of the early chunks runs while the last chunk is still being reduced; the logged gradient norm (native_scaler.py:56-65; no
        # clipping in the reference config: run_training_4m.py:102 clip_grad None) is accumulated by the AdamW kernels themselves
        opt.track_grad_norm = True
        opt.step()
        gnorm = opt.grad_norm()
        opt.zero_grad(set_to_none=True)
        return loss, mod_loss, gnorm

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # one staging stream for every end-to-end pass: the allocator's per-stream pool of batch-sized blocks is filled once (by the untimed
    # end-to-end warm-up below), not inside the timed region
    stage_stream = torch.cuda.Stream(device=dev)
    LAG = 2      # the host reads step i's loss while steps i+1 and i+2 are already queued (one step of slack against host hiccups)
    loss_host = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(LAG + 1)]
    loss_evt = [torch.cuda.Event() for _ in range(LAG + 1)]

    def timed(n_steps, e2e, step=step, host_batches=host_batches):
        calls0 = lib.CALLS["n"]
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        last = None
        t_cpu0 = time.perf_counter()
        if e2e:
            # every step's batch is copied from pinned host memory inside the timed region, one batch ahead on a side stream
            # device -> host read of EVERY step's loss, pipelined: step i's loss travels to pinned memory and is read by the host
            # while the next LAG steps are already queued (a blocking .item() would drain the GPU once per step)
            i = 0
            for batch in DevicePrefetcher((host_batches[i % 2] for i in range(n_steps)), dev, depth=LAG + 1, stream=stage_stream):
                loss, mod_loss, gnorm = step(batch)
                loss_host[i % (LAG + 1)].copy_(loss.detach().reshape(1), non_blocking=True)
                loss_evt[i % (LAG + 1)].record()
                if i >= LAG:
                    loss_evt[(i - LAG) % (LAG + 1)].synchronize()
                    last = float(loss_host[(i - LAG) % (LAG + 1)])
                i += 1
            for j in range(max(0, i - LAG), i):                       # drain: the last LAG losses
                loss_evt[j % (LAG + 1)].synchronize()
                last = float(loss_host[j % (LAG + 1)])
        else:
            for i in range(n_steps):
                loss, mod_loss, gnorm = step(dev_batches[i % 2])
        e1.record()
        timed.cpu_ms = (time.perf_counter() - t_cpu0) * 1e3 / n_steps       # host time to ISSUE a step (no sync inside)
        sync()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        n_calls = lib.CALLS["n"] - calls0
        if gstep is not None and gstep.graph is not None:
            n_calls += gstep.kernel_calls_per_step * n_steps        # launches replayed from the captured graph
        timed.outputs = (loss, mod_loss, gnorm)                      # the last step's results, valid until the next step
        return ms, n_calls, (last if last is not None else float(loss.item()))

    for _ in range(max(args.warmup, 3)):
        step(dev_batches[0])
    if os.environ.get("B200FM_NCU_ONE_STEP"):      # ncu --profile-from-start off: exactly one steady-state step is profiled
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        eager_step(dev_batches[1])
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms, launches, loss_val = timed(args.steps, e2e=False)
    cpu_issue_ms = timed.cpu_ms
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *timed.outputs, model)
    # end to end.  Wire format of the RGB modality: "uint8" (default) ships the raw 8-bit pixels and applies the loader's ToTensor +
    # Normalize inside the patchify kernel (fourm/models/encoder_embeddings.py, b200fm.masking): 22 MB per step over PCIe instead of the
    # 80 MB of the reference's fp32 wire format, which is measured as well (`e2e_fp32_wire`).  Same step otherwise.
    e2e_wire = os.environ.get("B200FM_E2E_WIRE", "uint8")
    timed(max(args.warmup, 3), e2e=True)                       # untimed: staging stream / pinned-copy path / read-back ring warm
    ms_e2e_f32, _, loss_e2e = timed(args.steps, e2e=True)
    ms_e2e, h2d_e2e = ms_e2e_f32, h2d
    if e2e_wire == "uint8":
        gu = torch.Generator().manual_seed(99 + rank)
        hb_u8 = []
        for hb in host_batches:
            nb = {m: dict(dd) for m, dd in hb.items()}
            shp = hb["rgb@224"]["tensor"].shape
            nb["rgb@224"]["tensor"] = torch.randint(0, 256, shp, dtype=torch.uint8, generator=gu).pin_memory()
            hb_u8.append(nb)
        step_u8 = eager_step
        if use_graph:
            gstep_u8 = GraphedTrainStep(net, opt, n_tok, n_tok, loss_type="mod")
            step_u8 = gstep_u8
        dev_u8 = {m: {k: v.to(dev) for k, v in dd.items()} for m, dd in hb_u8[0].items()}
        for _ in range(4):                                    # 2 eager calls + the capture + 1 replay
            step_u8(dev_u8)
        timed(max(args.warmup, 3), e2e=True, step=step_u8, host_batches=hb_u8)      # untimed warm-up of this wire format
        ms_e2e, _, loss_e2e = timed(args.steps, e2e=True, step=step_u8, host_batches=hb_u8)
        h2d_e2e = batch_bytes(hb_u8[0])
        if use_graph:
            gstep_u8.release()
    clocks = sampler.stop() if rank == 0 else None
    ms_nocomm, params_equal = None, None
    if world > 1:
        # every rank must hold bit-identical parameters after the synchronised steps (checked BEFORE the unsynchronised timing below)
        if gsync is not None:
            params_equal = gsync.params_equal_across_ranks()
        else:
            acc = torch.stack([p.detach().double().sum() for p in model.parameters()]).sum().reshape(1)
            lo, hi = acc.clone(), acc.clone()
            dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
            params_equal = bool(torch.equal(lo, hi))
        with net.no_sync():          # the same steps with the gradient all-reduce switched off: what the communication costs
            step_nc = eager_step
            if use_graph:            # (a second capture; the first graph is not replayed again after this point)
                g2 = GraphedTrainStep(net, opt, n_tok, n_tok, loss_type="mod", eager_steps=0)
                g2.eager_left = 0
                step_nc = g2
                step_nc(dev_batches[0])
            ms_nocomm, _, _ = timed(args.steps, e2e=False, step=step_nc)

    # roofline of the dominant kernel family (tcgen05 GEMM): CUDA events around every launch during extra steps
    ops.PROFILE = []
    static_head = model.static_head
    model.static_head = False          # exact per-modality row counts on the host -> exact FLOPs per launch (the static head launches
    eager_step(dev_batches[0]); eager_step(dev_batches[1])          # with upper-bound shapes); CUDA events need Python-issued launches
    model.static_head = static_head
    torch.cuda.synchronize()
    gemm_ms = sum(s.elapsed_time(e) for s, e, _, _ in ops.PROFILE)
    gemm_flops = sum(f for _, _, f, _ in ops.PROFILE)
    n_gemm = len(ops.PROFILE)
    if rank == 0 and os.environ.get("B200FM_DUMP_GEMM"):
        agg = {}
        for s_, e_, f_, key in ops.PROFILE:
            a_ = agg.setdefault(key, [0, 0.0, 0.0])
            a_[0] += 1; a_[1] += s_.elapsed_time(e_); a_[2] += f_
        rows = [dict(layout=k[0], epilogue=k[1], M=k[2], N=k[3], K=k[4], launches_per_step=v[0] // 2, ms_per_launch=v[1] / v[0],
                     tflops=v[2] / (v[1] * 1e-3) / 1e12) for k, v in sorted(agg.items(), key=lambda kv: -kv[1][1])]
        with open(os.environ["B200FM_DUMP_GEMM"], "w") as f:
            json.dump(rows, f, indent=1)
    ops.PROFILE = None
    step_ms_prof = None
    # the same launch sequence (every GEMM of one step, same operands, same order) replayed back to back as a CUDA graph: the GEMM
    # family's throughput under the step's own launch conditions (programmatic dependent launch between consecutive kernels; the
    # per-launch events above serialise the launches and break that overlap)
    gemm_graph_ms = None
    try:
        ops.RECORD = []
        model.static_head = False
        eager_step(dev_batches[0])
        recs, ops.RECORD = ops.RECORD, None
        model.static_head = static_head
        torch.cuda.synchronize()
        gg = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gg, capture_error_mode="thread_local"):
            for kw, _ in recs:
                kw = dict(kw)
                getattr(ops, kw.pop("_fn", "gemm"))(**kw)
        for _ in range(2):
            gg.replay()
        torch.cuda.synchronize()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        for _ in range(5):
            gg.replay()
        r1.record()
        torch.cuda.synchronize()
        gemm_graph_ms = r0.elapsed_time(r1) / 5
        gemm_graph_flops = sum(f for _, f in recs)
        del gg, recs
    except Exception as exc:      # measurement extra: never fail the bench line because of it
        ops.RECORD = None
        model.static_head = static_head
        print(f"[bench] GEMM-sequence replay skipped: {exc!r}", file=sys.stderr)

    if rank == 0:
        peaks = measured_peaks()
        tokens_per_step = world * B * 2 * n_tok
        tps = tokens_per_step / (ms / args.steps / 1e3)
        tps_e2e = tokens_per_step / (ms_e2e / args.steps / 1e3)
        blocks, total = flops_per_sample_fwd(n_tok, n_tok, wl["D"], wl["Le"], wl["Ld"], wl["H"])
        achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
        model_tflops = 3 * total * B * world / (ms / args.steps / 1e3) / 1e12
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cb = 8 if args.workload == "4m-b" else 2
            v, sec, cores = cpu_reference_steps(2, 1, cb, n_tok, model_name=args.model)
            cpu = dict(value=v, unit="tokens/s", cores=cores, kind="port",
                       sample=f"2 timed fwd+bwd steps (1 warm-up) of B={cb} x {2 * n_tok} tokens, oracle port of FourM.forward, fp32, {cores} threads of {os.cpu_count()}")
        line = dict(metric="tokens_per_sec", value=tps, unit="tokens/s", n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3),
                    ms_per_step=ms / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16", data="synthetic",
                    config=dict(workload=wl["name"],
                                model=args.model, global_batch=B * world, per_gpu_batch=B, seq_len=2 * n_tok, encoder_tokens=n_tok,
                                decoder_tokens=n_tok, parallelism=f"dp{world}", params_m=round(n_params / 1e6, 1),
                                l2_policy="per-step working set (activations+grads > 2 GB) exceeds the 126 MB L2; two alternating input batches"),
                    e2e=dict(value=tps_e2e, unit="tokens/s", h2d_bytes_per_step=h2d_e2e, d2h_bytes_per_step=4, ms_per_step=ms_e2e / args.steps,
                             rgb_wire_format=("uint8 pixels, normalised on the GPU" if e2e_wire == "uint8" else "fp32, normalised by the loader")),
                    e2e_fp32_wire=dict(value=tokens_per_step / (ms_e2e_f32 / args.steps / 1e3), unit="tokens/s", h2d_bytes_per_step=h2d,
                                       d2h_bytes_per_step=4, ms_per_step=ms_e2e_f32 / args.steps),
                    gpu_launches=launches, loss=loss_val, host_issue_ms_per_step=cpu_issue_ms,
                    launch_mode=("cuda-graph replay of the whole step (b200fm.graph.GraphedTrainStep)" if use_graph else "python-issued launches"),
                    model_tflops_per_gpu=model_tflops / world,
                    frac_of_bf16_peak=model_tflops / world / peaks["bf16"],
                    roofline=dict(bound="tensor", kernel="gemm_kernel<BN,LAYOUT,EPI> (all tcgen05 GEMM launches of a step)",
                                  achieved=(gemm_graph_flops / (gemm_graph_ms * 1e-3) / 1e12 if gemm_graph_ms else achieved),
                                  peak=peaks["bf16"], unit="TFLOP/s",
                                  frac=(gemm_graph_flops / (gemm_graph_ms * 1e-3) / 1e12 if gemm_graph_ms else achieved) / peaks["bf16"],
                                  how=("the step's GEMM launch sequence replayed back to back (CUDA graph, PDL on), CUDA events around 5 replays"
                                       if gemm_graph_ms else "CUDA events around every launch (serialised)"),
                                  achieved_serialised=achieved, frac_serialised=achieved / peaks["bf16"], gemm_ms_per_step_replayed=gemm_graph_ms,
                                  traffic=gemm_traffic_per_launch()[0],
                                  traffic_unit=f"bytes/launch (dram read+write, ncu: profiles/{gemm_traffic_per_launch()[1]})", peak_source=peaks["src"],
                                  launches_per_step=n_gemm // 2, gemm_ms_per_step=gemm_ms / 2),
                    clocks=clocks)
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if world > 1:
            line["comm"] = dict(kind=("nccl all-reduce of torch-DDP buckets" if comm == "ddp" else
                                      f"gradient arena + {gsync.transport.name} all-reduce ({gsync.n_ctas} CTAs, {len(gsync.chunks)} chunks)"),
                                ms_per_step_without_comm=ms_nocomm / args.steps, exposed_ms_per_step=(ms - ms_nocomm) / args.steps,
                                stats=None if gsync is None else gsync.stats)
            line["ddp_params_equal"] = params_equal
        print(json.dumps(line))
    if world > 1:
        if gsync is not None:
            torch.cuda.synchronize()
            dist.barrier()
            gsync.close()
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------------------------------
# VQ tokenizer workloads (BASELINE.json configs[4]: ViT-B @ 256^2, K = 16384, d = 32; per-GPU batch 64 = global 512 on 8 GPUs)
# ----------------------------------------------------------------------------------------------------------------------
VQ_KW = dict(enc_type="vit_b_enc", image_size=256, patch_size=16, codebook_size=16384, latent_dim=32, norm_codes=True, post_mlp=True)
VIT_B_GFLOP_FWD = 48.6            # SURVEY.md 8d: ViT-B encoder @ 256^2, GFLOP per image forward


def _vq_cpu_tokenize(n_img, steps, warmup):
    """The tokenizer forward on the host CPU: the unmodified reference `VQ.tokenize` (fourm/vq/vqvae.py:318-331) where the
    tree exists, else the oracle port (oracle/vq_oracle.py)."""
    torch.set_num_threads(cpu_threads())
    g = torch.Generator().manual_seed(0)
    x = torch.randn(n_img, 3, 256, 256, generator=g)
    if reference_tree() is not None and not os.environ.get("B200FM_CPU_PORT"):
        _import_real_reference()
        import fourm.vq as rvq
        torch.manual_seed(0)
        m = rvq.VQ(sync_codebook=False, **VQ_KW).eval()
        kind = "reference"

        def run():
            with torch.no_grad():
                return m.tokenize(x)
    else:
        from oracle import vq_oracle as V
        import fourm.vq as vq
        torch.manual_seed(0)
        sd = {k: v.detach().clone() for k, v in vq.VQ(sync_codebook=False, **VQ_KW).state_dict().items()}
        kind = "port"

        def run():
            with torch.no_grad():
                return V.vq_encode(x, sd, "vit_b_enc", 16, True, True)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        run()
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    sec = sum(times) / len(times)
    return n_img / sec, sec, torch.get_num_threads(), kind


def run_vq_reference_arm(args):
    if args.workload == "vqvae-train":
        # the reference's VQVAE training step needs `diffusers`-free imports only (vqvae.py); fwd+bwd on CPU through the real class
        torch.set_num_threads(cpu_threads())
        B = 2
        g = torch.Generator().manual_seed(0)
        x = torch.randn(B, 3, 256, 256, generator=g)
        kind = "port"
        if reference_tree() is not None and not os.environ.get("B200FM_CPU_PORT"):
            _import_real_reference()
            import fourm.vq as rvq
            torch.manual_seed(0)
            m = rvq.VQVAE(dec_type="vit_b_dec", sync_codebook=False, ema_decay=0.99, **VQ_KW).train()
            kind = "reference"

            def run():
                dec, code_loss = m(x)
                (torch.nn.functional.mse_loss(dec, x) + code_loss.sum()).backward()
                m.zero_grad(set_to_none=True)
        else:
            from oracle import vq_oracle as V
            import fourm.vq as vq
            torch.manual_seed(0)
            kw = dict(VQ_KW, dec_type="vit_b_dec", ema_decay=0.99)
            sd = {k: v.detach().clone().requires_grad_(v.is_floating_point() and "_codebook" not in k) for k, v in
                  vq.VQVAE(sync_codebook=False, **kw).state_dict().items()}

            def run():
                dec, code_loss = V.vqvae_forward_train(x, sd, kw)[:2]
                (torch.nn.functional.mse_loss(dec, x) + code_loss.sum()).backward()
                for t in sd.values():
                    t.grad = None
        times = []
        for it in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            run()
            if it >= args.warmup:
                times.append(time.perf_counter() - t0)
        sec = sum(times) / len(times)
        val, cores, n_img, what = B / sec, torch.get_num_threads(), B, "VQ-VAE training step fwd+bwd (ViT-B enc + ViT-B dec, K=16384)"
    else:
        n_img = 4
        val, sec, cores, kind = _vq_cpu_tokenize(n_img, args.steps, args.warmup)
        what = "VQ.tokenize (ViT-B encoder + codebook arg-max, K=16384)"
    line = dict(metric="images_per_sec", value=val, unit="img/s", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup, ms_per_step=sec * 1e3,
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic", impl="reference",
                config=dict(workload=f"{what} 256x256 on host CPU, fp32", global_batch=n_img, parallelism="cpu"),
                cpu_baseline=dict(value=val, unit="img/s", cores=cores, kind=kind, sample=f"{n_img} images of 256x256 per step, fp32, {cores} threads of {os.cpu_count()}"),
                e2e=dict(value=val, unit="img/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line))


def run_vq_arm(args):
    """`vq-tokenize`: VQ.tokenize on [B,3,256,256] (save_vq_tokens.py:288-303: fp32 images in, int16 tokens out).
    `vqvae-train`: one VQ-VAE training step (run_training_vqvae.py: encoder + quantizer w/ EMA codebook + ViT-B decoder, MSE, AdamW).
    Both shard by sample with replicas (vq-tokenize: no collective at all; vqvae-train: DDP + the packed codebook all-reduce)."""
    import torch.distributed as dist
    import torch.nn.functional as F
    import fourm.vq as vq
    from b200fm import lib, ops
    from b200fm.optim import FusedAdamW
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py (B200 arm) needs a GPU; there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib.load()
    B = args.batch or 64
    train = args.workload == "vqvae-train"
    torch.manual_seed(0)
    g = torch.Generator().manual_seed(100 + rank)
    host_x = [torch.randn(B, 3, 256, 256, generator=g).pin_memory() for _ in range(2)]
    dev_x = [h.to(dev) for h in host_x]
    if train:
        model = vq.VQVAE(dec_type="vit_b_dec", sync_codebook=world > 1, ema_decay=0.99, **VQ_KW).to(dev).train()
        opt = FusedAdamW([p for p in model.parameters() if p.requires_grad], lr=1e-4, betas=(0.9, 0.99), weight_decay=0.0)
        net = model
        if world > 1:
            net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local], gradient_as_bucket_view=True, broadcast_buffers=False)

        from b200fm.optim import FusedModelEma
        model_ema = FusedModelEma(model, decay=0.9999)          # run_training_vqvae.py:224, 683-688 (--model_ema defaults to True)

        def step(x):
            dec, code_loss = net(x)
            loss = F.mse_loss(dec.float(), x) + code_loss.sum()
            loss.backward()
            opt.step()
            opt.zero_grad(set_to_none=True)
            model_ema.update(model)                                # every step (run_training_vqvae.py:1169-1171), one multi-tensor launch
            return loss
    else:
        model = vq.VQ(sync_codebook=False, **VQ_KW).to(dev).eval()
        host_tok = torch.empty(B, 16, 16, dtype=torch.int16).pin_memory()

        if os.environ.get("B200FM_GRAPH", "1") != "0":
            from b200fm.graph import GraphedCall
            gcall = {}                                   # one per precision mode (the mode is baked into the captured launches)

            def step(x):
                key = os.environ.get("B200FM_VQ_PRECISION", "auto")
                if key not in gcall:
                    gcall[key] = GraphedCall(model.tokenize, clone=False)
                return gcall[key](x)
        else:
            def step(x):
                with torch.no_grad():
                    return model.tokenize(x)

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(n, e2e):
        c0 = lib.CALLS["n"]
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            if e2e:
                x = host_x[i % 2].to(dev, non_blocking=True)            # 50 MB of fp32 pixels per step from pinned host memory
                out = step(x)
                if train:
                    out.item()
                else:
                    host_tok.copy_(out.to(torch.int16), non_blocking=True)   # save_vq_tokens.py:293 stores int16
                    torch.cuda.current_stream().synchronize()
            else:
                out = step(dev_x[i % 2])
        e1.record()
        sync()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, lib.CALLS["n"] - c0

    for _ in range(max(args.warmup, 3)):
        step(dev_x[0])
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms, launches = timed(args.steps, False)
    ms_e2e, _ = timed(args.steps, True)
    ms_bf16 = None
    if not train:
        # the same call with bf16 operands (what a caller under torch.autocast(bfloat16) gets) instead of the fp32-faithful limb arithmetic
        os.environ["B200FM_VQ_PRECISION"] = "bf16"
        try:
            for _ in range(3):
                step(dev_x[0])
            ms_bf16, _ = timed(args.steps, False)
        finally:
            os.environ.pop("B200FM_VQ_PRECISION", None)
    clocks = sampler.stop() if rank == 0 else None
    ops.PROFILE = []
    if train:
        step(dev_x[0]); step(dev_x[1])
    else:                                               # eagerly: the per-GEMM events cannot be recorded into a graph replay
        with torch.no_grad():
            model.tokenize(dev_x[0]); model.tokenize(dev_x[1])
    torch.cuda.synchronize()
    gemm_ms = sum(s.elapsed_time(e) for s, e, _, _ in ops.PROFILE)
    gemm_flops = sum(f for _, _, f, _ in ops.PROFILE)
    n_gemm = len(ops.PROFILE)
    ops.PROFILE = None
    # the codebook scan alone (fp32-FMA bound, SURVEY.md 8d): n = B*256 latents x K = 16384 x d = 32
    z = F.normalize(torch.randn(B * 256, 32, device=dev), dim=-1)
    cbk = F.normalize(torch.randn(16384, 32, device=dev), dim=-1)
    for _ in range(3):
        ops.vq_argmax(z, cbk, cosine=True)
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); s0.record()
    for _ in range(10):
        ops.vq_argmax(z, cbk, cosine=True)
    s1.record(); torch.cuda.synchronize()
    scan_ms = s0.elapsed_time(s1) / 10
    if rank == 0:
        peaks = measured_peaks()
        per = ms / args.steps
        val = world * B / (per / 1e3)
        val_e2e = world * B / (ms_e2e / args.steps / 1e3)
        achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
        mult = 3 * 2 if train else 1
        model_tflops = mult * VIT_B_GFLOP_FWD * 1e9 * B / (per / 1e3) / 1e12
        cpu = None
        if world == 1 and not args.no_cpu_baseline and not train:
            v, sec, cores, kind = _vq_cpu_tokenize(2, 1, 1)
            cpu = dict(value=v, unit="img/s", cores=cores, kind=kind, sample=f"1 timed VQ.tokenize of 2 images 256x256 (1 warm-up), fp32, {cores} threads of {os.cpu_count()}")
        name = ("VQ-VAE training step (ViT-B enc + dec, K=16384, EMA codebook, MSE, AdamW, model EMA), BASELINE.json configs[4]" if train else
                "VQ.tokenize (ViT-B encoder + codebook arg-max K=16384, d=32), 256x256, called like save_vq_tokens.py:288 (no autocast -> "
                "fp32-faithful limb arithmetic, 3 bf16 limb products per contraction), BASELINE.json configs[4] tokenizer forward")
        mult = mult if train else 3                      # fp32-faithful: three limb GEMM terms per product
        line = dict(metric="images_per_sec", value=val, unit="img/s", n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3), ms_per_step=per,
                    higher_is_better=True, scaling="weak", vs_baseline=None, dtype=("bf16" if train else "bf16x3 (fp32-faithful)"), data="synthetic",
                    config=dict(workload=name, global_batch=B * world, per_gpu_batch=B, image_size=256, tokens_per_image=256, parallelism=f"dp{world}",
                                l2_policy="two alternating 50 MB input batches; activations exceed the 126 MB L2",
                                cuda_graph=(not train and os.environ.get("B200FM_GRAPH", "1") != "0")),
                    e2e=dict(value=val_e2e, unit="img/s", h2d_bytes_per_step=host_x[0].numel() * 4, d2h_bytes_per_step=4 if train else B * 256 * 2,
                             ms_per_step=ms_e2e / args.steps),
                    gpu_launches=launches, latents_per_sec=val * 256,
                    bf16_autocast_img_per_s=(None if ms_bf16 is None else world * B / (ms_bf16 / args.steps / 1e3)), model_tflops_per_gpu=model_tflops / 1, frac_of_bf16_peak=model_tflops / peaks["bf16"],
                    roofline=dict(bound="tensor", kernel="gemm_kernel<BN,LAYOUT,EPI> (all tcgen05 GEMM launches of a step)", achieved=achieved, peak=peaks["bf16"],
                                  unit="TFLOP/s", frac=achieved / peaks["bf16"], traffic=None, peak_source=peaks["src"], launches_per_step=n_gemm // 2,
                                  gemm_ms_per_step=gemm_ms / 2),
                    scan=dict(kernel="vq_scan_kernel<32>", bound="fp32 FMA (CUDA cores; HBM traffic is z + idx only)", n=B * 256, K=16384, d=32, ms=scan_ms,
                              tflops_fp32=2.0 * B * 256 * 16384 * 32 / (scan_ms * 1e-3) / 1e12, algorithmic_gbs=(B * 256 * (32 * 4 + 8) + 16384 * 32 * 4) / (scan_ms * 1e-3) / 1e9),
                    clocks=clocks)
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_gen_arm(args):
    from b200fm import genbench
    genbench.run(args, ClockSampler, measured_peaks, cpu_threads, reference_tree)


def run_gen_reference_arm(args):
    from b200fm import genbench
    genbench.run_reference(args, cpu_threads, reference_tree)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="4m-b", choices=["4m-b", "4m-l", "vq-tokenize", "vqvae-train", "gen"],
                    help="4m-b = BASELINE.json configs[1] (the headline metric, default); 4m-l = configs[2]; gen = configs[3] "
                         "(generation latency); vq-tokenize / vqvae-train = configs[4] (VQ tokenizer forward / training step)")
    ap.add_argument("--model", default=None)
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch (default: the workload's reference config)")
    ap.add_argument("--tokens", type=int, default=None, help="encoder tokens = decoder tokens per sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's loss, per-modality losses, gradient norm and a seeded parameter sample as "
                         "DIR/<name>.npy (4m-b / 4m-l on the GPU)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.workload not in WORKLOADS):
        ap.error("--dump-outputs is implemented for the GPU train step (--workload 4m-b / 4m-l)")
    if args.impl == "reference":
        run_reference_arm(args)
    elif args.workload in ("vq-tokenize", "vqvae-train"):
        run_vq_arm(args)
    elif args.workload == "gen":
        run_gen_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
