#!/usr/bin/env python
"""bench.py -- TGANv2-conditional G+D training step throughput (videos/s) on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host CPU cores
    python bench.py --impl torch_cuda                         # the same iteration on torch eager cuDNN/cuBLAS (B200)

Workload (BASELINE.json configs[3], the configuration the metric is quoted on): TGANv2 conditional,
64x64x16 clips, Bi-LSTM caption encoder, non-local blocks, RSGAN loss + zero-centred gradient penalty
(lambda 0.5), Adam(2e-4, (0.5, 0.999)), 1 D step + 1 G step per iteration, synthetic U(-1,1) clips and
MSRVDC-shaped captions (SURVEY.md 8d).  One "step" = one full training iteration over one batch.

Prints ONE JSON line (rank 0).  `value` = videos/s with inputs resident in HBM, device-timed (CUDA events,
max over ranks); `e2e` = the same through the public train_iteration() API with host (pinned) inputs
copied in and the two losses read back every step; `roofline` = the conv engine's tcgen05 kernel timed per
launch with CUDA events (t2v_profile_*) in a profiled pass of the same step right after the timed region;
`cpu_baseline` = the oracle (CPU restatement of the reference) on the host cores, bounded sample.
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import threading
import time
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GFLOP_PER_VIDEO_NOMINAL = 55.4      # SURVEY.md 8(d): config 4 incl. gradient penalty, padded taps counted
WORKLOAD = "TGANv2-cond 64x64x16 G+D train step (RSGAN + GP 0.5, Adam), synthetic clips + captions"


def peaks():
    p = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            m = json.load(f)
        p.update({k: m[k] for k in ("hbm_gbs", "bf16_tflops", "bf16_tflops_sustained") if k in m})
        p["source"] = "measured"
    except Exception:
        pass
    return p


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


DUMP_SAMPLE = 1 << 21      # parameter entries written per module by --dump-outputs (8 MB of float32 each)


def dump_outputs(out_dir, losses, modules):
    """What the timed step hands back, as DIR/<name>.npy: loss_d and loss_g (float64), and the parameters the step
    updated in place, flattened in named_parameters() order (float32) -- a fixed seeded sample of DUMP_SAMPLE
    positions when a module has more, so that runs with the same arguments compare position for position.  The inputs
    are the same from run to run; the outputs agree to a tolerance, not bit for bit, because the weight-gradient
    kernels accumulate with float atomics."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, v in zip(("loss_d", "loss_g"), losses):
        np.save(os.path.join(out_dir, name + ".npy"), np.array(float(v), dtype=np.float64))
    for name, m in modules:
        flat = torch.cat([p.detach().reshape(-1).float() for p in m.parameters()])
        if flat.numel() > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(flat.numel(), DUMP_SAMPLE, replace=False))
            flat = flat[torch.from_numpy(idx).to(flat.device)]
        np.save(os.path.join(out_dir, name + "_params.npy"), flat.cpu().numpy())


def train_params(gp_lambda, frame_sizes=(8, 16, 32, 64)):
    return SimpleNamespace(data_is_imgs=False, img_model=False, frame_sizes=list(frame_sizes), subsample_input=True,
                           discrim_steps=1, gen_steps=1, gp_lambda=gp_lambda, no_mean_discrim_loss=False,
                           no_mean_gen_loss=True)


# =========================================================================================== reference arm
def run_reference(args):
    """The reference's algorithm on the host CPU cores (oracle port: /root/reference is Python and does not
    travel to the GPU box).  Rank 0 only; bounded sample: batch 8 per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    out = cpu_baseline(steps=max(1, args.steps), warmup=max(1, min(args.warmup, 1)), batch=args.cpu_batch)
    line = {"metric": "TGANv2-cond G+D train videos/sec", "value": out["value"], "unit": "videos/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": out["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": WORKLOAD, "batch_per_step": args.cpu_batch, "device": "cpu"},
            "cpu_baseline": {k: out[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": out["value"], "unit": "videos/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def _oracle_arm(device, steps, warmup, batch, autocast=False):
    """the oracle's train_iteration (reference modules restated on torch ops) on `device`: seconds per iteration"""
    import torch
    import oracle.txt2vid_oracle as O
    from txt2vid_b200.factory import build_models as build_product_models
    from txt2vid_b200.data import SyntheticVideoCaptions
    V = 1000
    cuda = torch.device(device).type == "cuda"
    with contextlib.redirect_stdout(io.StringIO()):
        txt, gen, dis = build_product_models(True, vocab_size=V, seed=100)     # same constructors/init as the reference
    sd_g, sd_d, sd_t = (O.as_leaves({k: v.detach().clone().to(device) for k, v in m.state_dict().items()})
                        for m in (gen, dis, txt))
    del txt, gen, dis
    opt_g = O.Adam(O.param_names(sd_g), 2e-4, (0.5, 0.999))
    opt_d = O.Adam(O.param_names(sd_d), 2e-4, (0.5, 0.999))
    times = []
    for it in range(warmup + steps):
        x, tokens, lengths = SyntheticVideoCaptions(batch, 1, vocab_size=V, seed=1234 + it).batch(0)
        x = x.permute(0, 2, 1, 3, 4).contiguous().to(device)
        tokens = tokens.to(device)
        if cuda:
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        bt_real = O.draw_real(4, True)
        z = torch.randn(batch, 256).to(device)
        draws = O.draw_rest([batch, batch // 2, batch // 4, batch // 8], conditional=True, gp=True)
        draws["bt_real"] = bt_real
        with torch.autocast(torch.device(device).type, dtype=torch.bfloat16, enabled=autocast, cache_enabled=False):
            out = O.train_iteration(sd_g, sd_d, sd_t, x, tokens, lengths, z, draws, opt_g=opt_g, opt_d=opt_d)
        if cuda:
            float(out["lossD"]), float(out["lossG"])
            torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    return sum(times) / len(times), len(times)


def cpu_baseline(steps=2, warmup=1, batch=8):
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    per, n = _oracle_arm("cpu", steps, warmup, batch)
    return {"value": batch / per, "unit": "videos/s", "cores": cores, "kind": "port", "ms_per_step": per * 1e3,
            "sample": "%d timed iterations of batch %d (same model/loss/optimiser, fp32, torch CPU threads=%d)"
                      % (n, batch, cores)}


def library_baseline(batches=(64, 256), steps=3, warmup=2, device="cuda:0"):
    """The B200 LIBRARY comparator (BASELINE.md section 4 item 4, SURVEY 2.4 "the kernel to beat on the same box"):
    the same iteration -- the oracle's restatement of the reference modules, i.e. what the reference computes when run
    on this GPU through PyTorch eager -- on cuDNN / cuBLAS / ATen kernels: fp32 with TF32 off (the reference's
    numerics) and under torch.autocast(bfloat16) (the library's mixed-precision recipe).  None of this repo's kernels
    run here.  Largest batch first fails soft (out of memory -> recorded as null)."""
    import torch
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cudnn.benchmark = True            # the reference sets it (train/setup.py:17)
    out = {"what": "reference modules (oracle restatement) on torch eager cuDNN/cuBLAS, same iteration, same GPU",
           "unit": "videos/s", "runs": []}
    for autocast in (False, True):
        for bsz in batches:
            rec = {"precision": "bf16 autocast" if autocast else "fp32 (TF32 off)", "batch": bsz}
            try:
                per, n = _oracle_arm(device, steps, warmup, bsz, autocast=autocast)
                rec.update({"value": bsz / per, "ms_per_step": per * 1e3, "timed_steps": n})
            except torch.cuda.OutOfMemoryError:
                rec.update({"value": None, "note": "out of memory"})
            torch.cuda.empty_cache()
            out["runs"].append(rec)
    best = [r for r in out["runs"] if r.get("value")]
    out["best"] = max(best, key=lambda r: r["value"]) if best else None
    return out


def run_library(args):
    """--impl torch_cuda: the library comparator alone, one JSON line in the bench format (rank 0)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    lb = library_baseline(batches=tuple(args.lib_batches), steps=max(1, args.steps), warmup=max(1, args.warmup))
    best = lb["best"] or {"value": None, "ms_per_step": None, "batch": None, "precision": None}
    print(json.dumps({"metric": "TGANv2-cond G+D train videos/sec", "value": best["value"], "unit": "videos/s",
                      "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": best["ms_per_step"],
                      "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                      "dtype": best["precision"], "data": "synthetic", "impl": "torch_cuda",
                      "config": {"workload": WORKLOAD, "batch_per_gpu": best["batch"], "device": "cuda:0"},
                      "library_baseline": lb, "gpu_launches": 0}), flush=True)


# =========================================================================================== B200 arm
def run_b200(args):
    import numpy as np
    import torch
    from txt2vid_b200 import _lib, ops
    from txt2vid_b200 import kernels as K
    from txt2vid_b200.data import SyntheticVideoCaptions
    from txt2vid_b200.gan import CondGan, MixedGanLoss, RSGANLoss
    from txt2vid_b200.optim import FusedAdam
    from txt2vid_b200.parallel import DistContext
    from txt2vid_b200.trainer import GraphedTrainStep, train_iteration
    from txt2vid_b200.factory import build_models as build_product_models

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path (use --impl reference)")
    dist = DistContext()
    rank, world = dist.rank, dist.world
    torch.cuda.set_device(dist.local_rank)
    device = torch.device("cuda", dist.local_rank)
    b = args.batch
    V = 1000
    # --res 128: BASELINE configs[4] (128x128x32, frame sizes 16..128); default: configs[3] (64x64x16), the metric's
    res, frames = (128, 32) if args.res == 128 else (64, 16)
    fsizes = (16, 32, 64, 128) if args.res == 128 else (8, 16, 32, 64)
    gflop_nominal = 407.3 if args.res == 128 else GFLOP_PER_VIDEO_NOMINAL        # SURVEY.md 8(d)
    workload = WORKLOAD if args.res == 64 else WORKLOAD.replace("64x64x16", "128x128x32")
    with contextlib.redirect_stdout(io.StringIO()):
        txt, gen, dis = build_product_models(True, vocab_size=V, seed=100, width=res, height=res, num_frames=frames)
    txt, gen, dis = txt.to(device), gen.to(device), dis.to(device)
    torch.manual_seed(100)                       # CPU generator: identical frame offsets on every rank
    torch.cuda.manual_seed(100 + rank)
    np.random.seed(100 + rank)
    gan = CondGan(gen=gen, discrims=[dis], cond_encoder=txt, discrim_names=["video"])
    losses = MixedGanLoss(g_loss=RSGANLoss(), d_loss=RSGANLoss())
    optD = FusedAdam([{"params": dis.parameters()}], lr=2e-4, betas=(0.5, 0.999))
    optG = FusedAdam([{"params": gen.parameters()}], lr=2e-4, betas=(0.5, 0.999))
    params = train_params(0.5 * dist.gp_scale, fsizes)
    ddp = dist if dist.enabled else None

    nb = 4
    data = SyntheticVideoCaptions(b, nb, vocab_size=V, seed=1234 + 1000 * rank, frames=frames, size=res)
    # 4 distinct RESIDENT batches; only `nh` of them are also kept in pinned host memory for the fp32-host-batch leg
    # (3.2 GB each at b = 4096: eight ranks of one box would pin > 100 GB with all four)
    nh = 2 if b * frames * res * res >= 4096 * 16 * 64 * 64 else nb
    dev, host = [], []
    for i in range(nb):
        x, t, l = data.batch(i)
        x = x.contiguous()
        if i < nh:
            x, t = x.pin_memory(), t.pin_memory()
            host.append((x, t, l))
        dev.append((x.to(device), t.to(device), l))
        del x

    lib = _lib.lib()
    if args.eager:
        def run_step(x, t, l):
            ld, lg, _, _, _ = train_iteration(gan, x, [t, l], device, optD, optG, params, losses, end2end=False,
                                              dist=ddp)
            return ld, lg
    else:
        graphed = GraphedTrainStep(gan, optD, optG, params, losses, device, end2end=False, dist=ddp, warmup=2)

        def run_step(x, t, l):
            return graphed(x, [t, l])

    res_evt = [torch.cuda.Event() for _ in range(3)]
    last_out = {}

    def step_resident(i):
        x, t, l = dev[i % nb]
        out = run_step(x, t, l)
        last_out["losses"] = out
        # keep the host two steps ahead at most (what the launch queue allows on one GPU anyway): with NCCL between the
        # graph replays an unbounded run-ahead measured 128 ms / step at two GPUs against 92 ms through the e2e loop
        res_evt[i % 3].record()
        if i >= 2:
            res_evt[(i - 2) % 3].synchronize()
        return out

    # end-to-end leg: the public loop of gan/trainer.py:176-267 -- batches come from pinned HOST memory through
    # data_prefetcher (data/__init__.py:131-156: next batch copied on a side stream while the current one trains),
    # every step's H2D copy happens inside the timed region, and both losses are read back on the host each step.
    from txt2vid_b200.data import data_prefetcher
    e2e_state = {}

    def e2e_begin(n):
        e2e_state["pf"] = data_prefetcher(((host[i % nh][0], host[i % nh][1], host[i % nh][2]) for i in range(n)),
                                          device=device)

    LAG = int(os.environ.get("T2V_E2E_LAG", "2"))                  # the host logs step i-LAG while step i is enqueued
    loss_host = [torch.zeros(2).pin_memory() for _ in range(LAG + 1)]
    loss_evt = [torch.cuda.Event() for _ in range(LAG + 1)]
    variant = os.environ.get("T2V_E2E_VARIANT", "")      # diagnosis only: "nopf" = resident inputs, "noloss" = no read-back

    def read_loss(j):
        loss_evt[j % (LAG + 1)].synchronize()
        e2e_state["last"] = (float(loss_host[j % (LAG + 1)][0]), float(loss_host[j % (LAG + 1)][1]))

    def step_e2e(i):
        if variant == "nopf":
            x, y = dev[i % nb][0], dev[i % nb][1:]
        else:
            x, y = e2e_state["pf"].next(preload=False)
        ld, lg = run_step(x, y[0], y[1])
        if variant != "nopf":
            e2e_state["pf"].preload()                             # bulk copy of the next batch goes out behind this step
        if variant == "noloss":
            return
        # device->host read of EVERY step's result: asynchronous copy into pinned memory, consumed LAG steps later
        # (back-to-back graph launches need the host more than one step ahead of the device; every loss is read
        # inside the timed region, the last ones are drained before the clock stops)
        # (written into the pinned buffer by an SM copy kernel over UVA: a cudaMemcpyAsync D2H on the compute stream
        # queues behind the prefetcher's 48 MB H2D chunks on the copy engine and stalls the next step)
        K.multi_copy([torch.stack((ld.detach().float().reshape(()), lg.detach().float().reshape(())))],
                     [loss_host[i % (LAG + 1)]])
        loss_evt[i % (LAG + 1)].record()
        if i >= LAG:
            read_loss(i - LAG)

    def e2e_end(n):
        if variant == "noloss":
            return
        for j in range(max(0, n - LAG), n):
            read_loss(j)

    def timed(fn, n, begin=None, end=None):
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if begin is not None:
            begin(n)                                              # first H2D copy is issued inside the timed region
        for i in range(n):
            fn(i)
        if end is not None:
            end(n)
        e1.record()
        torch.cuda.synchronize()
        dist.barrier()
        return dist.all_reduce_max(e0.elapsed_time(e1) / 1e3)

    l0 = lib.t2v_launch_count()
    step_resident(0)
    step_resident(1)                                              # eager warm-ups (graph mode: then capture)
    l1 = lib.t2v_launch_count()
    launches_per_step = int(l1 - l0) // 2
    for i in range(2, max(5, args.warmup)):
        step_resident(i)
    torch.cuda.synchronize()
    clocks = ClockSampler(dist.local_rank)
    sample_clocks = rank == 0 and os.environ.get("T2V_BENCH_NO_CLOCKS", "0") != "1"      # (diagnosis switch)
    if sample_clocks:
        clocks.start()
    t_res = timed(step_resident, args.steps)
    launches = launches_per_step * args.steps
    clk = clocks.stop() if sample_clocks else None
    if args.dump_outputs and rank == 0:                           # the legs below keep training the same modules
        dump_outputs(args.dump_outputs, last_out["losses"], (("gen", gen), ("dis", dis)))
    timed(step_e2e, 3, begin=e2e_begin, end=e2e_end)               # e2e warm-up (staging slots, pinned pages)
    t_e2e = timed(step_e2e, args.steps, begin=e2e_begin, end=e2e_end)

    # the same loop fed with the frames as stored (uint8; ToTensor + Normalize run on the device inside
    # data_prefetcher): a quarter of the bytes over PCIe.  This is the line's `e2e`; the fp32-host-batch loop above is
    # reported next to it as `e2e_fp32_host`.
    data8 = SyntheticVideoCaptions(b, 2, vocab_size=V, seed=4321 + 1000 * rank, frames=frames, size=res, as_uint8=True)
    host8 = [data8.batch(i) for i in range(2)]
    host8 = [(x.contiguous().pin_memory(), t.pin_memory(), l) for x, t, l in host8]

    def e2e8_begin(n):
        e2e_state["pf"] = data_prefetcher(((host8[i % 2][0], host8[i % 2][1], host8[i % 2][2]) for i in range(n)),
                                          device=device, normalize=args.eager)   # graph mode: fused into the input fill
    timed(step_e2e, 3, begin=e2e8_begin, end=e2e_end)
    t_e2e8 = timed(step_e2e, args.steps, begin=e2e8_begin, end=e2e_end)
    t_res2 = timed(step_resident, args.steps)                      # resident again: thermal / power drift over the run
    x8 = host8[0][0]
    h2d8 = x8.numel() * x8.element_size() + host8[0][1].numel() * host8[0][1].element_size()
    # host -> device bandwidth of this box, copy alone (the fp32 e2e leg cannot beat bytes / this)
    hx = host[0][0]
    stage = torch.empty(hx.shape, dtype=hx.dtype, device=device)
    torch.cuda.synchronize()
    ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ea.record()
    stage.copy_(hx, non_blocking=True)
    eb.record()
    torch.cuda.synchronize()
    h2d_alone_ms = ea.elapsed_time(eb)
    del stage

    # ---- roofline pass: per-launch CUDA-event timing of the conv engine over the same step, run eagerly
    # (events cannot be read back from inside a replayed graph; kernels, shapes and launch order are the same)
    import ctypes
    prof_steps = 2

    def step_eager(i):
        x, t, l = dev[i % nb]
        train_iteration(gan, x, [t, l], device, optD, optG, params, losses, end2end=False, dist=ddp)
    step_eager(0)
    lib.t2v_profile_enable(1)
    timed(step_eager, prof_steps)
    lib.t2v_profile_enable(0)
    NK = 6
    buf = (ctypes.c_double * (3 * NK))()
    lib.t2v_profile_read6(buf)
    prof = list(buf)
    t_prof = t_res / args.steps * prof_steps                       # share is quoted against the timed step
    mem_gb = torch.cuda.max_memory_allocated() / 1e9

    if rank != 0:
        return
    pk = peaks()
    videos = world * b * args.steps
    value = videos / t_res
    e2e = videos / t_e2e
    x0, t0_, _ = host[0]
    h2d = x0.numel() * x0.element_size() + t0_.numel() * t0_.element_size()
    step_ms_prof = t_prof / prof_steps * 1e3
    names = ["igemm_fprop_kernel (generic tcgen05 implicit GEMM: conv fprop + dgrad, Linear, ConvLSTM gates)",
             "igemm_wgrad_kernel (generic tcgen05 weight gradient)",
             "halo_fprop_kernel (halo-resident tcgen05 fprop + dgrad of the 64-channel 3x3x3 stem convs)",
             "halo_wgrad_kernel (halo-resident tcgen05 weight gradient, two taps stacked per MMA)",
             "stem_fprop_kernel (RGB stem conv, im2col tile gathered into shared memory)",
             "stem_wgrad_kernel (RGB stem weight gradient, same tile as MN-major operand)"]
    kern = {}
    for i, nm in enumerate(names):
        ms, fl, n = prof[3 * i:3 * i + 3]
        kern[nm.split(" ")[0]] = {"achieved": fl / (ms * 1e-3) / 1e12 if ms > 0 else None,
                                  "launches_per_step": n / prof_steps, "ms_per_step_in_kernel": ms / prof_steps,
                                  "share_of_step": ms / prof_steps / step_ms_prof if step_ms_prof > 0 else None}
    top = max(range(NK), key=lambda i: prof[3 * i])
    tk = kern[names[top].split(" ")[0]]
    conv_ms = sum(prof[3 * i] for i in range(NK)) / prof_steps
    conv_fl = sum(prof[3 * i + 1] for i in range(NK)) / prof_steps
    # measured DRAM traffic of the dominant kernel: dram__bytes_read.sum + dram__bytes_write.sum per launch from the
    # committed ncu capture of one iteration at the same batch (profiles/r02_traffic_b2048.json, scripts/gpu_r02p.sh)
    traffic, traffic_note = None, "no ncu capture at this batch / resolution"
    tpath = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r02_traffic_b%d.json" % b)
    if res == 64 and os.path.exists(tpath):
        with open(tpath) as f:
            tj = json.load(f)
        fam = {"igemm_fprop_kernel": "igemm_fprop", "igemm_wgrad_kernel": "igemm_wgrad", "halo_fprop_kernel": "halo_fprop",
               "halo_wgrad_kernel": "halo_wgrad", "stem_fprop_kernel": "stem_fprop", "stem_wgrad_kernel": "stem_wgrad"}
        key = fam[names[top].split(" ")[0]]
        sel = [v for k, v in tj.items() if key in k]
        nl = sum(v["launches"] for v in sel)
        if nl > 0:
            traffic = sum(v["dram_bytes"] for v in sel) / nl
            fl_per_launch = prof[3 * top + 1] / max(1.0, prof[3 * top + 2])
            traffic_note = ("ncu dram__bytes_read.sum + dram__bytes_write.sum of every %s* launch of one iteration at "
                            "b = %d (%d launches, %.1f GB in total) / launches; %.0f useful FLOP per DRAM byte -- far "
                            "above the machine balance (~214 FLOP/B): tensor-bound, not HBM-bound"
                            % (key, b, nl, sum(v["dram_bytes"] for v in sel) / 1e9, fl_per_launch / traffic))
    roof = {"bound": "tensor", "kernel": names[top], "achieved": tk["achieved"], "peak": pk["bf16_tflops_sustained"],
            "unit": "TFLOP/s", "traffic": traffic, "traffic_note": traffic_note,
            "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step), %s" % pk["source"],
            "launches_per_step": tk["launches_per_step"], "ms_per_step_in_kernel": tk["ms_per_step_in_kernel"],
            "share_of_step": tk["share_of_step"],
            "flops_counted": "useful MACs x2 per launch (live taps only, zero channel padding excluded), summed over "
                             "the step's launches / summed CUDA-event durations",
            "kernels": kern,
            "conv_engine_all": {"achieved": conv_fl / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else None,
                                "frac": conv_fl / (conv_ms * 1e-3) / 1e12 / pk["bf16_tflops_sustained"] if conv_ms > 0 else None,
                                "ms_per_step": conv_ms, "share_of_step": conv_ms / step_ms_prof if step_ms_prof else None},
            # whole step on the FLOPs the kernels actually issue (dead taps, the even-plane stem convolution and the
            # skipped D weight gradients of the G step are not counted): the headline utilisation
            "step_issued_tflops_per_gpu": conv_fl / (t_res / args.steps) / 1e12,
            "step_issued_frac_of_sustained_peak": conv_fl / (t_res / args.steps) / 1e12 / pk["bf16_tflops_sustained"],
            "step_nominal_tflops_per_gpu": value / world * gflop_nominal / 1e3,
            "step_nominal_frac_of_sustained_peak": value / world * gflop_nominal / 1e3 / pk["bf16_tflops_sustained"]}
    roof["frac"] = roof["achieved"] / roof["peak"] if roof["achieved"] else None
    cpu = libb = None
    launch_mode = "eager" if args.eager else "%d CUDA graph(s) per step" % len(graphed.graphs or ())
    if not args.no_library_baseline:
        # free the product's graphs / pools first: the library arm needs its own activations
        if not args.eager:
            del graphed
        del dev
        torch.cuda.empty_cache()
        try:
            libb = library_baseline(batches=tuple(args.lib_batches))
        except Exception as e:                                    # noqa: BLE001 -- the product's line must still print
            libb = {"error": repr(e)[:200]}
    if not args.no_cpu_baseline:
        c = cpu_baseline(steps=2, warmup=1, batch=args.cpu_batch)
        cpu = {k: c[k] for k in ("value", "unit", "cores", "kind", "sample")}
    line = {"metric": "TGANv2-cond G+D train videos/sec", "value": value, "unit": "videos/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(5, args.warmup), "ms_per_step": t_res / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload, "batch_per_gpu": b, "global_batch": world * b,
                       "parallelism": "dp%d" % world, "launch": launch_mode,
                       "l2": "per-step working set (%.1f GB peak allocated) >> 126 MB L2; "
                       "%d distinct resident batches cycled" % (mem_gb, nb)},
            # headline end-to-end leg: pinned HOST batches hold the frames as stored (uint8), fed through the public
            # loader API (data_prefetcher), ToTensor + Normalize on the device (t2v_u8_normalize, bit-exact), every
            # step's H2D copy and loss read-back inside the timed region
            "e2e": {"value": videos / t_e2e8, "unit": "videos/s", "h2d_bytes_per_step": int(h2d8),
                    "d2h_bytes_per_step": 8, "ms_per_step": t_e2e8 / args.steps * 1e3,
                    "host_batch": "uint8 frames as stored + int64 tokens (pinned); ToTensor + Normalize fused into the "
                                  "fill of the graph's static input (t2v_u8_normalize)"},
            # same loop with fp32 host batches (the reference loader's format: ToTensor + Normalize on CPU workers,
            # data/__init__.py:362-364): four times the PCIe bytes
            "e2e_fp32_host": {"value": e2e, "unit": "videos/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 8,
                              "ms_per_step": t_e2e / args.steps * 1e3, "h2d_alone_ms": h2d_alone_ms,
                              "h2d_alone_gbs": int(h2d) / h2d_alone_ms / 1e6},
            "resident_again_ms_per_step": t_res2 / args.steps * 1e3,
            "gpu_launches": launches, "clocks": clk, "roofline": roof, "cpu_baseline": cpu,
            "library_baseline": libb, "peak_mem_gb": mem_gb}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "torch_cuda"])
    ap.add_argument("--batch", type=int, default=4096, help="videos per GPU per step (multiple of 8)")
    ap.add_argument("--res", type=int, default=64, choices=[64, 128],
                    help="64: 64x64x16 clips (the metric's configuration); 128: 128x128x32 (BASELINE configs[4])")
    ap.add_argument("--cpu_batch", type=int, default=8)
    ap.add_argument("--no_cpu_baseline", action="store_true")
    ap.add_argument("--no_library_baseline", action="store_true")
    ap.add_argument("--lib_batches", type=int, nargs="+", default=[64, 256],
                    help="batches of the torch-eager cuDNN comparator (library_baseline / --impl torch_cuda)")
    ap.add_argument("--eager", action="store_true", help="no CUDA graphs: launch every kernel from Python")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's losses and a sample of the updated G / D "
                         "parameters to DIR/<name>.npy (b200 arm)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "torch_cuda":
        run_library(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
