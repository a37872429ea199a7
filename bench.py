#!/usr/bin/env python
"""Headline benchmark: 512x512 Unet-VGG16 (21 classes) training throughput, batch 16 per GPU, data parallel.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one iteration of the reference's fit_one_epoch body (utils/utils_fit.py:26-97): forward, CE + Dice
(+ f_score), backward, gradient all-reduce (N > 1), Adam step, on one synthetic batch of 16 images per GPU.
Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every key.

  value        img/s over all GPUs, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e          img/s through UnetTrainer.train_step with HOST (pinned) batches: H2D of images + label maps and a
               D2H read of [loss, f_score] every step are inside the timed region
  roofline     conv_igemm_kernel (fprop + dgrad launches): algorithmic FLOPs / per-launch CUDA-event time,
               against MEASURED_PEAKS.json's sustained bf16 figure
  cpu_baseline the oracle (a torch-CPU restatement of the reference path; the reference itself is Python and does
               not travel to the GPU box) timed on this box's host cores on a bounded sample
  --impl reference   times that same CPU path with all host threads and prints the reference-arm line
  --dump-outputs DIR writes what the last timed step computed as DIR/<name>.npy (see dump_outputs), so that two builds
                     can be compared output for output on identical seeded inputs
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NUM_CLASSES = 21
BATCH_PER_GPU = 16
HW = 512
METRIC = "unet_vgg16_512x512_train_img_per_s"
WORKLOAD = ("Unet-VGG16 21-class 512x512 training step (fwd + CE + Dice + f_score + bwd + grad all-reduce + Adam), "
            "batch 16 per GPU, BASELINE configs[1]")
# fprop + dgrad + wgrad conv FLOPs per image (SURVEY.md 8d)
TRAIN_GFLOP_PER_IMG = 1351.99
# parameter / gradient values per --dump-outputs array: 16 MB each in float32
DUMP_SAMPLE = 1 << 22


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16_sustained": d.get("bf16_tflops_sustained", 1381.4), "bf16_burst": d.get("bf16_tflops", 1659.2),
                "hbm": d.get("hbm_gbs", 6556.2), "source": "measured"}
    return {"bf16_sustained": 1400.0, "bf16_burst": 1590.0, "hbm": 6650.0, "source": "fallback"}


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(power), "samples": len(sm),
                "reasons": sorted(reasons)}



class OperandBytes:
    """Counts, for ONE step, the bytes of every tensor operand that goes through the ops.* wrappers (inputs, outputs, `out=`
    buffers; workspaces excluded; each tensor once per call) -- the ALGORITHMIC HBM traffic of the step as the engine issues
    it: what `achieved HBM GB/s` of the memory-bound model families is quoted on."""
    SKIP_KW = {"ws"}

    def __init__(self, ops):
        self.ops, self.total, self.saved = ops, 0, {}

    def _count(self, args, kwargs, ret):
        import torch
        seen = set()

        def visit(x):
            if isinstance(x, torch.Tensor) and x.is_cuda:
                if x.data_ptr() not in seen:
                    seen.add(x.data_ptr())
                    self.total += x.numel() * x.element_size()
            elif isinstance(x, (tuple, list)):
                for y in x:
                    visit(y)
        visit(args)
        for k, v in kwargs.items():
            if k not in self.SKIP_KW:
                visit(v)
        visit(ret)

    def __enter__(self):
        import types
        for name in dir(self.ops):
            fn = getattr(self.ops, name)
            if isinstance(fn, types.FunctionType) and fn.__module__ == self.ops.__name__ and not name.startswith("_") and name not in (
                    "act_dtype", "set_timer", "set_validation_fp32", "conv_stat_rows", "lib", "check", "ptr", "stream_ptr"):
                self.saved[name] = fn

                def wrapped(*a, __fn=fn, **kw):
                    r = __fn(*a, **kw)
                    self._count(a, kw, r)
                    return r
                setattr(self.ops, name, wrapped)
        return self

    def __exit__(self, *exc):
        for name, fn in self.saved.items():
            setattr(self.ops, name, fn)


def dump_outputs(trainer, out, path):
    """What the last timed step hands its caller: the [loss, f_score] it returns and the model state it leaves behind --
    the updated parameters and the gradients it applied (summed over ranks), concatenated in state_dict order.  Of those
    24.9 M values, DUMP_SAMPLE fixed positions (numpy Generator seeded 0, sorted) are written."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    params = torch.cat([trainer.params[n].reshape(-1) for n in trainer.names])
    grads = torch.cat([trainer.grads[n].reshape(-1) for n in trainer.names])
    idx = np.sort(np.random.default_rng(0).choice(params.numel(), size=min(DUMP_SAMPLE, params.numel()), replace=False))
    idx = torch.from_numpy(idx).to(params.device)
    arrays = {"loss": out[0], "f_score": out[1], "params_sample": params[idx], "grads_sample": grads[idx]}
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.detach().float().cpu().numpy())


def _ev_ms(fn, iters, warm):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def side_measurements(b2u, ops, dev, peaks):
    """BASELINE configs[2..4] next to the headline line (VERDICT r1 item 8), compact: ~40 s.
      train          Unet-ResNet50 (21 classes), LightweightUnet, UltraLightweightUnet_large (2 classes): batch 16, 512x512, full
                     training step; img/s and achieved HBM GB/s of the step's algorithmic operand bytes (OperandBytes)
      fps            predict.py fps mode (unet.py:240-257): uint8 frame(s) H2D -> /255 -> forward -> per-pixel class -> uint8 mask
                     D2H, batch 1 (eager launches, and replayed from a CUDA graph) and batch 64
      fast_hist      get_miou's confusion matrix over 1000 distinct 512x512 uint8 mask pairs (524 MB > L2), n = 21 and 2
      gpu_library_baseline   the same headline step written with stock torch.nn and run by PyTorch eager + cuDNN (bf16 autocast,
                     channels_last, cudnn.benchmark, fused Adam) on this GPU: the library kernels to beat"""
    import numpy as np
    import torch
    out = {}
    # ---- other families
    train = {}
    for model, C in (("unet_resnet50", 21), ("lightweight", 2), ("ultralight_large", 2)):
        tr = b2u.UnetTrainer(num_classes=C, device=dev, model=model, lr=1e-4)
        imgs, pngs = b2u.synthetic.make_inputs(BATCH_PER_GPU, C, HW, HW, seed=3)
        imgs, pngs = imgs.to(dev), pngs.to(dev)
        ms = _ev_ms(lambda: tr.train_step(imgs, pngs), 8, 3)
        with OperandBytes(ops) as ob:
            tr.train_step(imgs, pngs)
        torch.cuda.synchronize()
        gb = ob.total / 1e9
        train[model] = {"classes": C, "img_per_s": BATCH_PER_GPU * 1e3 / ms, "ms_per_step": ms, "algorithmic_gb_per_step": gb,
                        "achieved_hbm_gbps": gb / (ms / 1e3), "frac_of_hbm_peak": gb / (ms / 1e3) / peaks["hbm"]}
        tr.engine.release()
        del tr
        torch.cuda.empty_cache()
    out["train_batch16_512"] = train
    # ---- fps mode
    C = NUM_CLASSES
    model = b2u.Unet(num_classes=C)
    model.load_state_dict(b2u.synthetic.make_params(C))
    model = model.to(dev).eval()
    fps = {}
    for B in (1, 64):
        frames = torch.randint(0, 256, (B, HW, HW, 3), dtype=torch.uint8).pin_memory()
        dframes = torch.empty_like(frames, device=dev)
        x32 = torch.empty((B, 3, HW, HW), dtype=torch.float32, device=dev)
        mask = torch.empty((B, HW, HW), dtype=torch.uint8, device=dev)
        host = torch.empty((B, HW, HW), dtype=torch.uint8).pin_memory()

        def body():
            with torch.no_grad():
                ops.u8hwc_to_nchw_f32(dframes, out=x32)
                ops.argmax_hist(model(x32), pred=mask)

        def frame():
            dframes.copy_(frames, non_blocking=True)
            body()
            host.copy_(mask, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        ms = _ev_ms(frame, 30 if B == 1 else 4, 3)
        fps[f"b{B}"] = {"fps": B * 1e3 / ms, "ms_per_call": ms, "h2d_bytes": frames.numel(), "d2h_bytes": host.numel()}
        if B == 1:
            try:        # the ~30 launches of a batch-1 frame replayed from one CUDA graph
                side = torch.cuda.Stream(device=dev)
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    body()
                torch.cuda.current_stream().wait_stream(side)
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    body()
                ref_mask = mask.clone()

                def gframe():
                    dframes.copy_(frames, non_blocking=True)
                    graph.replay()
                    host.copy_(mask, non_blocking=True)
                    torch.cuda.current_stream().synchronize()
                msg = _ev_ms(gframe, 30, 3)
                fps["b1_cuda_graph"] = {"fps": 1e3 / msg, "ms_per_call": msg, "same_mask": bool(torch.equal(mask, ref_mask))}
            except Exception as e:      # measurement aid only
                fps["b1_cuda_graph"] = {"error": str(e)[:200]}
    out["fps_mode_uint8_frames"] = fps
    for e in model._engines.values():
        e.release()
    del model
    torch.cuda.empty_cache()
    # ---- fast_hist over 1000 distinct masks
    hist_res = {}
    for n in (21, 2):
        g = torch.Generator(device=dev).manual_seed(n)
        gt = torch.randint(0, n, (1000, HW, HW), dtype=torch.uint8, device=dev, generator=g)
        pred = torch.where(torch.rand((1000, HW, HW), device=dev, generator=g) < 0.2,
                           torch.randint(0, n, (1000, HW, HW), dtype=torch.uint8, device=dev, generator=g), gt)
        gt = torch.where(torch.rand((1000, HW, HW), device=dev, generator=g) < 0.03, torch.full_like(gt, 255), gt)
        hist = torch.zeros(n * n + 1, dtype=torch.int64, device=dev)
        ms_one = _ev_ms(lambda: ops.fast_hist_accumulate(gt.reshape(-1), pred.reshape(-1), n, hist), 5, 2)
        pairs = [(gt[i].reshape(-1), pred[i].reshape(-1)) for i in range(1000)]
        table = ops.HistTable(pairs, dev)            # device pointer table, built once per evaluation set
        ms_tab = _ev_ms(lambda: ops.fast_hist_batch(table, n, hist), 5, 2)
        hist.zero_()
        ops.fast_hist_batch(table, n, hist)
        got = hist.cpu().numpy()
        keep = gt < n
        want = torch.bincount(gt[keep].long() * n + pred[keep].long(), minlength=n * n).cpu().numpy()
        gbytes = 2 * gt.numel() / 1e9
        hist_res[f"n{n}"] = {"masks": 1000, "bit_exact_vs_bincount": bool(got[-1] == 0 and np.array_equal(got[:-1], want)),
                             "one_call_ms": ms_one, "one_call_gbps": gbytes / (ms_one / 1e3), "frac_of_hbm_peak": gbytes / (ms_one / 1e3) / peaks["hbm"],
                             "pointer_table_ms": ms_tab, "pointer_table_gbps": gbytes / (ms_tab / 1e3), "masks_per_s": 1e6 / ms_tab}
        del gt, pred, pairs, keep, table
        torch.cuda.empty_cache()
    out["fast_hist_1k_masks_512"] = hist_res
    # ---- library yardstick
    try:
        sys.path.insert(0, os.path.join(ROOT, "scripts"))
        import torch_eager_baseline as TE
        out["gpu_library_baseline"] = TE.measure(steps=8, batch=BATCH_PER_GPU)
    except Exception as e:
        out["gpu_library_baseline"] = {"error": str(e)[:200]}
    return out


def variant_cpu_img_per_s(model, num_classes, batch=2, hw=HW, steps=1, warmup=1, threads=None):
    """cpu_baseline leg of the side measurements (scripts/variants_bench.py): the oracle port of another model family's
    forward + CE + Dice + backward on this box's host cores, `batch` images per step -> img/s."""
    import torch
    from oracle import unet_oracle as O
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    imgs, pngs = O.make_inputs(batch, num_classes, hw, hw, seed=0)
    w = torch.ones(num_classes)
    if model == "unet_vgg":
        sd = O.make_params(num_classes)
        step = lambda: O.train_step(sd, imgs, pngs, w, num_classes)
    elif model == "unet_resnet50":
        sd = O.make_resnet_unet_params(num_classes)
        step = lambda: O.resnet_unet_train_step(sd, imgs, pngs, w, num_classes)
    elif model == "traditional":
        sd = O.make_trad_params(num_classes)
        step = lambda: O.trad_train_step(sd, imgs, pngs, w, num_classes)
    elif model == "lightweight":
        sd = O.make_lw_params(num_classes)
        step = lambda: O.lw_train_step(sd, imgs, pngs, w, num_classes)
    elif model.startswith("ultralight"):
        sd = O.make_ulu_params(num_classes, model)
        step = lambda: O.ulu_train_step(sd, imgs, pngs, w, num_classes, model)
    else:
        raise ValueError(model)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        step()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    return {"value": batch / (sum(times) / len(times)), "unit": "img/s", "cores": threads, "kind": "port",
            "sample": f"{steps} step(s) of batch {batch} at {hw}x{hw}, fwd + CE + Dice + bwd (no optimizer), after {warmup} warm-up"}


def cpu_path_img_per_s(steps, warmup, batch=2, threads=None):
    """The reference's own CPU path for this workload, bounded sample: `batch` images per step.
    One step = forward, CE + Dice, f_score (no grad), backward, Adam -- the same work the GPU arm times.
    kind "reference": the UNMODIFIED reference (nets.unet.Unet, nets.unet_training.CE_Loss / Dice_loss,
    utils.utils_metrics.f_score staged under baseline/_ref/ by baseline/stage_ref.py) on torch CPU fp32;
    kind "port": the oracle restatement, only when the staged copy is absent."""
    import torch
    from oracle import unet_oracle as O
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    imgs, pngs = O.make_inputs(batch, NUM_CLASSES, HW, HW, seed=0)
    labels = O.one_hot(pngs, NUM_CLASSES)
    w = torch.ones(NUM_CLASSES)
    kind = "port"
    try:
        from baseline import stage_ref
        if stage_ref.stage() is not None and stage_ref.available():
            kind = "reference"
    except Exception:
        kind = "port"
    if kind == "reference":
        RU = stage_ref.import_reference("nets.unet")
        RT = stage_ref.import_reference("nets.unet_training")
        RM = stage_ref.import_reference("utils.utils_metrics")
        torch.manual_seed(11)
        model = RU.Unet(num_classes=NUM_CLASSES, pretrained=False, backbone="vgg").train()
        model.load_state_dict(O.make_params(NUM_CLASSES, seed=11))
        opt = torch.optim.Adam(model.parameters(), lr=1e-4, betas=(0.9, 0.999))

        def step():
            opt.zero_grad()
            logits = model(imgs)
            loss = RT.CE_Loss(logits, pngs, w, num_classes=NUM_CLASSES) + RT.Dice_loss(logits, labels)
            with torch.no_grad():
                RM.f_score(logits, labels)
            loss.backward()
            opt.step()
            return loss.item()
    else:
        params = {k: v.clone().requires_grad_(True) for k, v in O.make_params(NUM_CLASSES, seed=11).items()}
        opt = torch.optim.Adam(list(params.values()), lr=1e-4, betas=(0.9, 0.999))

        def step():
            opt.zero_grad()
            logits = O.unet_forward(params, imgs)
            loss = O.ce_loss(logits, pngs, w, NUM_CLASSES) + O.dice_loss(logits, labels)
            with torch.no_grad():
                O.f_score(logits, labels)
            loss.backward()
            opt.step()
            return loss.item()
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    total = sum(times)
    return batch * len(times) / total, total / len(times), threads, batch, kind


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = args.steps
    warmup = 1 if args.warmup > 0 else 0
    v, s_per_step, threads, batch, kind = cpu_path_img_per_s(steps, warmup)
    cpu_model = ""
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                cpu_model = ln.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    what = ("the unmodified reference staged under baseline/_ref (nets.unet.Unet, CE_Loss, Dice_loss, f_score)" if kind == "reference"
            else "the oracle port (reference not staged)")
    sample = (f"{steps} timed step(s) of batch {batch} (of the 16-image batch), 512x512, 21 classes, fp32 torch CPU, {what}, "
              f"fwd + CE + Dice + f_score + bwd + Adam, after {warmup} warm-up; {cpu_model}")
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "img/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": s_per_step * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": BATCH_PER_GPU, "global_batch": BATCH_PER_GPU * args.gpus,
                       "parallelism": f"dp{args.gpus}",
                       "sample": f"CPU arm: each step is a bounded sample of {batch} of the {BATCH_PER_GPU} images, same work per image as the GPU arm"},
            "cpu_baseline": {"value": v, "unit": "img/s", "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": v, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def run_ours(args):
    import torch
    import torch.distributed as dist
    import unet_pytorch_b200 as b2u
    from unet_pytorch_b200 import ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    peaks = _peaks()
    K, W = args.steps, args.warmup
    B = args.batch

    params = b2u.synthetic.make_params(NUM_CLASSES, seed=11)
    trainer = b2u.UnetTrainer(num_classes=NUM_CLASSES, device=dev, lr=1e-4, betas=(0.9, 0.999), state_dict=params,
                              bucket_mb=int(os.environ.get("B2U_BUCKET_MB", "16")),      # experiment knob (all-reduce bucket size)
                              dice_loss=True)
    # a few distinct resident batches, different per rank (DistributedSampler semantics)
    nb = 2
    host = [b2u.synthetic.make_inputs(B, NUM_CLASSES, HW, HW, seed=100 * rank + i) for i in range(nb)]
    host = [(i.pin_memory(), p.pin_memory()) for i, p in host]
    resident = [(i.to(dev), p.to(dev)) for i, p in host]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            if os.environ.get("B2U_RANK_TIMES"):          # diagnostic: every rank's own time on stderr
                print(f"[rank {rank}] {ms:.3f} ms", file=sys.stderr, flush=True)
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return t.item()
        return ms

    # ---------------- device-resident leg (value) + roofline timing of the conv launches
    for i in range(W):
        trainer.train_step(*resident[i % nb])
    barrier()
    lib = b2u._lib.lib()
    lib.b2u_reset_launch_count()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        out = trainer.train_step(*resident[i % nb])
    e1.record()
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    launches = int(lib.b2u_launch_count())
    clocks = sampler.stop() if rank == 0 else None
    loss_val = out.tolist()
    if args.dump_outputs and rank == 0:
        dump_outputs(trainer, out, args.dump_outputs)
    if args.kernels_only:
        if rank == 0:
            print(json.dumps({"kernels_only": True, "note": "profiling pass, not a bench value", "steps": K, "warmup": W,
                              "ms_per_step": ms_total / K, "gpu_launches": launches}))
        if world > 1:
            dist.destroy_process_group()
        return

    # per-launch timing of the tensor-core kernels (separate pass: the events add launch gaps)
    timer = ops.KernelTimer()
    ops.set_timer(timer)
    tsteps = max(1, min(K, 5))
    for i in range(tsteps):
        trainer.train_step(*resident[i % nb])
    kt = timer.read()
    ops.set_timer(None)

    # ---------------- end-to-end leg: host batches, H2D + D2H inside the timed region
    h2d = host[0][0].numel() * host[0][0].element_size() + host[0][1].numel() * host[0][1].element_size()
    for i in range(min(W, 3)):
        trainer.stage(*host[i % nb])
        trainer.train_step().tolist()
    barrier()
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    trainer.stage(*host[0])
    for i in range(K):
        res = trainer.train_step()                 # consumes the staged batch (waits for its copy)
        if i + 1 < K:
            trainer.stage(*host[(i + 1) % nb])     # next batch's H2D overlaps this step's kernels
        res = res.tolist()                         # D2H read of [loss, f_score], per-iteration sync (utils_fit.py:96)
    t1.record()
    barrier()
    ms_e2e = max_over_ranks(t0.elapsed_time(t1))

    # ---------------- the same loop fed with RAW uint8 batches (NHWC image, uint8 label map): /255, CHW and the int64
    # map are produced on the device (SURVEY.md 8(f) rank 3) -- 4 B/pixel over PCIe instead of 20
    host_u8 = [((im.permute(0, 2, 3, 1) * 255.0).round().to(torch.uint8).contiguous().pin_memory(),
                pn.to(torch.uint8).contiguous().pin_memory()) for im, pn in host]
    h2d_u8 = host_u8[0][0].numel() + host_u8[0][1].numel()
    for i in range(min(W, 3)):
        trainer.stage(*host_u8[i % nb])
        trainer.train_step().tolist()
    barrier()
    u0 = torch.cuda.Event(enable_timing=True); u1 = torch.cuda.Event(enable_timing=True)
    u0.record()
    trainer.stage(*host_u8[0])
    for i in range(K):
        res = trainer.train_step()
        if i + 1 < K:
            trainer.stage(*host_u8[(i + 1) % nb])
        res = res.tolist()
    u1.record()
    barrier()
    ms_e2e_u8 = max_over_ranks(u0.elapsed_time(u1))

    # data-parallel invariant: after all these steps every rank must hold bit-identical parameters (train.py:346: DDP)
    dp_diff = None
    if world > 1:
        ref_p = trainer.flat_param.clone()
        dist.broadcast(ref_p, src=0)
        d = (trainer.flat_param - ref_p).abs().max().reshape(1)
        dist.all_reduce(d, op=dist.ReduceOp.MAX)
        dp_diff = float(d.item())
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    variants = None
    if world == 1 and not args.no_variants:
        trainer.engine.release()
        torch.cuda.empty_cache()
        variants = side_measurements(b2u, ops, dev, peaks)

    imgs_total = B * world * K
    value = imgs_total / (ms_total / 1e3)
    e2e_value = imgs_total / (ms_e2e / 1e3)
    def agg(prefix):
        recs = [v for k, v in kt.items() if k.startswith(prefix + "|")]
        return {"launches": sum(r["launches"] for r in recs), "ms": sum(r["ms"] for r in recs),
                "flops": sum(r["flops"] for r in recs)}
    ig, wg = agg("conv_igemm"), agg("conv_wgrad")
    if args.detail:
        rows = [{"kernel": k, "launches": v["launches"], "avg_ms": v["ms"] / v["launches"],
                 "tflops": v["flops"] / (v["ms"] / 1e3) / 1e12, "share_of_conv_ms": v["ms"] / (ig["ms"] + wg["ms"])}
                for k, v in sorted(kt.items(), key=lambda kv: -kv[1]["ms"])]
        with open(args.detail, "w") as f:
            json.dump({"steps_timed": tsteps, "rows": rows}, f, indent=1)

    traffic = {}
    for name in ("r2_traffic.json", "r1_traffic.json"):      # the latest committed ncu capture of this command
        tp = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tp):
            traffic = json.load(open(tp))
            break

    def roof(rec, traffic=None):
        if rec["ms"] <= 0:
            return None
        ach = rec["flops"] / (rec["ms"] / 1e3) / 1e12
        return {"bound": "tensor", "achieved": ach, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                "frac": ach / peaks["bf16_sustained"], "traffic": traffic, "peak_source": peaks["source"] + " (sustained)",
                "launches_timed": rec["launches"], "avg_launch_ms": rec["ms"] / max(rec["launches"], 1),
                "flops_per_launch": rec["flops"] / max(rec["launches"], 1)}

    line = {
        "metric": METRIC, "value": value, "unit": "img/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "batch_per_gpu": B, "global_batch": B * world, "parallelism": f"dp{world}",
                   "l2": "inputs larger than L2 (>= 4.7 GB of activations per step), no explicit flush"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "img/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 8,
                "ms_per_step": ms_e2e / K},
        "e2e_u8_inputs": {"value": imgs_total / (ms_e2e_u8 / 1e3), "unit": "img/s", "h2d_bytes_per_step": h2d_u8,
                          "d2h_bytes_per_step": 8, "ms_per_step": ms_e2e_u8 / K,
                          "note": "raw uint8 NHWC images + uint8 label maps; /255, CHW, int64 map on the device"},
        "gpu_launches": launches,
        # traffic: DRAM bytes per launch from the committed ncu capture of this same command (profiles/r2_traffic.json)
        "roofline": roof(ig, traffic.get("conv_igemm", {}).get("dram_bytes_per_launch")),
        "roofline_wgrad": roof(wg, traffic.get("conv_wgrad", {}).get("dram_bytes_per_launch")),
        "model_tflops": value * TRAIN_GFLOP_PER_IMG / 1e3 / world,
        "loss": loss_val[0], "f_score": loss_val[1],
    }
    if dp_diff is not None:
        line["dp_param_max_diff"] = dp_diff          # max over ranks of |param - rank 0's param| after the run: must be 0
    if variants is not None:
        line["variants"] = variants
    if world == 1 and not args.no_cpu_baseline:
        v, s_per_step, threads, batch, kind = cpu_path_img_per_s(2, 1)
        what = "the unmodified reference (baseline/_ref: nets.unet.Unet + CE_Loss + Dice_loss + f_score)" if kind == "reference" else "the oracle port"
        line["cpu_baseline"] = {"value": v, "unit": "img/s", "cores": threads, "kind": kind,
                                "sample": f"2 timed steps of batch {batch} (512x512, 21 classes, fp32 torch CPU, {what}, "
                                          f"fwd + CE + Dice + f_score + bwd + Adam) after 1 warm-up, {s_per_step:.2f} s/step"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=BATCH_PER_GPU, help="images per GPU per step (BASELINE: 16)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-variants", action="store_true", help="skip the side measurements of BASELINE configs[2..4] (variants key)")
    ap.add_argument("--kernels-only", action="store_true",
                    help="profiling pass (ncu): warm-up + the K device-resident steps, nothing else; prints a reduced line that is NOT a bench value")
    ap.add_argument("--detail", default=None, help="write the per-layer conv kernel timing table (JSON) here")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last timed step's loss, f_score and a fixed sample of the updated "
                         "parameters and of the gradients as DIR/<name>.npy (float32, 32 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the product path (--impl ours)")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
