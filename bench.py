#!/usr/bin/env python
"""bench.py -- the BASELINE.json metric (images/s of the DINOv2 -> hard-VLAD descriptor pipeline) plus the
retrieval configurations, on N GPUs of one node.

    python bench.py --gpus N --steps K --warmup W                  # this repo (CUDA, sm_100a), workload c2
    python bench.py --impl reference --gpus N --steps K ...         # the reference's CPU path (oracle port)
    python bench.py --workload c3|c4 ...                            # retrieval: 10k / 100k-image database, 1k queries

Pipeline workloads (c1 / c2 / c5).  A step = one pass of the hot path over one batch of synthetic images per
GPU -- DinoV2ExtractFeatures.__call__ (ViT forward, early exit at the hooked layer) -> VLAD.generate_multi --
followed by the pipeline's one data-path collective: the all-gather of that batch's [B, K*D] descriptors into the
database every rank keeps for retrieval (BASELINE config 4: "NCCL all-gather of the 49152-D descriptors before
top-k"; scripts/dino_v2_vlad.py:219-264 builds the database VLADs, utilities.py:435-450 searches them).  The
all-gather of step i is enqueued asynchronously and overlaps the ViT of step i+1; the timed region ends when every
gather has landed.  N=1: the gather degenerates to the copy into the database buffer.  Weak scaling: per-GPU batch
fixed.  After the timed loops the gathered database is checked bitwise against the local descriptors and searched
with both sharded top-k strategies (anyloc_b200/dist.py).

Retrieval workloads (c3 / c4).  A step = descriptor all-gather (c4) + database index build + 1k-query top-5
search, queries sharded over the ranks, results gathered.

Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    "c1": dict(kind="pipeline", model="dinov2_vits14", layer=9, facet="value", H=224, W=224, K=8, B=16,
               name="c1: ViT-S/14 layer-9 value, 224x224, K=8 VLAD, batch 16"),
    "c2": dict(kind="pipeline", model="dinov2_vitg14", layer=31, facet="value", H=322, W=322, K=32, B=32,
               name="c2: ViT-G/14 layer-31 value, 322x322, K=32 VLAD, batch 32"),
    "c5": dict(kind="pipeline", model="dinov2_vitl14", layer=20, facet="value", H=518, W=518, K=128, B=64,
               name="c5: ViT-L/14 layer-20 value, 518x518, K=128 VLAD, batch 64"),
    "c3": dict(kind="retrieval", n_db_per_rank=10000, n_q=1000, Dv=49152, k=5,
               name="c3: 10k-image database of 49152-D (ViT-G K=32) VLADs, 1k-query cosine top-5, 1 GPU"),
    "c4": dict(kind="retrieval", n_db_per_rank=12500, n_q=1000, Dv=49152, k=5,
               name="c4: 12.5k-image database shard per GPU (100k images at 8 GPUs) of 49152-D VLADs, NCCL all-gather, "
                    "1k-query cosine top-5"),
}
METRIC = "images/sec end-to-end DINOv2-VLAD descriptors"
UNIT = "images/s"
NVLINK_GBS_PER_DIR = 900.0      # B200 NVLink 5 per GPU per direction (B200_PROFILING.md / task statement)


def vit_flops_per_image(model, layer, H, W):
    """SURVEY.md 8(d): 2*N*588*D + L*(24*T*D^2 + 4*T^2*D) + 2*T*D^2 (early-exit form)."""
    from anyloc_b200.vit import ARCHS, ffn_hidden
    D, _, _, kind = ARCHS[model]
    N = (H // 14) * (W // 14)
    T = N + 1
    hid = ffn_hidden(D, kind)
    ffn = (2 * T * D * 2 * hid + 2 * T * hid * D) if kind != "mlp" else 4 * T * D * hid
    per_block = 2 * T * D * 3 * D + 2 * T * D * D + 4 * T * T * D + ffn
    return 2 * N * 588 * D + layer * per_block + 2 * T * D * D


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        p = json.load(open(path))
        return dict(hbm_gbs=p["hbm_gbs"], tflops_burst=p["bf16_tflops"],
                    tflops_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, tflops_burst=1590.0, tflops_sustained=1400.0, source="fallback")


def usable_cores():
    """Host threads this process can really use: min(affinity, cgroup CPU quota).  (On the GPU boxes
    os.cpu_count() says 128 while cpu.max grants 16 CPUs; 128 threads then run 40x slower.)"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // p))
        except Exception:
            pass
    return n


def ncu_traffic(kernel_substrs, tag, per_call=False):
    """DRAM bytes (read + write) of the kernels whose name contains one of `kernel_substrs`, from the committed
    `ncu --set full ... --page raw --csv` export profiles/r*_ncu_<tag>_raw.csv (newest round first): the mean per launch, or
    with per_call the sum over the distinct kernels of their per-launch means (a call = one launch of each).
    -> (bytes, file) or (None, None)."""
    import csv
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", f"r*_ncu_{tag}_raw.csv")), reverse=True):
        try:
            rows = list(csv.reader(open(path, newline="")))
            hdr = next(i for i, r in enumerate(rows) if "Kernel Name" in r)
            h, units = rows[hdr], rows[hdr + 1]
            kn, rd, wr = h.index("Kernel Name"), h.index("dram__bytes_read.sum"), h.index("dram__bytes_write.sum")
        except Exception:
            continue
        scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        per_kernel = {}
        for r in rows[hdr + 2:]:
            if len(r) <= max(kn, rd, wr) or not any(k in r[kn] for k in kernel_substrs):
                continue
            v = float(r[rd].replace(",", "")) * scale.get(units[rd], 1.0) + float(r[wr].replace(",", "")) * scale.get(units[wr], 1.0)
            per_kernel.setdefault(r[kn].split("(")[0], []).append(v)
        if per_kernel:
            means = [sum(v) / len(v) for v in per_kernel.values()]
            allv = [x for v in per_kernel.values() for x in v]
            return (sum(means) if per_call else sum(allv) / len(allv)), os.path.relpath(path, ROOT)
    return None, None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons, power = [], [], set(), []
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------ reference arm / cpu baseline
_REF_MODELS = {}


def _ref_model(name, seed=0):
    """the restated hub model with ALL blocks (the reference runs them all), built once per process"""
    from oracle import dinov2_restated as dr
    if (name, seed) not in _REF_MODELS:
        _REF_MODELS[(name, seed)] = dr.build(name, seed=seed)
    return _REF_MODELS[(name, seed)]


def cpu_reference(wl, n_images, steps, warmup, seed=0):
    """The reference's own CPU path, restated (oracle/): per image, batch 1, the FULL model forward
    with the facet hook (scripts/dino_v2_vlad.py:164-188 -> utilities.py:263-285), then
    VLAD.generate per image with the [N,K,D] residual tensor (utilities.py:819-890, :956-962).
    Returns (images_per_s, ms_per_step, cores)."""
    import torch
    from oracle import anyloc_oracle as ao
    cores = usable_cores()
    torch.set_num_threads(cores)
    model = _ref_model(wl["model"], seed)
    D = model.embed_dim
    g = torch.Generator().manual_seed(1234)
    imgs = torch.randn(n_images, 3, wl["H"], wl["W"], generator=g)
    centers = 0.6 * torch.nn.functional.normalize(torch.randn(wl["K"], D, generator=g), dim=1)

    def one_step():
        feats = [ao.extract_features_full_forward(model, imgs[i:i + 1], wl["layer"], wl["facet"]) for i in range(n_images)]
        feats = torch.cat(feats)
        return torch.stack([ao.vlad_generate_faithful(f, centers) for f in feats])

    for _ in range(warmup):
        one_step()
    t0 = time.perf_counter()
    for _ in range(steps):
        one_step()
    dt = time.perf_counter() - t0
    return n_images * steps / dt, dt / steps * 1e3, cores


def gpu_reference(wl, n_images, seed=0):
    """The north star's 10x denominator -- 'the reference GPU PyTorch path' on this GPU: the loop of
    scripts/dino_v2_vlad.py:164-188,233-237 with the restated hub model .cuda() in fp32 (TF32 off, as torch's
    defaults), ONE image per forward (all blocks + hook), `.cpu()` per image, then the CPU VLAD.generate per image
    (oracle restatement with the [N,K,D] residuals).  torch / cuBLAS kernels only -- none of this repo's.
    Returns (images_per_s, ms_per_image_vit_part)."""
    import torch
    from oracle import anyloc_oracle as ao
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.set_num_threads(usable_cores())
    model = _ref_model(wl["model"], seed).cuda()
    try:
        g = torch.Generator().manual_seed(1234)
        imgs = torch.randn(n_images, 3, wl["H"], wl["W"], generator=g)
        centers = 0.6 * torch.nn.functional.normalize(torch.randn(wl["K"], model.embed_dim, generator=g), dim=1)

        def path(n, vlad=True):
            feats = [ao.extract_features_full_forward(model, imgs[i:i + 1].cuda(), wl["layer"], wl["facet"]).cpu()
                     for i in range(n)]
            return torch.stack([ao.vlad_generate_faithful(f, centers) for f in torch.cat(feats)]) if vlad else None

        path(2)
        torch.cuda.synchronize(); t0 = time.perf_counter()
        path(n_images)
        torch.cuda.synchronize(); t_all = time.perf_counter() - t0
        t0 = time.perf_counter()
        path(n_images, vlad=False)
        torch.cuda.synchronize(); t_vit = time.perf_counter() - t0
    finally:
        model.cpu()
        torch.cuda.empty_cache()
    return n_images / t_all, t_vit / n_images * 1e3


def run_reference_arm(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if wl["kind"] != "pipeline":
        print(json.dumps({"impl": "reference", "unavailable": "the reference arm times the descriptor pipeline (c1/c2/c5) only"}))
        return
    n = args.ref_images
    ips, ms, cores = cpu_reference(wl, n, args.steps, max(args.warmup, 1))
    sample = f"{n} of {wl['B']} images per step, batch 1 per image, all blocks + hook, CPU VLAD with [N,K,D] residuals"
    line = {"impl": "reference", "metric": METRIC, "value": ips, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["name"], "sample": sample},
            "cpu_baseline": {"value": ips, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": ips, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------ shared plumbing of our arms
class Ranks:
    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device (anyloc_b200 has no CPU fallback); use --impl reference")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()

    def max_ms(self, ms):
        if self.world == 1:
            return ms
        t = self.torch.tensor([ms], device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def all_true(self, flag):
        if self.world == 1:
            return bool(flag)
        t = self.torch.tensor([1 if flag else 0], device=self.dev, dtype=self.torch.int32)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return bool(t.item())

    def timed(self, fn, steps):
        """barrier + synchronize on both sides, CUDA events on the current stream, max over ranks -> total ms"""
        torch = self.torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        self.barrier()
        return self.max_ms(e0.elapsed_time(e1))

    def finish(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def dump_outputs(dirpath, tensors):
    """--dump-outputs: each tensor as DIR/<name>.npy, floats as float32, integers (indices) as float64, which holds
    them exactly.  The largest dump, c5's [64, 131072] descriptors, is 34 MB."""
    import numpy as np
    os.makedirs(dirpath, exist_ok=True)
    for name, t in tensors.items():
        a = t.detach().cpu().numpy()
        np.save(os.path.join(dirpath, name + ".npy"), a.astype(np.float32 if a.dtype.kind == "f" else np.float64))


def collective_alone(R, shape, iters=10):
    """the step's all-gather timed on its own: -> (us per call, bus GB/s per rank = received bytes / time)"""
    torch, dist = R.torch, R.dist
    if R.world == 1:
        return None, None
    src = torch.randn(*shape, device=R.dev)
    dst = torch.empty((R.world * shape[0],) + tuple(shape[1:]), device=R.dev)
    for _ in range(3):
        dist.all_gather_into_tensor(dst, src)
    ms = R.timed(lambda i: dist.all_gather_into_tensor(dst, src), iters) / iters
    recv = (R.world - 1) * src.numel() * 4
    return ms * 1e3, recv / (ms / 1e3) / 1e9


# ------------------------------------------------------------------ descriptor pipeline (c1 / c2 / c5)
def run_pipeline(args, wl):
    import numpy as np
    R = Ranks()
    torch, dist, dev, world, rank = R.torch, R.dist, R.dev, R.world, R.rank
    from anyloc_b200 import _lib, dist as adist, utilities as u
    from anyloc_b200.vit import random_state_dict, ARCHS

    B, H, W, K = wl["B"], wl["H"], wl["W"], wl["K"]
    D = ARCHS[wl["model"]][0]
    Dv = K * D
    sd = random_state_dict(wl["model"], seed=0, device=dev, depth=wl["layer"] + 1)
    ext = u.DinoV2ExtractFeatures(wl["model"], wl["layer"], wl["facet"], device=dev, weights=sd,
                                  gemm_engine=args.engine, precision=args.precision)
    ext.check_finite = "deferred"            # fp16-range guard without a host sync per call; checked after the loops
    sd_host = None
    if rank == 0 and world == 1 and not args.no_parity_check:
        sd_host = {k: v.cpu() for k, v in sd.items()}
    del sd
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    img_dev = torch.randn(B, 3, H, W, device=dev, generator=g)
    img_host = img_dev.cpu().pin_memory()
    feats = ext(img_dev)
    np.random.seed(42)
    vlad = u.VLAD(K)
    if args.vocab == "fit":
        vlad.fit(feats.reshape(-1, D))      # vocabulary on this batch's features (GPU k-means)
        if world > 1:                       # replicated vocabulary: rank 0's
            c = vlad.c_centers.contiguous()
            dist.broadcast(c, 0)
            vlad.c_centers = vlad.kmeans.centroids = c
    else:                                   # profiling runs: skip the k-means launches
        vlad.kmeans = u._KMeans(K, mode="cosine")
        idx = torch.randperm(feats.shape[0] * feats.shape[1], device=dev, generator=g)[:K]
        vlad.c_centers = vlad.kmeans.centroids = 0.7 * feats.reshape(-1, D)[idx].contiguous()
        vlad.desc_dim = D
    del feats
    out_host = [torch.empty(B, Dv, dtype=torch.float32).pin_memory() for _ in range(2)]
    # the database every rank keeps for retrieval: a ring of the last SLOTS gathered step chunks [world*B, Dv]
    SLOTS = 4
    db_ring = torch.zeros(SLOTS, world * B, Dv, device=dev)
    pending = []

    def gather(desc, i):
        """the pipeline's one collective: this step's [B, Dv] descriptors of every rank -> database chunk i"""
        slot = db_ring[i % SLOTS]
        if world == 1:
            slot.copy_(desc)
            return
        while len(pending) >= SLOTS - 1:      # chunk i reuses the slot of chunk i - SLOTS: that gather must be done
            pending.pop(0).wait()
        pending.append(dist.all_gather_into_tensor(slot, desc, async_op=True))

    def drain():
        while pending:
            pending.pop(0).wait()

    def step_device(i):
        desc = vlad.generate_multi(ext(img_dev))
        gather(desc, i)
        return desc

    e2e_marks = []          # (before H2D, after H2D, after compute + gather launch, after D2H) events per e2e step

    def step_e2e(i):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        x = img_host.to(dev, non_blocking=True)                    # H2D of this step's inputs
        ev[1].record()
        desc = vlad.generate_multi(ext(x))
        gather(desc, i)
        ev[2].record()
        out_host[i & 1].copy_(desc, non_blocking=True)             # D2H of the result
        ev[3].record()
        e2e_marks.append(ev)

    def loop(fn):
        def body(i):
            out = fn(i)
            if i == loop.n - 1:
                drain()                                             # every gather has landed inside the timed region
                loop.last = out
        return body

    for i in range(args.warmup):
        step_device(i)
    drain()
    if os.environ.get("ANYLOC_BENCH_PROFILE_STEP"):      # `ncu --profile-from-start off ...`: exactly one step's launches
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStart()
        step_device(0)
        drain()
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStop()
    sampler = ClockSampler(R.local)
    if rank == 0:
        sampler.start()
    launches0 = _lib.launch_count()
    loop.n = args.steps
    ms_total = R.timed(loop(step_device), args.steps)               # un-instrumented: this is `value`
    launches = _lib.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"descriptors": loop.last})

    # end-to-end through the public API with host buffers (pinned), copies inside the timed region
    for i in range(max(1, args.warmup // 2)):
        step_e2e(i)
    drain()
    e2e_marks.clear()
    ms_e2e = R.timed(loop(step_e2e), args.steps)
    e2e_phase = [sum(m[j].elapsed_time(m[j + 1]) for m in e2e_marks) / len(e2e_marks) for j in range(3)]

    # separate instrumented pass (a cudaEvent pair per launch group): time shares and the kernels' live durations
    n_prof = min(args.steps, 3)
    _lib.profile_enable(True)
    loop.n = n_prof
    ms_prof = R.timed(loop(step_device), n_prof)
    prof = _lib.profile_read()
    _lib.profile_enable(False)
    ext.raise_if_overflowed()
    # the VLAD call alone, back to back, on the step's own features and vocabulary (what the in-pipeline figure of the
    # instrumented pass differs from: there the call follows the ViT with the features freshly written and cold centres)
    feats_now = ext(img_dev)
    for _ in range(3):
        vlad.generate_multi(feats_now)
    vlad_alone_ms = R.timed(lambda i: vlad.generate_multi(feats_now), 20) / 20
    del feats_now

    # ---- checks after the timed loops (untimed)
    desc = step_device(0)
    drain()
    torch.cuda.synchronize()
    chk = {"allgather_bitwise": R.all_true(torch.equal(db_ring[0, rank * B:(rank + 1) * B], desc))}
    for i in range(1, SLOTS):
        step_device(i)
    drain()
    db_all = db_ring.reshape(-1, Dv)
    # queries: noisy copies of this rank's rows of chunk 0 -> the global index of the source row is known
    nq_loc = 4
    qn = torch.randn(nq_loc, Dv, device=dev, generator=g)
    qu_loc = desc[:nq_loc] + 0.1 * qn / qn.norm(dim=1, keepdim=True)
    truth = torch.arange(nq_loc, device=dev) + rank * B
    res = {}
    for strategy in ("gather_db", "gather_queries"):
        s, e = adist.shard_range(db_all.shape[0])
        d_, i_ = adist.sharded_top_k(db_all[s:e].contiguous(), qu_loc, 3, strategy=strategy)
        res[strategy] = (d_, i_)
    i_db = res["gather_db"][1]
    chk["topk_strategies_equal"] = R.all_true(torch.equal(i_db, res["gather_queries"][1]))
    # identical images every step -> chunks 1..3 hold duplicates of chunk 0's rows; the lowest index must win
    chk["top1_is_source_row"] = R.all_true(torch.equal(i_db[rank * nq_loc:(rank + 1) * nq_loc, 0], truth))
    coll_us, coll_gbs = collective_alone(R, (B, Dv))

    if rank != 0:
        R.finish()
        return
    peaks = measured_peaks()
    ms_step = ms_total / args.steps
    value = world * B * args.steps / (ms_total / 1e3)
    e2e_value = world * B * args.steps / (ms_e2e / 1e3)
    g_ms, g_n, g_fl = prof["gemm_tc"]
    flops_img = vit_flops_per_image(wl["model"], wl["layer"], H, W)
    f16 = ext.precision == "f16x3"
    roof = None
    if g_n:
        ach = g_fl / (g_ms / 1e3) / 1e12
        passes = 3.0 if f16 else 6.0       # bf16-rate-equivalent tensor passes per algorithmic product
        two_cta = os.environ.get("ANYLOC_GEMM_2CTA", "1") != "0"
        kname = ("gemm_tc3_2cta_kernel<%s> (tcgen05 cta_group::2 M256xN256, kind::%s" if two_cta else
                 "gemm_tc3_kernel<256,%s> (tcgen05 cta_group::1 M128xN256, kind::%s") % (
                     "true" if f16 else "false", "f16" if f16 else "tf32")
        # the four per-block GEMMs (qkv <1,1,1>, w12 <1,3,1>, proj / w3 <1,4,1>) of the committed capture of this shape
        traffic, tsrc = (ncu_traffic(["kernel<1, 1, 1>", "kernel<1, 3, 1>", "kernel<1, 4, 1>"], "vit")
                         if (args.workload == "c2" and f16 and two_cta) else (None, None))
        roof = {"kernel": kname + ", 3-term split, fp32 accumulate, RN chunk accumulation)",
                "bound": "tensor", "achieved": ach, "peak": peaks["tflops_sustained"], "unit": "TFLOP/s",
                "frac": ach / peaks["tflops_sustained"], "traffic": traffic, "traffic_source": tsrc,
                "algorithmic_flops_per_launch": g_fl / g_n,
                "peak_source": f"{peaks['source']} cuBLAS bf16 sustained (MEASURED_PEAKS.json)",
                "contract_ceiling": 1.0 / passes,
                "note": "achieved = algorithmic 2MNK FLOPs / live device time of the launches (CUDA events, separate "
                        "instrumented pass); fp32-equivalent results need 3 MMAs per product at %s the bf16 rate = %d "
                        "bf16-equivalent passes, so frac <= contract_ceiling on this precision contract; "
                        "frac / contract_ceiling estimates the tensor-pipe utilisation"
                        % ("1x" if f16 else "0.5x", int(passes)),
                "tensor_pipe_frac_est": passes * ach / peaks["tflops_sustained"],
                "launches": g_n, "avg_launch_ms": g_ms / g_n, "share_of_step": g_ms / ms_prof}
    v_ms, v_n, v_bytes = prof["vlad"]
    vroof = None
    if v_n:
        gbs = v_bytes / (v_ms / 1e3) / 1e9
        vtraffic, vsrc = ncu_traffic(["vlad_assign_tc_kernel", "vlad_accumulate3_kernel"], "vlad_" + args.workload, per_call=True)
        vroof = {"kernel": u.VLAD_KERNEL_DESCRIPTION,
                 "bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                 "traffic": vtraffic, "traffic_source": vsrc,
                 "algorithmic_bytes_per_launch_group": v_bytes / v_n,
                 "avg_launch_ms": v_ms / v_n, "share_of_step": v_ms / ms_prof,
                 "standalone_ms_same_inputs": vlad_alone_ms,
                 "standalone_frac": v_bytes / v_n / (vlad_alone_ms / 1e3) / 1e9 / peaks["hbm_gbs"]}
    shares = {c: round(prof[c][0] / ms_prof, 4) for c in prof if prof[c][1]}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None,
            "dtype": "f32-equivalent (tcgen05 %s 3-term split, fp32 accumulate)" % ("fp16" if f16 else "tf32"),
            "data": "synthetic",
            "config": {"workload": wl["name"], "per_gpu_batch": B, "global_batch": B * world,
                       "weights": "random-init (upstream recipe), no checkpoint offline",
                       "parallelism": (f"dp{world}: images sharded; one ncclAllGather of the step's [{B},{Dv}] fp32 "
                                       f"descriptors per rank into the replicated retrieval database, asynchronous, "
                                       f"overlapping the next step's ViT" if world > 1 else
                                       "dp1: the descriptor all-gather degenerates to the copy into the database buffer"),
                       "precision": ext.precision,
                       "cache": "inputs larger than L2: weights (hi+lo) streamed every step"},
            "vit_tflops_algorithmic": flops_img * value / 1e12,
            "roofline": roof, "roofline_vlad": vroof, "time_shares": shares,
            "collective": {"name": "ncclAllGather (torch.distributed all_gather_into_tensor)" if world > 1 else "none (N=1: device copy)",
                           "bytes_per_rank_per_step": B * Dv * 4, "recv_bytes_per_rank_per_step": (world - 1) * B * Dv * 4,
                           "alone_us": coll_us, "alone_busbw_GBs": coll_gbs, "nvlink_peak_GBs_per_dir": NVLINK_GBS_PER_DIR,
                           "in_timed_region": True, "overlapped": world > 1, "checks": chk},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": world * img_host.numel() * 4,
                    "d2h_bytes_per_step": world * B * Dv * 4, "ms_per_step": ms_e2e / args.steps,
                    "rank0_phase_ms": {"h2d": e2e_phase[0], "compute_and_gather_launch": e2e_phase[1], "d2h": e2e_phase[2]}},
            "gpu_launches": launches, "clocks": clocks}
    if sd_host is not None:
        line["parity"] = pipeline_parity(wl, sd_host, img_host, vlad, desc, ext, u)
        del sd_host
    if world == 1 and not args.no_cpu_baseline:
        n_ref = max(args.ref_images, 4)        # ~14 s of timed CPU work at c2 (0.85-0.9 img/s on the box's 16 usable cores)
        ips, ms, cores = cpu_reference(wl, n_ref, 3, 1)
        line["cpu_baseline"] = {"value": ips, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"{n_ref} images x 3 steps of the same workload, batch 1 per image, "
                                          "all blocks + hook, CPU VLAD with [N,K,D] residuals"}
        if not args.no_gpu_reference:
            del ext
            _lib.workspaces.clear()
            torch.cuda.empty_cache()
            n_g = 16
            ips_g, vit_ms = gpu_reference(wl, n_g)
            line["reference_gpu"] = {"value": ips_g, "unit": UNIT, "vit_ms_per_image": vit_ms,
                                     "what": "the reference GPU PyTorch path on this GPU: restated hub model .cuda() fp32 "
                                             "(TF32 off), batch 1, all blocks + hook, .cpu() per image, CPU VLAD.generate "
                                             "with [N,K,D] residuals (scripts/dino_v2_vlad.py:164-188,233-237); torch/cuBLAS "
                                             "kernels only", "sample": f"{n_g} images",
                                     "e2e_over_reference_gpu": e2e_value / ips_g}
    print(json.dumps(line), flush=True)
    R.finish()


def pipeline_parity(wl, sd_host, img_host, vlad, desc, ext, u, n=2):
    """bench.py checks what it timed: the first `n` images of the timed batch through the CPU oracle (restated hub model
    with the SAME weights, reference VLAD arithmetic with the SAME vocabulary) against the features / descriptors the
    timed configuration produced.  Relative inf-norm errors (north_star tolerance 1e-4)."""
    import torch
    from oracle import anyloc_oracle as ao
    from oracle import dinov2_restated as dr
    torch.set_num_threads(usable_cores())
    with torch.device("meta"):
        model = dr.DinoVisionTransformer(wl["model"], depth_override=wl["layer"] + 1)
    model.load_state_dict(sd_host, strict=False, assign=True)
    model.eval()
    ref_f = ao.extract_features(model, img_host[:n].clone(), wl["layer"], wl["facet"])
    got_f = ext(img_host[:n].to(ext.device)).cpu()
    centers = vlad.c_centers.cpu()
    err_f = float((got_f - ref_f).abs().max() / ref_f.abs().max())
    got_v = desc[:n].cpu()
    # (1) the VLAD kernels alone: reference arithmetic on the SAME (GPU) features
    same_v = torch.stack([ao.vlad_generate(f, centers) for f in got_f])
    err_v_same = float((got_v - same_v).abs().max() / same_v.abs().max())
    # (2) end to end: reference arithmetic on the reference features.  With the vocabulary fitted on this very batch the
    # residual sums cancel heavily (sum over a cluster's members of x^ - c_k is ~0 by construction), so the feature
    # error is amplified by the conditioning of the descriptor itself; reported, not gated.
    ref_v = torch.stack([ao.vlad_generate(f, centers) for f in ref_f])
    err_v = float((got_v - ref_v).abs().max() / ref_v.abs().max())
    lab_ref = torch.stack([ao.vlad_labels(f, centers) for f in ref_f])
    lab_got = torch.stack([ao.vlad_labels(f, centers) for f in got_f])
    return {"images": n, "features_rel_err": err_f, "descriptors_rel_err_same_features": err_v_same,
            "descriptors_rel_err_end_to_end": err_v, "labels_differ": int((lab_ref != lab_got).sum()),
            "labels_total": int(lab_ref.numel()), "tolerance": 1e-4, "ok": bool(err_f < 1e-4 and err_v_same < 1e-4),
            "note": "end-to-end descriptor error = feature error x conditioning of the descriptor (vocabulary fitted on the "
                    "batch itself: residual sums nearly cancel); gated: features and the VLAD kernels on equal features"}


# ------------------------------------------------------------------ retrieval (c3 / c4)
def run_retrieval(args, wl):
    R = Ranks()
    torch, dist, dev, world, rank = R.torch, R.dist, R.dev, R.world, R.rank
    from anyloc_b200 import _lib, dist as adist, utilities as u
    n_loc, n_q, Dv, k = wl["n_db_per_rank"], wl["n_q"], wl["Dv"], wl["k"]
    if args.small:
        n_loc, n_q = n_loc // 10, n_q // 10
    n_db = n_loc * world
    g = torch.Generator(device=dev).manual_seed(7 + rank)
    db_local = torch.nn.functional.normalize(torch.randn(n_loc, Dv, device=dev, generator=g), dim=1)
    qs, qe = adist.shard_range(n_q)
    nq_loc = qe - qs
    src = torch.randperm(n_loc, device=dev, generator=g)[:nq_loc]
    qu_local = db_local[src] + 0.1 * torch.nn.functional.normalize(torch.randn(nq_loc, Dv, device=dev, generator=g), dim=1)
    truth_local = src + rank * n_loc
    top_k = [1, k]

    # persistent buffers of the gather_db step (a service keeps them; allocating 2 x 20 GB per step would time cudaMalloc)
    db_all_buf = torch.empty(n_db, Dv, device=dev) if world > 1 else db_local
    index_all = u.FlatIndex(Dv, "cosine", True, capacity=n_db, device=dev)
    d_all, i_all = torch.empty(n_q, k, device=dev), torch.empty(n_q, k, device=dev, dtype=torch.int64)

    def step_gather_db(i):
        """BASELINE config 4's pattern: all-gather the database descriptors, index them, every rank answers its own
        query shard, the [n_q, k] results are gathered.  (Equal shards: n_db_per_rank rows and n_q / world queries.)"""
        if world > 1 and args.gather_chunks > 1:
            # THE collective ([n_loc, Dv] fp32 per rank), in pieces, each prepared into the index while the next travels
            adist.all_gather_into_index(index_all, db_local, staging=db_all_buf, chunks=args.gather_chunks)
        else:
            if world > 1:
                dist.all_gather_into_tensor(db_all_buf, db_local)
            index_all.reset()
            index_all.add(db_all_buf)
        d, ix = index_all.search(qu_local, k)
        if world == 1:
            return d, ix
        if n_q % world == 0:
            dist.all_gather_into_tensor(d_all, d.contiguous())
            dist.all_gather_into_tensor(i_all, ix.contiguous())
            return d_all, i_all
        return adist.all_gather_rows(d), adist.all_gather_rows(ix)

    index_local = u.FlatIndex(Dv, "cosine", True)
    index_local.add(db_local)

    def step_search_only(i):
        return index_local.search(qu_local, k)

    def step_gather_queries(i):
        """database stays sharded (index built once, resident): all-gather the queries, local top-k with global
        offsets, all-gather + merge the candidates"""
        return adist.sharded_top_k(db_local, qu_local, k, strategy="gather_queries",
                                   search=lambda db, qu, kk, method, norm: index_local.search(qu, kk))

    # c3 (one GPU): the database is indexed once (what `index.add(db)` does, utilities.py:449) and every step is one
    # 1k-query search on the resident index; c4 (N GPUs): a step is the whole retrieval exchange of BASELINE config 4 --
    # all-gather of the database descriptors, index build, search of the rank's query shard, gather of the results
    step = step_gather_db if (wl is WORKLOADS["c4"] or world > 1) else step_search_only
    step_name = "gather_db" if step is step_gather_db else "search_resident_index"
    for i in range(args.warmup):
        step(i)
    sampler = ClockSampler(R.local)
    if rank == 0:
        sampler.start()
    l0 = _lib.launch_count()
    last = {}

    def timed_step(i):
        last["out"] = step(i)
    ms_total = R.timed(timed_step, args.steps)
    launches = _lib.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:          # before any later call reuses the gather_db result buffers
        dump_outputs(args.dump_outputs, {"distances": last["out"][0], "indices": last["out"][1]})
    for i in range(2):
        step_gather_queries(i)
        step_gather_db(i)
    ms_gq = R.timed(step_gather_queries, args.steps)
    ms_search = R.timed(step_search_only, args.steps)
    ms_gdb = R.timed(step_gather_db, args.steps)

    def build_only(i):
        ix = u.FlatIndex(Dv, "cosine", True, capacity=n_loc, device=dev)
        ix.add(db_local)
    build_only(0)
    ms_build = R.timed(build_only, max(2, args.steps // 2)) / max(2, args.steps // 2)
    _lib.profile_enable(True)
    n_prof = min(args.steps, 3)
    R.timed(step, n_prof)
    prof = _lib.profile_read()
    _lib.profile_enable(False)
    coll_us, coll_gbs = collective_alone(R, (n_loc, Dv), iters=3)

    # correctness: the noisy copy's source row is the top-1; both strategies agree; fp64 scores on this rank's queries
    d_db, i_db = step_gather_db(0)
    d_gq, i_gq = step_gather_queries(0)
    truth = adist.all_gather_rows(truth_local)
    ok_top1 = R.all_true(torch.equal(i_db[:, 0], truth))
    ok_same = R.all_true(torch.equal(i_db, i_gq))
    db_all = adist.all_gather_descriptors(db_local)    # rank-major reference copy (the staging buffer is piece-major)
    n_chk = nq_loc                                   # every query of this rank, database converted chunk by chunk
    qd = qu_local.double()
    qd = qd / qd.norm(dim=1, keepdim=True)
    sc = torch.empty(n_chk, db_all.shape[0], device=dev, dtype=torch.float64)
    for c0 in range(0, db_all.shape[0], 8192):
        blk = db_all[c0:c0 + 8192].double()
        sc[:, c0:c0 + 8192] = qd @ (blk / blk.norm(dim=1, keepdim=True)).T
    rd, ri = torch.sort(sc, dim=1, descending=True, stable=True)
    ok_fp64 = R.all_true(torch.equal(ri[:, :k], i_db[qs:qs + n_chk]))
    dist_err = float((rd[:, :k] - d_db[qs:qs + n_chk].double()).abs().max())

    # e2e through the reference-facing call with HOST tensors (N=1 only: get_top_k_recall has no multi-GPU form)
    e2e = None
    if world == 1:
        db_h, qu_h = db_local.cpu().pin_memory(), qu_local.cpu().pin_memory()
        import numpy as np
        gt = np.empty(n_q, dtype=object)
        for j, t in enumerate(truth_local.tolist()):
            gt[j] = np.array([t])
        u.get_top_k_recall(top_k, db_h, qu_h, gt)
        n_e2e = max(1, min(args.steps, 3))
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            dd, ii, rec = u.get_top_k_recall(top_k, db_h, qu_h, gt)
        dt = (time.perf_counter() - t0) / n_e2e
        e2e = {"value": n_q / dt, "unit": "queries/s", "ms_per_step": dt * 1e3,
               "h2d_bytes_per_step": (n_db + n_q) * Dv * 4, "d2h_bytes_per_step": n_q * k * 12,
               "recall@1": rec[1], "call": "get_top_k_recall(top_k, db, qu, gt_pos) with host tensors (index.add + search)"}
    if rank != 0:
        R.finish()
        return
    peaks = measured_peaks()
    ms_step = ms_total / args.steps
    g_ms, g_n, g_fl = prof["gemm_tc"]
    roof = None
    if g_n:
        ach = g_fl / (g_ms / 1e3) / 1e12
        roof = {"kernel": u.TOPK_KERNEL_DESCRIPTION, "bound": "tensor", "achieved": ach, "peak": peaks["tflops_sustained"],
                "unit": "TFLOP/s", "frac": ach / peaks["tflops_sustained"], "traffic": ncu_traffic(["gemm_tc3_2cta_kernel<1, 0, 0>"], "topk")[0],
                "algorithmic_flops_per_launch": g_fl / g_n, "avg_launch_ms": g_ms / g_n, "launches": g_n,
                "contract_ceiling": 1.0 / 3.0}
    line = {"metric": "queries/sec cosine top-%d retrieval over a %d-image database of %d-D VLAD descriptors" % (k, n_db, Dv),
            "value": n_q * args.steps / (ms_total / 1e3), "unit": "queries/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32-equivalent (tcgen05 fp16-pair 3-term split on unit rows, fp32 accumulate)", "data": "synthetic",
            "config": {"workload": wl["name"], "n_db_total": n_db, "n_db_per_gpu": n_loc, "n_q": n_q, "Dv": Dv, "k": k,
                       "step": ("all-gather of the database descriptors + index build (normalise + fp16-pair split) + search "
                                "of this rank's query shard + gather of the [n_q,k] results" if step is step_gather_db else
                                "1k-query search on the resident (prepared) database index; index build reported separately"),
                       "parallelism": f"database and queries sharded over {world} GPU(s); strategy gather_db (BASELINE config 4)",
                       "cache": "database larger than L2"},
            "roofline": roof,
            "alternatives": {"step": step_name, "gather_db_ms_per_step": ms_gdb / args.steps,
                             "gather_queries_ms_per_step": ms_gq / args.steps,
                             "search_only_local_shard_ms": ms_search / args.steps, "index_build_local_shard_ms": ms_build,
                             "note": "gather_queries keeps the database sharded with a resident index (all-gathers the queries "
                                     "and the [n_q,k] candidates instead): identical results"},
            "collective": {"name": "ncclAllGather of [n_db_per_gpu, Dv] fp32" if world > 1 else "none",
                           "bytes_per_rank_per_step": n_loc * Dv * 4, "alone_us": coll_us, "alone_busbw_GBs": coll_gbs,
                           "nvlink_peak_GBs_per_dir": NVLINK_GBS_PER_DIR},
            "parity": {"top1_is_source_row": ok_top1, "strategies_identical": ok_same,
                       "top%d_equals_fp64_all_%d_queries" % (k, n_q): ok_fp64, "max_abs_dist_err_vs_fp64": dist_err},
            "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
            "time_shares": {c: round(prof[c][0] / (ms_step * n_prof), 4) for c in prof if prof[c][1]}}
    print(json.dumps(line), flush=True)
    R.finish()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--engine", default="auto", choices=["auto", "tc3", "simt"])
    ap.add_argument("--ref-images", type=int, default=2, help="images per CPU-reference step (bounded sample)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true")
    ap.add_argument("--no-parity-check", action="store_true")
    ap.add_argument("--small", action="store_true", help="retrieval workloads at 1/10 size (smoke runs)")
    ap.add_argument("--gather-chunks", type=int, default=4, help="c4: pieces of the database all-gather (1 = one collective)")
    ap.add_argument("--vocab", default="fit", choices=["fit", "random"])
    ap.add_argument("--precision", default="f16x3", choices=["f16x3", "tf32x3", "auto"],
                    help="operand pair format of the tensor-core GEMMs (both fp32-equivalent; see DESIGN.md)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned on rank 0 as DIR/<name>.npy (seeded inputs: two "
                         "builds run with the same arguments can be compared output for output)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference_arm(args, wl)
    elif wl["kind"] == "pipeline":
        run_pipeline(args, wl)
    else:
        run_retrieval(args, wl)


if __name__ == "__main__":
    main()
