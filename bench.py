#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's configs, on N GPUs of one node.

    metric   : embed+top-k query images/sec  (whole job: embed gallery + queries with the descriptor network,
               L2-normalise, all-pairs dot-product similarity, per-query top-k)
    default  : configs[1] (C2) "10k query x 100k gallery, SSCD ResNet-50 embed+top-k on 1 B200"; at N > 1 every rank
               holds a 100k-image gallery shard and a 10k block of queries (weak scaling), all queries are scored against
               every shard, per-shard top-k lists are all-gathered and merged (dcr_b200/dist.py).
    --config c3      configs[2]: DINO ViT-S/16 instead of the SSCD ResNet-50, same sizes
    --config c4      configs[3]: FID, 50k generated vs 50k real 299x299 images: Inception-v3 forward + streaming fp64
                     mean/covariance + Frechet distance (metric: FID images/sec)
    --config c5      configs[4]: 50k query x 1M gallery TOTAL, sharded 1/N per rank (strong scaling; needs N >= 2 for HBM)
    --scaling strong the C2/C3 totals stay fixed and every rank takes 1/N of the gallery and of the queries
    one step : embed G_local + Q_local synthetic 256x256 uint8 images, normalise, sharded top-k (k = 10).

`value` times the step with the images already resident in HBM; `e2e` times the same step through the public API
from pinned HOST memory (H2D of every image batch and D2H of the result inside the timed region).
`roofline` is the fused similarity kernel (tensor bound), timed by CUDA events inside dcr_sim_topk.
`precision_modes` repeats the device-resident measurement in the `parity` (split-bf16, fp32-level) network mode -- the
mode whose scores stay within the 1e-4 tolerance of BASELINE.json; the headline runs the networks in bf16 (`fast`).
`cpu_baseline` / `--impl reference` time the CPU restatement of the reference path (oracle/) on a bounded sample.
`--dump-outputs DIR` writes what the last timed step returned -- top-k values and indices plus the query and gallery
descriptors, or the FID value for c4 -- as DIR/<name>.npy; the inputs are seeded, so the dumps of two builds of the
project compare output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K_TOP = 10
IMG = 256
FID_IMG = 299
METRIC = "embed+top-k query images/sec"
DUMP_LIMIT = 60_000_000      # bytes of array data in one --dump-outputs directory (npy headers add 128 bytes a file)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"burst": float(d["bf16_tflops"]), "sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                "hbm": float(d["hbm_gbs"]), "src": "measured"}
    return {"burst": 1590.0, "sustained": 1400.0, "hbm": 6650.0, "src": "fallback"}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 7:
                    self.samples.append(parts)
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(s[0]) for s in self.samples)
        reasons = []
        for i, name in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
            if any(s[3 + i].lower().startswith("active") for s in self.samples):
                reasons.append(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons,
                "samples": len(sm)}


def gen_images_cuda(n: int, seed: int, device, copies_of=None, copy_frac: float = 0.1, chunk: int = 2048,
                    size: int = IMG):
    """uint8 [n,size,size,3] on `device`: low-frequency random fields; a fraction are brightness/shift-augmented copies
    of `copies_of` rows (planted matches, so similarities span [0,1] as in DCR's use)."""
    out = torch.empty((n, size, size, 3), dtype=torch.uint8, device=device)
    g = torch.Generator(device=device).manual_seed(seed)
    for s in range(0, n, chunk):
        b = min(chunk, n - s)
        img = 0.4 * torch.rand((b, 3, 1, 1), device=device, generator=g)            # per-image colour offset
        for res, amp in ((4, 0.35), (16, 0.3), (64, 0.25)):                          # three noise scales, random mixing
            field = torch.rand((b, 3, res, res), device=device, generator=g)
            gain = amp * torch.rand((b, 1, 1, 1), device=device, generator=g)
            img = img + gain * torch.nn.functional.interpolate(field, size=(size, size), mode="bilinear",
                                                              align_corners=False)
        img = img + 0.04 * torch.randn((b, 3, size, size), device=device, generator=g)
        out[s:s + b] = (img.clamp_(0, 1) * 255.0).round_().to(torch.uint8).permute(0, 2, 3, 1)
    if copies_of is not None and n > 0 and copy_frac > 0:
        n_c = int(round(copy_frac * n))
        dst = torch.randperm(n, device=device, generator=g)[:n_c]
        src = torch.randint(0, copies_of.shape[0], (n_c,), device=device, generator=g)
        gain = 0.8 + 0.4 * torch.rand((n_c, 1, 1, 1), device=device, generator=g)
        sh = int(torch.randint(-8, 9, (1,), device=device, generator=g).item())
        for s in range(0, n_c, chunk):         # chunked: the float copy of 10^5 images would not fit beside them
            base = torch.roll(copies_of[src[s:s + chunk]].float(), shifts=(sh, -sh), dims=(1, 2)) * gain[s:s + chunk]
            out[dst[s:s + chunk]] = base.clamp_(0, 255).round_().to(torch.uint8)
    return out


def synthetic_sscd_weights(dev, whiten_floor: float = 1e-2, head: str = "pca"):
    """Seeded random-init SSCD ResNet-50 weights (no network access, no checkpoints), made data-consistent the way
    a freshly initialised PyTorch model becomes after its first training-mode batches: the BatchNorm running
    statistics are set from 512 synthetic images (torch ops, set-up only -- nothing of this runs in a timed region),
    and the head Linear is PCA-whitened on 2048 synthetic images.  Without this a random trunk maps every image
    to nearly the same direction; trained SSCD descriptors are spread over the sphere by construction."""
    import torchvision
    from dcr_b200 import nets
    from oracle import models as om
    sd = om.make_sscd_state_dict(0)
    cal_imgs = gen_images_cuda(512, seed=999, device=dev)
    m = torchvision.models.resnet50(weights=None)
    tv = {k[len("backbone."):]: v for k, v in sd.items() if k.startswith("backbone.")}
    tv["fc.weight"], tv["fc.bias"] = m.fc.weight.detach(), m.fc.bias.detach()
    m.load_state_dict(tv)
    m = m.to(dev).train()
    for mod in m.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.momentum = None            # cumulative average over the calibration batches
            mod.reset_running_stats()
    x = om.preprocess(cal_imgs.cpu()).to(dev)
    with torch.no_grad():
        for s in range(0, x.shape[0], 128):
            m(x[s:s + 128])
    for k, v in m.state_dict().items():
        if "running_mean" in k or "running_var" in k:
            sd["backbone." + k] = v.detach().float().cpu()
    del m, x
    # PCA-whiten the head on 2048 synthetic images: SSCD is trained (entropy regulariser) to spread its descriptors
    # uniformly over the sphere; a random head on a random trunk concentrates them in a few directions instead.
    cal = nets.build_sscd_resnet50(sd, max_batch=128, precision="fast", l2_normalize=False)
    emb = torch.cat([cal(cal_imgs), cal(gen_images_cuda(1536, seed=998, device=dev))]).double().cpu()
    del cal
    mean = emb.mean(dim=0)
    if head == "diag":
        # milder alternative: standardise every head output (zero mean, unit variance over the calibration images) -- a
        # diagonal rescaling, condition number = ratio of the output standard deviations, no rotation into noise directions
        std = emb.std(dim=0).clamp_min(1e-12)
        w, bias = sd["embeddings.1.weight"].double(), sd["embeddings.1.bias"].double()
        sd["embeddings.1.weight"] = (w / std[:, None]).float()
        sd["embeddings.1.bias"] = ((bias - mean) / std).float()
        torch.cuda.empty_cache()
        return sd
    cov = torch.cov((emb - mean).T)
    lam, u = torch.linalg.eigh(cov)
    # floor on the whitened spectrum: directions with less than `whiten_floor` of the top variance are numerical noise of
    # the random trunk; amplifying them to unit variance (floor 1e-6) makes the descriptor an amplifier of rounding error
    # -- no trained model behaves like that -- so they are capped at a 10x gain
    lam = lam.clamp_min(lam.max() * whiten_floor)
    wh = (u / lam.sqrt()).T                                    # Lambda^-1/2 U^T
    w, bias = sd["embeddings.1.weight"].double(), sd["embeddings.1.bias"].double()
    sd["embeddings.1.weight"] = (wh @ w).float()
    sd["embeddings.1.bias"] = (wh @ (bias - mean)).float()
    torch.cuda.empty_cache()
    return sd


# --------------------------------------------------------------------------------------------------------------------
# the reference's CPU path (oracle restatement), bounded samples
_CPU_THREADS = None


def _cpu_threads() -> int:
    """SURVEY.md 8d: the CPU baseline uses every host core.  torchrun exports OMP_NUM_THREADS=1, so torch's default
    would be one thread under the multi-GPU launch; the count is set explicitly.  On a hyper-threaded host one thread per
    LOGICAL cpu can be several times slower than one per physical core for MKL/oneDNN kernels (measured on the B200 box:
    2.6 img/s with 128 threads against 18.8 with 64), so both are tried on a small ResNet-50 forward and the FASTER one is
    used and reported -- the baseline is the reference path at its best on this host."""
    global _CPU_THREADS
    if _CPU_THREADS is not None:
        torch.set_num_threads(_CPU_THREADS)
        return _CPU_THREADS
    from oracle import models as om
    n = os.cpu_count() or 1
    cands = sorted({n, max(1, n // 2)}, reverse=True)
    sd = om.make_sscd_state_dict(0)
    x = torch.randn(16, 3, 224, 224, generator=torch.Generator().manual_seed(0))
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        om.sscd_forward(sd, x[:2])
        t0 = time.perf_counter()
        om.sscd_forward(sd, x)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    _CPU_THREADS = best
    torch.set_num_threads(best)
    return torch.get_num_threads()


def cpu_reference_sample(net_kind: str, embed_imgs: int, sim_q: int, g_total: int, q_total: int, d_desc: int,
                         seed: int = 0):
    """Times the oracle (CPU restatement of the reference path) on a bounded sample and extrapolates to the workload.
    Returns (value queries/s, details)."""
    from oracle import models as om
    from oracle import similarity as osim  # noqa: F401  (documented dependency; torch.mm/topk is the literal path)
    from dcr_b200 import synthetic
    cores = _cpu_threads()
    imgs = synthetic.images(embed_imgs, seed=seed)
    x = om.preprocess(imgs)
    if net_kind == "dino":
        sd = om.make_vit_state_dict(0)
        fwd = lambda xb: om.vit_forward(sd, xb)      # noqa: E731  dino_vits.py:248-256
        name = "oracle DINO ViT-S/16 fp32 forward"
    else:
        sd = om.make_sscd_state_dict(0)
        fwd = lambda xb: om.sscd_forward(sd, xb)     # noqa: E731
        name = "oracle SSCD ResNet-50 fp32 forward"
    fwd(x[:2])                                       # warm the thread pool / allocator
    t0 = time.perf_counter()
    for s in range(0, embed_imgs, 64):               # loader batch 64, diff_retrieval.py:352
        fwd(x[s:s + 64])
    t_img = (time.perf_counter() - t0) / embed_imgs
    q, g = synthetic.descriptors(sim_q, g_total, d_desc, seed=seed)
    t0 = time.perf_counter()
    sim = torch.mm(g, q.T)                           # diff_retrieval.py:402 (fp32, CPU)
    sim.T.topk(K_TOP, dim=1, largest=True)           # diff_retrieval.py:417/621
    t_sim = (time.perf_counter() - t0) * (q_total / sim_q)
    total = t_img * (g_total + q_total) + t_sim
    details = {"cores": cores, "embed_img_per_s": 1.0 / t_img, "sim_topk_s_full": t_sim,
               "sample": f"{name} on {embed_imgs} images (batch 64) + torch.mm/topk({K_TOP}) on {sim_q} x {g_total} "
                         f"descriptors, extrapolated linearly to {q_total} queries + {g_total} gallery, {cores} threads"}
    return q_total / total, details


def cpu_reference_fid_sample(n_imgs: int, n_total: int, seed: int = 0):
    """FID on the CPU path: Inception forward on a sample (scaled), np.cov + sqrtm at full d = 2048 size."""
    from oracle import fid as ofid
    from oracle import models as om
    cores = _cpu_threads()
    sd = om.make_inception_state_dict(0)
    g = torch.Generator().manual_seed(seed)
    imgs = torch.randint(0, 256, (n_imgs, FID_IMG, FID_IMG, 3), dtype=torch.uint8, generator=g)
    x = om.fid_preprocess(imgs)
    om.fid_inception_forward(sd, x[:2])
    t0 = time.perf_counter()
    acts = []
    for s in range(0, n_imgs, 50):                   # batch_size 50, diff_retrieval.py:597-600
        acts.append(om.fid_inception_forward(sd, x[s:s + 50]))
    t_img = (time.perf_counter() - t0) / n_imgs
    rng = np.random.default_rng(seed)
    a1 = rng.standard_normal((4096, 2048))
    a2 = rng.standard_normal((4096, 2048)) + 0.1
    t0 = time.perf_counter()
    m1, s1 = ofid.activation_statistics(a1)          # metrics/fid.py:219-220 (np.mean / np.cov)
    m2, s2 = ofid.activation_statistics(a2)
    t_cov = (time.perf_counter() - t0) * (n_total / 8192.0)
    t0 = time.perf_counter()
    ofid.frechet_distance(m1, s1, m2, s2)            # metrics/fid.py:142-196
    t_fd = time.perf_counter() - t0
    total = t_img * n_total + t_cov + t_fd
    details = {"cores": cores, "inception_img_per_s": 1.0 / t_img, "cov_s_full": t_cov, "frechet_s": t_fd,
               "sample": f"oracle Inception-v3 fp32 forward on {n_imgs} images (batch 50) scaled to {n_total}; np.cov on "
                         f"2 x 4096 x 2048 scaled to {n_total} rows; scipy sqrtm Frechet at d=2048 (full size), {cores} threads"}
    return n_total / total, details


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=["c2", "c3", "c4", "c5"],
                    help="BASELINE.json configs[1..4] (c2 = the config the metric is quoted on)")
    ap.add_argument("--net", default=None, choices=["sscd", "dino"], help="descriptor network (default: by --config)")
    ap.add_argument("--scaling", default=None, choices=["weak", "strong"],
                    help="weak: --queries/--gallery per rank (default for c2/c3); strong: totals fixed, 1/N per rank (c5)")
    ap.add_argument("--queries", type=int, default=None, help="queries per rank (weak) / in total (strong)")
    ap.add_argument("--gallery", type=int, default=None, help="gallery images per rank (weak) / in total (strong)")
    ap.add_argument("--precision", default="fast", choices=["fast", "parity"],
                    help="network arithmetic of the HEADLINE run: fast = bf16 tensor cores (the product mode), "
                         "parity = 6-term split-bf16 on the same tensor cores (fp32-level descriptors)")
    ap.add_argument("--parity-steps", type=int, default=1,
                    help="timed steps of the secondary fp32-level measurements (0 = skip); 1 warm-up step before them")
    ap.add_argument("--other-modes", default="bf16x3,parity",
                    help="comma-separated network modes measured after the headline one (same full workload)")
    ap.add_argument("--batch", type=int, default=384,
                    help="images per network launch (measured on B200: 73.5k img/s at 256, 79.9k at 384 -- wave quantisation of the "
                         "persistent kernels over 148 SMs)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-embed-sample", type=int, default=128)
    ap.add_argument("--cpu-sim-sample", type=int, default=1000)
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200 (the reference arm times samples, not the workload)")
    if args.net is None:
        args.net = "dino" if args.config == "c3" else "sscd"
    if args.scaling is None:
        args.scaling = "strong" if args.config == "c5" else "weak"
    if args.config == "c5":
        args.queries = 50000 if args.queries is None else args.queries
        args.gallery = 1000000 if args.gallery is None else args.gallery
    elif args.config == "c4":
        args.queries = 50000 if args.queries is None else args.queries      # generated images
        args.gallery = 50000 if args.gallery is None else args.gallery      # real images
    else:
        args.queries = 10000 if args.queries is None else args.queries
        args.gallery = 100000 if args.gallery is None else args.gallery
    return args


def shard_sizes(args, rank: int, world: int):
    """(q_total, g_total, q_local, g_local, g_base)"""
    from dcr_b200 import dist as ddist
    if args.scaling == "strong":
        q_total, g_total = args.queries, args.gallery
        qlo, qhi = ddist.shard_bounds(q_total, rank, world)
        glo, ghi = ddist.shard_bounds(g_total, rank, world)
        return q_total, g_total, qhi - qlo, ghi - glo, glo
    return args.queries * world, args.gallery * world, args.queries, args.gallery, rank * args.gallery


def make_config(args, world, q_total, g_total, d_desc, precision):
    net_name = "SSCD ResNet-50" if args.net == "sscd" else "DINO ViT-S/16"
    per = (f"{args.queries} q + {args.gallery} g per GPU" if args.scaling == "weak"
           else f"1/{world} of the gallery and of the queries per GPU")
    imgs_per_gpu = (q_total + g_total) / world
    return {"workload": f"{net_name} embed + dot-product top-{K_TOP}: {q_total} query x {g_total} gallery "
                        f"synthetic 256x256 images ({per})",
            "baseline_config": args.config, "network": net_name, "precision": precision,
            "precision_note": ("networks in bf16 (one plane) on tcgen05, fp32 accumulate; similarity scores are exact "
                               "fp64-accumulated dot products of the fp32 descriptors the network produced.  bf16 descriptors "
                               "deviate from the fp32 reference path by more than the 1e-4 score tolerance (see "
                               "precision_modes.measured_deviation_from_fp32); the fp32-level modes are reported beside it"
                               if precision == "fast" else
                               "networks in split-bf16 (two / three planes) on tcgen05: fp32-level descriptors"),
            "queries": q_total, "gallery": g_total, "descriptor_dim": d_desc, "k": K_TOP,
            "images_embedded_per_step": q_total + g_total, "parallelism": f"gallery-shard x{world}",
            "l2": f"inputs ({imgs_per_gpu * IMG * IMG * 3 / 1e9:.1f} GB of images per GPU) are larger than "
                  "the 126 MB L2; no explicit flush"}


def run_reference(args, rank, world):
    """The reference's own CPU path, restated (the reference scripts cannot be imported/installed: torch._six, clip,
    natsort, NCCL-only init -- SURVEY.md 8c); rank 0 only, bounded sample per step, all host threads."""
    if rank != 0:
        return
    q_total, g_total, _, _, _ = shard_sizes(args, 0, world)
    d_desc = 512 if args.net == "sscd" else 384
    vals, det = [], None
    for i in range(args.warmup + args.steps):
        if args.config == "c4":
            v, det = cpu_reference_fid_sample(max(16, args.cpu_embed_sample // 4), q_total + g_total, seed=i)
        else:
            v, det = cpu_reference_sample(args.net, max(32, args.cpu_embed_sample // 2), args.cpu_sim_sample, g_total,
                                          q_total, d_desc, seed=i)
        if i >= args.warmup:
            vals.append(v)
    v = float(np.mean(vals))
    if args.config == "c4":
        metric, unit, n_units = "FID images/sec", "images/s", q_total + g_total
        config = {"workload": f"FID: {q_total} generated vs {g_total} real synthetic 299x299 images, Inception-v3 pool3 + "
                              "fp64 mean/covariance + Frechet distance", "baseline_config": "c4", "precision": "fp32"}
    else:
        metric, unit, n_units = METRIC, "query images/s", q_total
        config = make_config(args, world, q_total, g_total, d_desc, "fp32 (CPU)")
    line = {"impl": "reference", "metric": metric, "value": v, "unit": unit,
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * n_units / v, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": v, "unit": unit, "cores": det["cores"], "kind": "port", "sample": det["sample"]},
            "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def build_net(args, dev, precision, weights_cache):
    from dcr_b200 import nets
    from oracle import models as om   # only for the seeded weight generators
    if args.net == "dino":
        if "dino" not in weights_cache:
            weights_cache["dino"] = om.make_vit_state_dict(0)
        return nets.build_dino_vit(weights_cache["dino"], max_batch=args.batch, precision=precision)
    if "sscd" not in weights_cache:
        weights_cache["sscd"] = synthetic_sscd_weights(dev)
    return nets.build_sscd_resnet50(weights_cache["sscd"], max_batch=args.batch, precision=precision)


def check_result(values, indices, qf_all_fn, gf, g_base, world, dev, n_check: int = 64):
    """Validates the step's own output: for a query subsample, every rank recomputes its local exact top-k with plain
    torch (fp64 matmul over its gallery descriptors), the lists are gathered and merged on the host by
    (score desc, index asc) and compared with the rows the sharded path returned."""
    import torch.distributed as dist
    q_all = qf_all_fn()
    nq = q_all.shape[0]
    sel = torch.linspace(0, nq - 1, steps=min(n_check, nq), device=dev).long()
    s = q_all[sel].double() @ gf.double().T                          # [n_check, G_local]
    k = min(K_TOP, s.shape[1])
    lv, li = torch.sort(s, dim=1, descending=True, stable=True)
    lv, li = lv[:, :k].contiguous(), li[:, :k] + g_base             # fp64 scores: the ranking key of the product path
    if world > 1:
        lvs = [torch.empty_like(lv) for _ in range(world)]
        lis = [torch.empty_like(li) for _ in range(world)]
        dist.all_gather(lvs, lv.contiguous())
        dist.all_gather(lis, li.contiguous())
        lv, li = torch.cat(lvs, dim=1), torch.cat(lis, dim=1)
    lv, li = lv.cpu().numpy(), li.cpu().numpy()
    got_v, got_i = values[sel].cpu().numpy(), indices[sel].cpu().numpy()
    same, max_err = True, 0.0
    for r in range(lv.shape[0]):
        order = np.lexsort((li[r], -lv[r]))[:K_TOP]
        same = same and bool(np.array_equal(li[r][order], got_i[r]))
        max_err = max(max_err, float(np.abs(lv[r][order].astype(np.float32) - got_v[r]).max()))
    return {"queries_checked": int(lv.shape[0]), "indices_equal": bool(same), "max_score_err": max_err,
            "against": "per-rank fp64 torch matmul + stable sort on a query subsample, merged on the host"}


def dump_outputs(out_dir: str, arrays: dict, limit: int = DUMP_LIMIT) -> dict:
    """Writes every tensor of `arrays` (rows first) as out_dir/<name>.npy: float64 stays float64, other floating types
    become float32, integers become float64 (exact below 2**53).  The arrays share `limit` bytes: the smallest ones are
    written whole, and an array larger than an equal share of what is left keeps evenly spaced rows (row r*n//m of n,
    r < m).  The same shapes give the same rows, so the dumps of two builds compare file by file.
    Returns {name: [rows written, rows in the output]}."""
    os.makedirs(out_dir, exist_ok=True)
    written = {}
    left = limit
    order = sorted(arrays, key=lambda name: arrays[name].numel())
    for i, name in enumerate(order):
        t = arrays[name].detach()
        t = t.to(torch.float64 if t.dtype == torch.float64 or not t.is_floating_point() else torch.float32)
        n = t.shape[0]
        row_bytes = max(1, t[:1].numel()) * t.element_size()
        m = min(n, (left // (len(order) - i)) // row_bytes)
        if m < n:
            t = t[(torch.arange(m, dtype=torch.int64) * n // m).to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())
        left -= m * row_bytes
        written[name] = [m, n]
    return written


def run_retrieval_bench(args, rank, local_rank, world):
    import torch.distributed as dist
    from dcr_b200 import dist as ddist
    from dcr_b200 import retrieval, similarity

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    q_total, g_total, q_local, g_local, g_base = shard_sizes(args, rank, world)
    need_gb = (q_local + g_local) * IMG * IMG * 3 / 1e9
    if need_gb > 150:
        raise SystemExit(f"this rank would hold {need_gb:.0f} GB of images: use more GPUs for --config {args.config}")
    q_sizes = [shard_sizes(args, r, world)[2] for r in range(world)]

    gal_u8 = gen_images_cuda(g_local, seed=100 + rank, device=dev)
    weights = {}
    net = build_net(args, dev, args.precision, weights)
    d_desc = net.out_dim
    qry_u8 = gen_images_cuda(q_local, seed=200 + rank, device=dev, copies_of=gal_u8)
    config = make_config(args, world, q_total, g_total, d_desc, args.precision)
    keep = {}

    def make_step(the_net):
        def step(gal, qry):
            gf = retrieval.extract_features(the_net, gal, args.batch)
            qf = retrieval.extract_features(the_net, qry, args.batch)
            similarity.l2_normalize_(gf)
            similarity.l2_normalize_(qf)
            keep["gf"], keep["qf"] = gf, qf
            return ddist.sharded_topk(qf, gf, K_TOP, g_base, ddist.cuda_local_topk, ddist.cuda_merge, query_sizes=q_sizes)
        return step

    step = make_step(net)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        kms = []
        for _ in range(steps):
            fn()
            kms.append(similarity.sim_topk_stats()["kernel_ms"])
        ev1.record()
        barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), kms

    for _ in range(args.warmup):
        step(gal_u8, qry_u8)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = similarity.kernel_launch_count()

    def timed_step():
        keep["out"] = step(gal_u8, qry_u8)

    ms_total, kernel_ms = timed(timed_step, args.steps)
    launches = similarity.kernel_launch_count() - l0
    ms_per_step = ms_total / args.steps
    value = q_total / (ms_per_step / 1e3)
    st = similarity.sim_topk_stats()
    if rank == 0:
        sampler.stop_flag.set()
        sampler.join(timeout=2)
    dumped = None
    if args.dump_outputs and rank == 0:
        # every rank holds the merged top-k of all queries; the descriptors are this rank's queries and gallery shard
        dumped = dump_outputs(args.dump_outputs, {"values": keep["out"][0], "indices": keep["out"][1],
                                                  "query_features": keep["qf"], "gallery_features": keep["gf"]})
    del keep["out"]

    # ---- the step validates its own output (all ranks take part: collectives inside) -------------------------------
    out_v, out_i = step(gal_u8, qry_u8)
    check = check_result(out_v, out_i, lambda: ddist.all_gather_rows(keep["qf"], q_sizes) if world > 1 else keep["qf"],
                         keep["gf"], g_base, world, dev)

    # ---- end to end through the public API from pinned host memory ------------------------------------------------
    e2e = None
    if not args.no_e2e:
        host_kind = "pinned"
        try:
            gal_h = torch.empty(gal_u8.shape, dtype=torch.uint8, pin_memory=True)
            qry_h = torch.empty(qry_u8.shape, dtype=torch.uint8, pin_memory=True)
        except RuntimeError:        # page-locking ~22 GB per rank can fail on a crowded host: pageable copies still work
            host_kind = "pageable"
            gal_h = torch.empty(gal_u8.shape, dtype=torch.uint8)
            qry_h = torch.empty(qry_u8.shape, dtype=torch.uint8)
        gal_h.copy_(gal_u8)
        qry_h.copy_(qry_u8)
        torch.cuda.synchronize()

        def e2e_step():
            v, i = step(gal_h, qry_h)
            return v.cpu(), i.cpu()           # D2H of the step's result

        e2e_step()
        ms_e2e, _ = timed(e2e_step, args.steps)
        e2e = {"value": q_total / (ms_e2e / args.steps / 1e3), "unit": "query images/s",
               "h2d_bytes_per_step": int((q_total + g_total) * IMG * IMG * 3),
               "d2h_bytes_per_step": int(q_total * K_TOP * 12) * world, "host_memory": host_kind}
        del gal_h, qry_h

    # ---- the other precision modes, device-resident inputs, the SAME full workload ----------------------------------
    notes = {"parity": "6-term split-bf16 networks (3 planes): fp32-level descriptors; algorithmic FLOPs counted once (the tensor cores do 6x)",
             "bf16x3": "3-term split-bf16 networks (2 planes: hi*hi + hi*lo + lo*hi): as close to the exactly rounded fp32 path as "
                       "`parity` in tests/test_round2_gpu.py at half the planes; algorithmic FLOPs counted once (the tensor cores do 3x)",
             "fast": "bf16 networks"}
    others = {}
    flops_net = net.flops_per_image
    if args.parity_steps > 0:
        del net
        step = None          # the closure held the fast-mode network (and its fork's activations) alive
        for other_name in [m for m in args.other_modes.split(",") if m and m != args.precision]:
            keep.clear()
            torch.cuda.empty_cache()
            net2 = build_net(args, dev, other_name, weights)
            step2 = make_step(net2)
            step2(gal_u8, qry_u8)
            ms2, _ = timed(lambda: step2(gal_u8, qry_u8), args.parity_steps)
            ms2 /= args.parity_steps
            v2, i2 = step2(gal_u8, qry_u8)
            check2 = check_result(v2, i2, lambda: ddist.all_gather_rows(keep["qf"], q_sizes) if world > 1 else keep["qf"],
                                  keep["gf"], g_base, world, dev)
            others[other_name] = {"precision": other_name, "value": q_total / (ms2 / 1e3), "unit": "query images/s",
                                  "ms_per_step": ms2, "steps": args.parity_steps, "warmup": 1,
                                  "images_embedded_per_s": (q_total + g_total) / (ms2 / 1e3),
                                  "embed_tflops": net2.flops_per_image * (q_total + g_total) / (ms2 / 1e3) / 1e12,
                                  "note": notes.get(other_name, ""), "check": check2}
            del net2, step2

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = load_peaks()
    k_ms = float(np.mean(kernel_ms))
    flops = 2.0 * q_total * g_local * d_desc          # one launch: all queries x this rank's gallery shard
    achieved = flops / (k_ms * 1e-3) / 1e12
    # DRAM traffic of the fused kernel comes from an `ncu --set full` capture (profiles/); it is only quoted when this
    # run's launch has the shape that capture was taken on
    traffic = None
    prof = os.path.join(ROOT, "profiles", "sim_topk_traffic.json")
    if os.path.exists(prof):
        with open(prof) as f:
            pj = json.load(f)
        if pj.get("shape", [10000, 100000, 512, 10]) == [q_total, g_local, d_desc, K_TOP]:
            traffic = pj.get("dram_bytes_per_launch")
    roofline = {"kernel": "sim_topk_kernel<2> (fused Q.G^T + per-query top-k, tcgen05 cta_group::2)",
                "bound": "tensor", "achieved": achieved, "peak": peaks["sustained"], "unit": "TFLOP/s",
                "frac": achieved / peaks["sustained"], "frac_of_burst_peak": achieved / peaks["burst"],
                "peak_source": f"{peaks['src']} bf16_tflops_sustained (kernel timed inside a long step)",
                "kernel_ms": k_ms, "flops_per_launch": flops, "traffic": traffic, "launch": st}
    embed_tflops = flops_net * (q_total + g_total) / (ms_per_step / 1e3) / 1e12
    line = {"metric": METRIC, "value": value, "unit": "query images/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "bf16" if args.precision == "fast" else "bf16x3 (fp32-level)",
            "data": "synthetic", "config": config,
            "images_embedded_per_s": (q_total + g_total) / (ms_per_step / 1e3), "embed_tflops": embed_tflops,
            "gpu_launches": int(launches), "clocks": sampler.summary(), "roofline": roofline, "check": check}
    # the step's time is dominated by the descriptor network (conv/linear GEMM family, many shapes): its aggregate
    # tensor throughput over the whole step, against the same measured peak, reported beside the graded kernel's roofline
    line["roofline_embed"] = {"kernel": f"descriptor network forward ({config['network']}, all layers, per GPU)",
                              "bound": "tensor", "achieved": embed_tflops / world, "peak": peaks["sustained"],
                              "unit": "TFLOP/s", "frac": embed_tflops / world / peaks["sustained"]}
    if e2e is not None:
        line["e2e"] = e2e
    if dumped is not None:
        line["dump_outputs"] = {"dir": args.dump_outputs, "rows_written_of": dumped}
    if others:
        line["precision_modes"] = {args.precision: {"value": value, "unit": "query images/s", "ms_per_step": ms_per_step,
                                                    "note": notes.get(args.precision, "")}}
        line["precision_modes"].update(others)
        line["precision_modes"]["measured_deviation_from_fp32"] = (
            "tests/test_round2_gpu.py::test_precision_mode_contracts_against_fp32_mode (B200, 2304 images): max |score error| "
            "fast 9.7e-5 / bf16x3 3.6e-7 / parity 5.6e-7 on contractive random-init weights; fast 2.1e-1 / bf16x3 9.2e-4 / parity "
            "9.1e-4 on THIS benchmark's calibrated (chaotic) synthetic weights; every replicated image is found in every mode")
    if world == 1:
        v, det = cpu_reference_sample(args.net, args.cpu_embed_sample, args.cpu_sim_sample, g_total, q_total, d_desc)
        line["cpu_baseline"] = {"value": v, "unit": "query images/s", "cores": det["cores"], "kind": "port",
                                "sample": det["sample"], "embed_img_per_s": det["embed_img_per_s"],
                                "sim_topk_s_full": det["sim_topk_s_full"]}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_fid_bench(args, rank, local_rank, world):
    """configs[3]: FID of `--queries` generated vs `--gallery` real images (Inception-v3 pool3 -> fp64 mean/cov ->
    Frechet).  Each rank processes 1/N of both image sets; the (sum, X^T X, n) accumulators would be all-reduced in a
    multi-rank job -- here every rank finishes its own FID on its share (replicas), rank 0 reports."""
    import torch.distributed as dist
    from dcr_b200 import fid as dfid
    from dcr_b200 import nets, similarity
    from oracle import models as om

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    n_gen, n_real = args.queries // world, args.gallery // world
    bs = 200
    net = nets.build_fid_inception(om.make_inception_state_dict(0), max_batch=bs, precision=args.precision)
    real = gen_images_cuda(n_real, seed=300 + rank, device=dev, size=FID_IMG)
    gen = gen_images_cuda(n_gen, seed=400 + rank, device=dev, size=FID_IMG)
    result = {}

    def step(r, g):
        result["fid"] = dfid.fid_from_images(net, r, g, batch_size=bs)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        for _ in range(steps):
            fn()
        ev1.record()
        barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    for _ in range(args.warmup):
        step(real, gen)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = similarity.kernel_launch_count()
    ms = timed(lambda: step(real, gen), args.steps) / args.steps
    launches = similarity.kernel_launch_count() - l0
    dumped = None
    if args.dump_outputs and rank == 0:
        dumped = dump_outputs(args.dump_outputs, {"fid": torch.tensor([result["fid"]], dtype=torch.float64)})
    n_total = (n_gen + n_real) * world
    e2e = None
    if not args.no_e2e:
        real_h = torch.empty(real.shape, dtype=torch.uint8, pin_memory=True).copy_(real)
        gen_h = torch.empty(gen.shape, dtype=torch.uint8, pin_memory=True).copy_(gen)
        torch.cuda.synchronize()
        step(real_h, gen_h)
        ms_e = timed(lambda: step(real_h, gen_h), args.steps) / args.steps
        e2e = {"value": n_total / (ms_e / 1e3), "unit": "images/s", "h2d_bytes_per_step": int(n_total * FID_IMG * FID_IMG * 3),
               "d2h_bytes_per_step": int(2 * (2048 * 2048 + 2048) * 8) * world, "host_memory": "pinned"}
    if rank == 0:
        sampler.stop_flag.set()
        sampler.join(timeout=2)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = load_peaks()
    tfl = net.flops_per_image * n_total / (ms / 1e3) / 1e12
    line = {"metric": "FID images/sec", "value": n_total / (ms / 1e3), "unit": "images/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "bf16" if args.precision == "fast" else "bf16x3 (fp32-level)", "data": "synthetic",
            "config": {"workload": f"FID: {n_gen * world} generated vs {n_real * world} real synthetic 299x299 images, "
                                   "Inception-v3 pool3 + streaming fp64 mean/covariance + Frechet distance",
                       "baseline_config": "c4", "precision": args.precision, "batch": bs,
                       "l2": "inputs (tens of GB of images) are larger than the 126 MB L2; no explicit flush"},
            "fid_value": result.get("fid"), "gpu_launches": int(launches), "clocks": sampler.summary(),
            "roofline": {"kernel": "FID Inception-v3 forward (all conv GEMMs, per GPU)", "bound": "tensor",
                         "achieved": tfl / world, "peak": peaks["sustained"], "unit": "TFLOP/s",
                         "frac": tfl / world / peaks["sustained"], "traffic": None}}
    if e2e is not None:
        line["e2e"] = e2e
    if dumped is not None:
        line["dump_outputs"] = {"dir": args.dump_outputs, "rows_written_of": dumped}
    if world == 1:
        v, det = cpu_reference_fid_sample(max(16, args.cpu_embed_sample // 4), n_total)
        line["cpu_baseline"] = {"value": v, "unit": "images/s", "cores": det["cores"], "kind": "port", "sample": det["sample"]}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback)")
    if args.config == "c4":
        run_fid_bench(args, rank, local_rank, world)
    else:
        run_retrieval_bench(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
