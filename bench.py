#!/usr/bin/env python
"""bench.py -- pseudo-label images/s of the IRN hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 2|3|4|5] [--batch B] [--impl reference] [--dump-outputs DIR]

--config selects the BASELINE.json configuration (1-based, as BASELINE.json lists them):
  2  batch=64 synthetic 512x512, multi-scale CAM forward (scales 0.5/1.0/1.5/2.0) + merge            (make_cam body)
  3  batch=64 synthetic 512x512, CAM -> IRNet edge -> 256-iter random walk -> sem-seg label          (DEFAULT; contains 2)
  4  VOC12 train_aug-sized list (10,582 ids at 8 GPUs; 10,582*N/8 at N) of 512x512 JPEG files through the reference's
     step entry points (step.make_cam / step.make_sem_seg_labels `_work`, files in -> .npy / .png files out)
  5  instance path: IRNet displacement -> centroids -> clusters -> per-instance random walk -> detections, batch=32
One "step" = one pass of the path over one batch per GPU (configs 2,3,5) or over the rank's share of the list (config 4).
N > 1 is launched by torchrun (one rank per GPU); images shard across ranks (rank r takes ids r, r+N, ...: the reference's
stride partition) with no data-path collective; NCCL only gathers the per-image label maps to the writer rank (rank 0) on
a side stream, overlapped with the next step.  Rank 0 prints ONE JSON line.  `--impl reference` times the CPU oracle port
of the reference's own algorithm (dense (hw)^2 transition matrix squared 8 times, really executed) on the host cores.
`--dump-outputs DIR` writes what the last timed step returned (rank 0's share) as DIR/<name>.npy; the inputs and weights
are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "pseudo-label images/sec (CAM+random-walk)"
UNIT = "images/s"
H = W = 512
SCALES = (1.0, 0.5, 1.5, 2.0)
GFLOP_CAM, GFLOP_IRN = 974.04, 149.61       # SURVEY.md section 8(d): 4-scale CAM, EdgeDisplacement, per image
N_TRAIN_AUG = 10582
CONV_MODES = {0: "SIMT fp32", 1: "tcgen05 3xTF32", 2: "tcgen05 f16x3 (fp16 hi/lo split operands, fp32 accumulate)"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", type=int, default=3, choices=[2, 3, 4, 5])
    ap.add_argument("--batch", type=int, default=0, help="images per GPU per step (default: 64; 32 for --config 5)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--parity-images", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--conv-mode", type=int, default=-1, help="0 SIMT fp32, 1 tcgen05 3xTF32, 2 tcgen05 f16x3; -1 = library default")
    ap.add_argument("--list-limit", type=int, default=0, help="--config 4: ids in the list (default 10,582 * N / 8)")
    ap.add_argument("--step-batch", type=int, default=64, help="--config 4: --step_batch of the step entry points")
    ap.add_argument("--num-workers", type=int, default=-1, help="--config 4: DataLoader workers per GPU")
    ap.add_argument("--dump-outputs", default="", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy (64 MB at most)")
    a = ap.parse_args()
    if a.batch <= 0:
        a.batch = 32 if a.config == 5 else 64
    return a


WORKLOADS = {
    2: "batch=%d synthetic 512x512 per GPU: multi-scale CAM forward (0.5/1.0/1.5/2.0, image+flip) + merge/normalise (BASELINE.json configs[1])",
    3: "batch=%d synthetic 512x512 per GPU: multi-scale CAM (0.5/1.0/1.5/2.0, image+flip) -> IRNet edge -> 256-iter random walk -> "
       "sem-seg label (BASELINE.json configs[2])",
    5: "instance-seg path, batch=%d synthetic 512x512 per GPU: IRNet edge+displacement -> centroid refinement (300 it) -> clusters -> "
       "per-instance 256-iter random walk -> detections (BASELINE.json configs[4]); CAM seeds precomputed, as step/make_ins_seg_labels.py reads them",
}


def config(a, n_gpus):
    batch = a.batch
    cfg = {"workload": WORKLOADS.get(a.config, "")  % batch if a.config in WORKLOADS else "", "baseline_config": a.config,
           "global_batch": batch * n_gpus, "image": [H, W], "scales": list(SCALES), "rw_iters": 256, "beta": 10,
           "parallelism": "dp%d (images sharded by the reference's stride partition; NCCL gather of per-image label maps to the writer rank on a side stream)" % n_gpus,
           "inputs": "decoded uint8 images [batch,512,512,3]; the 4-scale bicubic / normalise / flip pyramids (C1) are built on the device "
                     "inside the timed region",
           "l2": "every step writes and re-reads %.1f GB of fp32 pyramids plus the activations between two reads of the inputs: "
                 "far beyond the 126 MB L2, nothing survives from one step to the next" % (batch * 47.2e6 / 1e9),
           "weights": "seeded synthetic checkpoints in the reference's state_dict format (irn_b200/synth.py)"}
    return cfg


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False
        self.proc = None

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def cpu_threads():
    # measured on the B200 host (profiles/r01_cpu_threads_probe.txt): 128 torch threads are 50x slower than 16-32
    return min(os.cpu_count(), int(os.environ.get("IRN_CPU_THREADS", "32")))


# ----------------------------------------------------------------------------------------------- CPU legs (oracle port)
def oracle_image(index, walk):
    """One image of the synthetic list through the oracle port of the reference chain on the host cores.
    walk='dense' REALLY executes the reference's algorithm (misc/indexing.py:112-139: 16384^2 fp32 matrix, 8 squarings)."""
    import torch
    from irn_b200 import synth
    from oracle import pipeline as opipe
    torch.set_num_threads(cpu_threads())
    torch.set_flush_denormal(True)     # the favourable setting for the reference's dense squarings (SURVEY.md section 6)
    if not hasattr(oracle_image, "sd"):
        oracle_image.sd = (synth.cam_state_dict(), synth.irn_state_dict())
    cam_sd, irn_sd = oracle_image.sd
    lab, t, aux = opipe.pseudo_label(synth.image(index, H, W), synth.label(index), cam_sd, irn_sd, SCALES, walk=walk)
    return lab, t


def cpu_baseline_and_parity(gpu_labels, ids, n_parity):
    """cpu_baseline: image ids[0] through the oracle port with the reference's dense walk, every squaring executed (no
    extrapolation).  parity: the first `n_parity` images of the batch through the oracle with the exact float64 stencil
    walk; label agreement and mIoU of the GPU label maps scored against the oracle's."""
    from oracle import steps as osteps
    t0 = time.perf_counter()
    _, t = oracle_image(ids[0], "dense")
    total = time.perf_counter() - t0
    cpu = {"value": 1.0 / total, "unit": UNIT, "cores": cpu_threads(), "kind": "port",
           "sample": "1 image (id %d) of the batch, every stage really executed: preprocess %.2fs + 4-scale CAM %.2fs + EdgeDisplacement %.2fs + "
                     "dense walk (16384^2 fp32 transition matrix, 8 squarings) %.2fs + labels %.2fs; torch CPU, flush-denormal on" %
                     (ids[0], t["preprocess"], t["cam"], t["irn"], t["walk"], t["labels"])}
    n = max(1, min(n_parity, len(ids)))
    labs = [oracle_image(i, "stencil")[0] for i in ids[:n]]
    got = [gpu_labels[k].cpu().numpy() for k in range(n)]
    agree = [float((a == b).mean()) for a, b in zip(labs, got)]
    _, miou = osteps.confusion_miou(got, labs)
    parity = {"images": n, "image_ids": [int(i) for i in ids[:n]], "label_agreement_vs_oracle": float(np.mean(agree)),
              "label_agreement_min": float(np.min(agree)), "miou_vs_oracle_labels": miou, "miou_pt_diff": 100.0 * (1.0 - miou),
              "oracle_walk": "float64 stencil (exact operator)",
              "unpinned": "skimage.measure.label and chainercv AP are absent in this image (scipy / restated): not part of this check"}
    return cpu, parity


def run_reference(a, rank, out_stream):
    """CPU oracle port of the reference path: each step = ONE image of the workload through every stage, nothing extrapolated
    (the dense walk alone is ~30 s on 32 cores), so the number of executed steps is capped to keep the run within minutes."""
    if rank != 0:
        return
    steps = max(1, min(a.steps, int(os.environ.get("IRN_REF_MAX_STEPS", "3"))))
    parts = {}
    t_all = time.perf_counter()
    for i in range(steps):
        lab, t = oracle_image(i, "dense")
        for k, v in t.items():
            parts[k] = parts.get(k, 0.0) + v / steps
    dt = time.perf_counter() - t_all
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {"labels": lab[None]})
    val = steps / dt
    sample = "1 image/step, %d of the requested %d steps executed (bounded: ~35 s of CPU per image), no warm-up, nothing extrapolated: PIL 4-scale " \
             "preprocessing + 4-scale CAM (torch CPU fp32) + EdgeDisplacement + dense 256-step walk (16384^2 fp32 transition matrix, all 8 squarings, " \
             "flush-denormal on) + labels; mean stage seconds %s" % (steps, a.steps, {k: round(v, 3) for k, v in parts.items()})
    cfg = config(a, a.gpus)      # the workload of the CUDA arm; every step here walks a bounded sample of it
    cfg["inputs"] = "decoded uint8 images; pyramids built by PIL on the host, as the reference's loader does"
    cfg["l2"] = "n/a (host run)"
    cfg["sample"] = "1 image of the batch per step"
    out_stream.write(json.dumps({"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": steps,
                                 "steps_requested": a.steps, "warmup": 0, "extrapolated": False,
                                 "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                                 "data": "synthetic", "config": cfg,
                                 "cpu_baseline": {"value": val, "unit": UNIT, "cores": cpu_threads(), "kind": "port", "sample": sample},
                                 "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}) + "\n")
    out_stream.flush()


def clocks_mhz(clocks):
    try:
        return float(clocks.get("sm_mhz") or 1800.0)
    except Exception:
        return 1800.0


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Native libraries (NCCL prints its version banner there when NCCL_DEBUG is set)
    write to file descriptor 1 behind Python's back, so fd 1 is pointed at stderr for the whole run and the JSON line goes to
    a private duplicate of the original stdout."""
    sys.stdout.flush()
    keep = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(keep, "w")


# ----------------------------------------------------------------------------------------------- --dump-outputs
DUMP_BYTES = 64_000_000


def dump_outputs(dirname, arrays):
    """Write each array as DIR/<name>.npy: int64 / int32 / float64 data as float64, everything else (labels, masks, classes,
    float32 maps) as float32 -- exact either way.  The files share DUMP_BYTES: the smaller arrays are stored whole first and
    the rest split what is left equally; an array larger than its share is stored as the sample of its flattened elements at
    a seeded set of indices, in increasing order: the same indices for the same shape in every run."""
    os.makedirs(dirname, exist_ok=True)
    arrays = {k: np.asarray(v.detach().cpu() if hasattr(v, "detach") else v) for k, v in arrays.items()}
    left, total = DUMP_BYTES - 1024 * len(arrays), 0          # 1 KB per file for the .npy header
    for i, name in enumerate(sorted(arrays, key=lambda k: arrays[k].size)):
        a = arrays[name]
        dt = np.float64 if a.dtype == np.float64 or (a.dtype.kind in "iu" and a.itemsize >= 4) else np.float32
        n = left // (len(arrays) - i) // np.dtype(dt).itemsize
        if a.size > n:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, n, replace=False))]
        a = np.ascontiguousarray(a, dtype=dt)
        np.save(os.path.join(dirname, name + ".npy"), a)
        left -= a.nbytes
        total += a.nbytes
    print("[bench] --dump-outputs: %d arrays, %.1f MB in %s" % (len(arrays), total / 1e6, dirname), file=sys.stderr)


def step_outputs(config_id, out):
    """What a caller of the timed step receives; per-image lists are concatenated along their first axis, with the
    per-image lengths beside them (-1: no detection dict for that image)."""
    import torch
    if config_id == 5:
        dets = out["detections"]
        got = [d for d in dets if d is not None]
        arrays = {"detections_per_image": [len(d["score"]) if d is not None else -1 for d in dets]}
        if got:
            for k in ("score", "class", "mask"):
                arrays["detection_" + k] = np.concatenate([np.asarray(d[k]) for d in got])
        return arrays
    arrays = {"keys_per_image": [len(k) for k in out["keys"]], "keys": np.concatenate(out["keys"]), "cams": torch.cat(out["cams"])}
    if out.get("high_res") is not None:
        arrays["high_res"] = torch.cat(out["high_res"])
    for k in ("labels", "edge", "dp"):
        if k in out:
            arrays[k] = out[k]
    return arrays


def stored_outputs(root, tag, n_ids, n_sample=16):
    """--config 4 returns files: the CAM dicts and label maps the pass `tag` wrote, for a seeded sample of the ids."""
    from PIL import Image
    pick = np.sort(np.random.default_rng(0).choice(n_ids, min(n_sample, n_ids), replace=False))
    cams = [np.load(os.path.join(root, "out_%s_cam" % tag, "2007_%06d.npy" % i), allow_pickle=True).item() for i in pick]
    return {"ids": pick, "keys_per_image": [len(c["keys"]) for c in cams], "keys": np.concatenate([np.asarray(c["keys"]) for c in cams]),
            "cams": np.concatenate([np.asarray(c["cam"]) for c in cams]), "high_res": np.concatenate([c["high_res"] for c in cams]),
            "labels": np.stack([np.asarray(Image.open(os.path.join(root, "out_%s_sem" % tag, "2007_%06d.png" % i))) for i in pick])}


# ----------------------------------------------------------------------------------------------- torch-eager context arm
def eager_baseline(dev, batch_images):
    """The 'existing Blackwell path' for the convolution part (BASELINE.md section 3): the oracle's functional restatement of
    the reference networks run by torch eager on this GPU (cuDNN / ATen), CAM forward at the four scales + IRNet forward on
    `batch_images` image pairs -- with cuDNN's TF32 convolutions (torch's default; misses the 1e-4 contract by ~20x, SURVEY.md
    H1) and with allow_tf32=False (IEEE fp32, the accuracy-equivalent arm).  Context only: it is not the reference arm."""
    import torch
    import torch.nn.functional as F
    from irn_b200 import synth
    from oracle import nets
    sd_c = {k: v.to(dev) for k, v in synth.cam_state_dict().items()}
    sd_i = {k: v.to(dev) for k, v in synth.irn_state_dict().items()}
    out = {}
    sizes = [(int(round(H * s)), int(round(W * s))) for s in SCALES]
    xs = [torch.randn(2 * batch_images, 3, h, w, device=dev) for h, w in sizes]

    def fwd():
        for x in xs:
            f = nets.trunk(x, sd_c)[-1]
            F.relu(F.conv2d(f, sd_c["classifier.weight"]))
        nets.irn_forward(xs[0], sd_i)
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cudnn.benchmark)
    try:
        torch.backends.cudnn.benchmark = True
        with torch.no_grad():
            for name, tf32 in (("cudnn_tf32", True), ("cudnn_fp32", False)):
                torch.backends.cudnn.allow_tf32 = tf32
                for _ in range(2):
                    fwd()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(3):
                    fwd()
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / 3 / batch_images
                out[name] = {"conv_path_ms_per_image": ms, "algorithmic_tflops": (GFLOP_CAM + GFLOP_IRN) / ms}
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cudnn.benchmark = old
    out["note"] = "torch %s eager (cuDNN/ATen) running oracle.nets on cuda, %d image pairs per forward, convolution path only (CAM x4 scales + IRNet, " \
                  "no pyramids / merge / walk / labels)" % (torch.__version__, batch_images)
    return out


# ----------------------------------------------------------------------------------------------- config 4: files through the steps
def _write_jpeg(job):
    from PIL import Image
    from irn_b200 import synth
    idx, path = job
    Image.fromarray(synth.image(idx, H, W)).save(path, quality=95)
    return path


def build_voc_tree(root, n_ids, distinct=128):
    """A synthetic VOC tree: JPEGImages/<id>.jpg for n_ids ids (`distinct` seeded 512x512 images encoded once as real JPEG
    files, the other ids are symlinks cycling over them: every id costs a real file read + JPEG decode), an id list and the
    class-label dict (1-3 classes per image, the K histogram of voc12/cls_labels.npy)."""
    import multiprocessing as mp
    from irn_b200 import synth
    os.makedirs(os.path.join(root, "JPEGImages"), exist_ok=True)
    distinct = min(distinct, n_ids)
    ids = ["2007_%06d" % i for i in range(n_ids)]
    jobs = [(i, os.path.join(root, "JPEGImages", ids[i] + ".jpg")) for i in range(distinct)]
    with mp.get_context("fork").Pool(min(32, os.cpu_count() or 1)) as pool:
        pool.map(_write_jpeg, jobs)
    for i in range(distinct, n_ids):
        dst = os.path.join(root, "JPEGImages", ids[i] + ".jpg")
        if not os.path.lexists(dst):
            os.symlink(ids[i % distinct] + ".jpg", dst)
    with open(os.path.join(root, "list.txt"), "w") as f:
        f.write("\n".join(ids) + "\n")
    labels = {int(n.replace("_", "")): synth.label(i) for i, n in enumerate(ids)}
    np.save(os.path.join(root, "cls_labels.npy"), labels, allow_pickle=True)
    return ids


def run_config4(a, rank, world, local, dev, out_stream):
    """BASELINE.json configs[3]: the image list through the reference's step entry points -- `step.make_cam._work` then
    `step.make_sem_seg_labels._work` on this rank's stride shard (torchrun replaces the reference's multiprocessing.spawn;
    one process per GPU either way), JPEG files in, .npy and .png files out.  Wall-clock timed (loader workers, file
    I/O and writer threads are part of the path), max over ranks."""
    import shutil
    import types
    import torch
    import torch.distributed as dist
    from irn_b200 import synth
    from irn_b200.cam import CAM
    from irn_b200.irn import EdgeDisplacement
    from irn_b200.misc import torchutils
    from irn_b200.step import _common, make_cam, make_sem_seg_labels
    from irn_b200.voc12 import dataloader as vd
    from irn_b200 import _lib
    L = _lib.lib()
    n_ids = a.list_limit or (N_TRAIN_AUG * world + 7) // 8
    root = os.environ.get("IRN_BENCH_TMP", "/tmp/irn_bench_voc")
    if rank == 0:
        shutil.rmtree(root, ignore_errors=True)
        t0 = time.perf_counter()
        build_voc_tree(root, n_ids)
        print("[bench] synthetic VOC tree: %d ids in %.1f s" % (n_ids, time.perf_counter() - t0), file=sys.stderr)
    if world > 1:
        dist.barrier()
    vd._cls_labels["voc12/cls_labels.npy"] = np.load(os.path.join(root, "cls_labels.npy"), allow_pickle=True).item()
    workers = a.num_workers if a.num_workers >= 0 else max(2, min(12, (os.cpu_count() or 8) // max(world, 1) // 2))
    n_vis = max(torch.cuda.device_count(), 1)

    def mk_args(tag, list_path):
        d = {k: os.path.join(root, "out_%s_%s" % (tag, k)) for k in ("cam", "sem")}
        for p in d.values():
            os.makedirs(p, exist_ok=True)
        return types.SimpleNamespace(num_workers=workers * n_vis, voc12_root=root, train_list=list_path, infer_list=list_path,
                                     cam_scales=SCALES, cam_out_dir=d["cam"], sem_seg_out_dir=d["sem"], beta=10, exp_times=8,
                                     sem_seg_bg_thres=0.25, synthetic=0, step_batch=a.step_batch, device_pyramid=True)

    cam = CAM()
    cam.load_state_dict(synth.cam_state_dict(), strict=True)
    irn = EdgeDisplacement()
    irn.load_state_dict(synth.irn_state_dict(), strict=False)
    cam.cuda(dev), irn.cuda(dev)
    if a.conv_mode >= 0:
        for m in (cam, irn):
            _lib.check(L.irn_net_set_conv_mode(m._get_plan(dev).handle, a.conv_mode))

    pass_seconds = {}

    def one_pass(args, n):
        """process_id = local rank: the shard list is indexed by it exactly as the reference's spawn would."""
        for name, scales, work, model in (("make_cam", SCALES, make_cam._work, cam), ("make_sem_seg_labels", (1.0,), make_sem_seg_labels._work, irn)):
            t_pass = time.perf_counter()
            ds = vd.VOC12ClassificationDatasetMSF(args.train_list, voc12_root=root, scales=scales, decode_only=True,
                                                  cls_labels_path="voc12/cls_labels.npy",
                                                  cam_dir=args.cam_out_dir if name == "make_sem_seg_labels" else None)   # as step.*.run does
            shards = torchutils.split_dataset(ds, world)
            pad = [None] * n_vis
            pad[local] = shards[rank]
            work(local, model, pad, args)
            torch.cuda.synchronize()
            if n:
                pass_seconds[name] = pass_seconds.get(name, 0.0) + time.perf_counter() - t_pass

    # warm-up: three passes over a two-batch list per rank (plans, pinned buffers, loader start-up, file-system caches)
    warm_list = os.path.join(root, "warm.txt")
    if rank == 0:
        with open(warm_list, "w") as f:
            f.write("\n".join("2007_%06d" % i for i in range(min(n_ids, 2 * a.step_batch * world))) + "\n")
    if world > 1:
        dist.barrier()
    for _ in range(max(a.warmup, 3)):
        one_pass(mk_args("warm", warm_list), 0)
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = L.irn_total_launch_count()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(a.steps):
        one_pass(mk_args("run%d" % k, os.path.join(root, "list.txt")), n_ids)
    wall = time.perf_counter() - t0
    launches = int(L.irn_total_launch_count() - launches0)
    clocks = sampler.stop()
    t = torch.tensor([wall], device=dev, dtype=torch.float64)
    per_rank = [wall]
    if world > 1:
        allw = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allw, t)
        per_rank = [float(x) for x in allw]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    wall = float(t[0])
    n_png = len(os.listdir(os.path.join(root, "out_run0_sem")))
    if world > 1:
        dist.barrier()
    value = n_ids * a.steps / wall
    cfg = config(a, world)
    cfg.update({"workload": "VOC12 train_aug-sized list: %d ids (10,582 * %d/8) of synthetic-filled 512x512 JPEG files (128 distinct seeded images, the "
                            "other ids symlink to them) through step.make_cam._work + step.make_sem_seg_labels._work (--step_batch %d, %d loader "
                            "workers per GPU): JPEG decode -> 4-scale CAM -> .npy files -> IRNet edge -> 256-iter walk -> .png files "
                            "(BASELINE.json configs[3])" % (n_ids, world, a.step_batch, workers),
                "global_batch": n_ids, "inputs": "JPEG files on local disk, decoded by DataLoader workers (PIL); pyramids built on the device",
                "outputs": "%d .npy CAM dicts + %d .png label maps per pass (reference formats)" % (n_ids, n_png)})
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
            "ms_per_step": 1e3 * wall / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": cfg, "timing": "wall clock around the step entry points, max over ranks",
            "per_rank_seconds": per_rank, "rank0_pass_seconds": pass_seconds,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": int(n_ids // world * H * W * 3), "d2h_bytes_per_step": None,
                    "api": "step.make_cam._work + step.make_sem_seg_labels._work (reference entry points), files in / files out"},
            "gpu_launches": launches, "clocks": clocks, "conv_mode": conv_mode_name(L, cam, dev)}
    if rank == 0:
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, stored_outputs(root, "run%d" % (a.steps - 1), n_ids))
        out_stream.write(json.dumps(line) + "\n")
        out_stream.flush()
        shutil.rmtree(root, ignore_errors=True)


def conv_mode_name(L, cam, dev):
    try:
        return CONV_MODES.get(int(L.irn_net_get_conv_mode(cam._get_plan(dev).handle)), "?")
    except Exception:
        return "?"


# ----------------------------------------------------------------------------------------------- main
def main():
    a = parse()
    out_stream = _claim_stdout()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if a.impl == "reference":
        run_reference(a, rank, out_stream)
        return

    import torch
    import torch.distributed as dist
    import __graft_entry__ as entry
    if not os.path.exists(entry.LIB):
        entry.build()
    from irn_b200 import _lib, synth
    from irn_b200.cam import CAM
    from irn_b200.irn import EdgeDisplacement
    from irn_b200.pipeline import PseudoLabelPipeline

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback; use --impl reference for the CPU oracle)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.lib()
    if a.config == 4:
        run_config4(a, rank, world, local, dev, out_stream)
        if world > 1:
            dist.destroy_process_group()
        return

    cam = CAM()
    cam.load_state_dict(synth.cam_state_dict(), strict=True)
    irn = EdgeDisplacement()
    irn.load_state_dict(synth.irn_state_dict(), strict=False)
    cam.cuda(dev), irn.cuda(dev)
    if a.conv_mode >= 0:
        for m in (cam, irn):
            _lib.check(L.irn_net_set_conv_mode(m._get_plan(dev).handle, a.conv_mode))
    pipe = PseudoLabelPipeline(cam, irn, dev, SCALES, rw_sub_batch=64)

    # ---- synthetic inputs: rank r takes images r, r+N, ... of the global list (misc/torchutils.py:66-68)
    B = a.batch
    ids = [rank + world * i for i in range(B)]
    labels = np.stack([synth.label(i) for i in ids])
    host_inputs = torch.from_numpy(np.stack([synth.image(i, H, W) for i in ids])).pin_memory()     # uint8 [B,H,W,3]
    dev_inputs = host_inputs.to(dev)
    h2d_bytes = int(host_inputs.numel())
    side = torch.cuda.Stream(device=dev)

    # ---- per-config step functions; each returns the step's device result, result_to_host() reads it back for the e2e leg
    if a.config == 3:
        host_labels = torch.empty((B, H, W), dtype=torch.uint8).pin_memory()
        d2h_bytes = B * H * W
        send = [torch.empty((B, H, W), dtype=torch.uint8, device=dev) for _ in range(2)] if world > 1 else None
        recv = [[torch.empty((B, H, W), dtype=torch.uint8, device=dev) for _ in range(world)] for _ in range(2)] if world > 1 and rank == 0 else None
        pending = [None, None]
        counter = [0]

        def step(from_host):
            out = pipe.run_u8(host_inputs if from_host else dev_inputs, labels, want_highres=False)
            if world > 1:
                # the one collective: this step's label maps to the writer rank, on a side stream, overlapped with the next step
                k = counter[0] & 1
                counter[0] += 1
                main = torch.cuda.current_stream(dev)
                if pending[k] is not None:
                    main.wait_event(pending[k])            # the gather that last read send[k] has finished
                send[k].copy_(out["labels"])
                ready = torch.cuda.Event()
                ready.record(main)
                with torch.cuda.stream(side):
                    side.wait_event(ready)
                    dist.gather(send[k], recv[k] if rank == 0 else None, dst=0)
                    done = torch.cuda.Event()
                    done.record(side)
                pending[k] = done
            if from_host:
                host_labels.copy_(out["labels"], non_blocking=True)
            return out

        def finish():
            main = torch.cuda.current_stream(dev)
            for ev in pending:
                if ev is not None:
                    main.wait_event(ev)
        api = "PseudoLabelPipeline.run_u8 on pinned host uint8 images (decoded JPEGs); label maps copied back to pinned host memory"
    elif a.config == 2:
        d2h_bytes = None
        host_out = {}

        def step(from_host):
            xs = pipe.pyramids(host_inputs if from_host else dev_inputs)
            keys, strided, highres = pipe.cam_stage(xs, labels, (H, W), want_highres=True)
            out = {"keys": keys, "cams": strided, "high_res": highres}
            if from_host:      # what make_cam stores per image: the stride-4 CAMs and the full-resolution CAMs
                lo, hi = torch.cat(strided, 0), torch.cat(highres, 0)
                for name, t in (("lo", lo), ("hi", hi)):
                    if name not in host_out or host_out[name].shape != t.shape:
                        host_out[name] = torch.empty(t.shape, dtype=t.dtype).pin_memory()
                    host_out[name].copy_(t, non_blocking=True)
            return out

        def finish():
            pass
        api = "PseudoLabelPipeline.pyramids + cam_stage on pinned host uint8 images; stride-4 and full-resolution CAMs (what make_cam saves) copied back"
    else:   # config 5
        with torch.no_grad():
            keys0, strided0, _ = pipe.cam_stage(pipe.pyramids(dev_inputs), labels, (H, W), want_highres=False)
        strided0 = [s.clone() for s in strided0]
        host_seeds = [s.cpu().pin_memory() for s in strided0]
        torch.cuda.synchronize()
        d2h_bytes = None

        def step(from_host):
            seeds = [s.to(dev, non_blocking=True) for s in host_seeds] if from_host else strided0
            dets = pipe.run_instances_u8(host_inputs if from_host else dev_inputs, keys0, seeds)    # detections arrive on the host (masks D2H inside)
            return {"detections": dets, "keys": keys0}

        def finish():
            pass
        h2d_bytes += int(sum(s.numel() * 4 for s in host_seeds))
        api = "PseudoLabelPipeline.run_instances_u8 on pinned host uint8 images + the stored stride-4 CAMs; detection dicts (scores, masks, classes) on the host"

    def timed(n_steps, from_host):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        out = None
        for _ in range(n_steps):
            out = step(from_host)
        finish()
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        if world > 1:
            dist.barrier()
        ms = max(e0.elapsed_time(e1), 0.0)
        t = torch.tensor([ms, wall * 1e3], device=dev, dtype=torch.float64)
        per_rank = [ms]
        if world > 1:
            allt = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(allt, t)
            per_rank = [float(x[0]) for x in allt]
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]), out, per_rank

    for _ in range(max(a.warmup, 3)):
        step(False)
    finish()
    torch.cuda.synchronize()

    sampler = ClockSampler(local)
    sampler.start()
    L.irn_rw_set_timing(1)
    launches0 = L.irn_total_launch_count()
    ms_dev, wall_dev, out, per_rank_ms = timed(a.steps, False)
    launches = int(L.irn_total_launch_count() - launches0)
    import ctypes
    step_ms, n_it = ctypes.c_float(), ctypes.c_int()
    have_rw = a.config in (3, 5) and L.irn_rw_last_step_ms(ctypes.byref(step_ms), ctypes.byref(n_it)) == 0
    L.irn_rw_set_timing(0)
    if a.dump_outputs and rank == 0:             # before any further step reuses the device buffers
        dump_outputs(a.dump_outputs, step_outputs(a.config, out))
    step(True)                                   # warm the host path (pinned copies)
    finish()
    ms_e2e, wall_e2e, out, _ = timed(a.steps, True)

    # ---- convolution path alone (CAM forward at the four scales + IRNet forward of the same batch), CUDA events
    conv_ms = None
    if a.config in (2, 3):
        with torch.no_grad():
            xs = pipe.pyramids(dev_inputs)

            def conv_path():
                for k, s in enumerate(SCALES):
                    sub = max(1, int(pipe.cam_sub * (2.0 / s) ** 2))
                    for i in range(0, B, sub):
                        cam.forward_batch(xs[k][2 * i:2 * min(i + sub, B)])
                if a.config == 3:
                    pipe.irn_stage(xs[0])
            conv_path()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(2):
                conv_path()
            e1.record()
            torch.cuda.synchronize()
            conv_ms = e0.elapsed_time(e1) / 2
    clocks = sampler.stop()

    value = world * B * a.steps / (ms_dev / 1e3)
    e2e = world * B * a.steps / (max(ms_e2e, wall_e2e) / 1e3)   # host-side time counts for the end-to-end number

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    roofline = None
    if have_rw and a.config == 3:
        counts = [len(k) for k in out["keys"]]
        last = counts[-(len(counts) % pipe.rw_sub or pipe.rw_sub):]
        n_img, totc, N = len(last), sum(last), (H // 4) * (W // 4)
        # SURVEY.md section 8(d) B_rw per walk step with e = 8 (fp64 state): N * [4*34 (A^beta) + 4 (1/s)] per image + 2*8*N per channel
        alg_step = N * (n_img * (4 * 34 + 4) + 2 * 8 * totc)
        src = "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s"
        if L.irn_rw_last_was_fused():
            # the whole walk is ONE launch: algorithmic bytes = n_iter x the per-step figure (SURVEY.md 8(d) B_rw; DESIGN.md 4)
            launch_ms = step_ms.value * n_it.value
            alg = alg_step * n_it.value
            traffic = None
            try:
                t = json.load(open(os.path.join(ROOT, "profiles", "rw_fused_traffic.json")))
                traffic = int(t["dram_bytes_per_item"] * totc)
            except Exception:
                pass
            ach = alg / (launch_ms * 1e-3) / 1e9
            wf_per_warp_step = (34 * 2 - 16) * 4 + 108 * 2      # weight LDS.32 (16 planes' forward taps come from registers) + state LDS.64 x 2 wavefronts
            clusters = max(1, int(L.irn_rw_last_was_fused()))
            per = -(-totc // clusters)                         # items walked by the busiest cluster
            smem_cycles = wf_per_warp_step * 8 * per * n_it.value   # 8 warps per CTA, one 128-byte wavefront per cycle per SM
            roofline = {"kernel": "rw_fused_kernel", "bound": "hbm", "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm,
                        "traffic": traffic, "peak_source": src, "launch_us": 1e3 * launch_ms, "steps_per_launch": n_it.value,
                        "images_per_launch": n_img, "channels_per_launch": totc, "algorithmic_bytes_per_launch": alg,
                        "algorithmic_bytes_formula": "256 steps x N=16384 x [images x (4*34 + 4) + channels x 2*8] (SURVEY.md 8(d), fp64 state)",
                        "note": "weights stay resident in shared memory for all steps of a launch, so DRAM traffic (`traffic`) is a small "
                                "fraction of the algorithmic bytes and frac may exceed 1; the kernel's real ceiling is shared-memory bandwidth, which scales "
                                "with the SM clock: the launch is timed INSIDE the step, at the clock the power cap leaves the conv kernels "
                                "(`clocks.sm_mhz`): 0.80 at ~1830 MHz (round 1's lighter conv path), ~0.70 at ~1570 MHz; it occupies 7 clusters x 16 "
                                "CTAs = 112 of 148 SMs (one 16-CTA cluster per GPC that has 16 free SMs)",
                        "clusters": clusters, "smem_wavefront_frac": smem_cycles / (launch_ms * 1e-3 * clocks_mhz(clocks) * 1e6)}
        else:
            traffic = None
            try:
                traffic = json.load(open(os.path.join(ROOT, "profiles", "rw_step_traffic.json")))["dram_bytes_per_launch"]
            except Exception:
                pass
            ach = alg_step / (step_ms.value * 1e-3) / 1e9
            roofline = {"kernel": "rw_step_tma_kernel", "bound": "hbm", "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm,
                        "traffic": traffic, "peak_source": src, "launch_us": 1e3 * step_ms.value, "images_per_launch": n_img,
                        "channels_per_launch": totc, "algorithmic_bytes_per_launch": alg_step}
    mode = int(L.irn_net_get_conv_mode(cam._get_plan(dev).handle))
    mode_irn = int(L.irn_net_get_conv_mode(irn._get_plan(dev).handle))
    bf16_peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    tf32_peak = bf16_peak / 2.0
    roofline_conv = None
    if conv_ms:
        gflop = B * (GFLOP_CAM + (GFLOP_IRN if a.config == 3 else 0.0))
        ach_tf = gflop / conv_ms                              # GFLOP / ms = TFLOP/s
        # tensor time the issued MMAs need at the measured peak of their kind (3 MMA passes per product in every split mode)
        cam_peak = bf16_peak if mode == 2 else tf32_peak
        irn_peak = bf16_peak if mode_irn == 2 else tf32_peak
        t_issued = 3 * B * GFLOP_CAM / cam_peak + (3 * B * GFLOP_IRN / irn_peak if a.config == 3 else 0.0)      # ms
        roofline_conv = {"bound": "tensor", "kernel": "conv_tc_* (tcgen05 implicit-GEMM convolutions)", "achieved": ach_tf, "unit": "TFLOP/s",
                         "peak": cam_peak, "frac": ach_tf / cam_peak, "frac_issued": t_issued / conv_ms,
                         "conv_path_ms_per_step": conv_ms, "share_of_step": conv_ms / (ms_dev / a.steps),
                         "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained%s" % (" (kind::f16 MMAs run at the bf16 rate)" if mode == 2 else " / 2 (tf32 runs at half the bf16 rate)"),
                         "note": "achieved = algorithmic conv FLOPs (974.04 CAM + 149.61 IRNet GFLOP/image) / CUDA-event time of the CAM x4-scale and "
                                 "IRNet forwards of one batch (re-run after the timed region; includes their ~4% of pooling / GroupNorm glue kernels); "
                                 "frac = achieved / peak of the MMA kind the CAM trunk uses; frac_issued = tensor time of the issued MMAs (3 per "
                                 "product: hi*hi + hi*lo + lo*hi) at their kind's measured peak / that time"}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
            "ms_per_step": ms_dev / a.steps, "wall_ms_per_step": wall_dev / a.steps, "per_rank_ms_per_step": [m / a.steps for m in per_rank_ms],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": config(a, world),
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "ms_per_step": max(ms_e2e, wall_e2e) / a.steps, "event_ms_per_step": ms_e2e / a.steps, "wall_ms_per_step": wall_e2e / a.steps,
                    "api": api},
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "roofline_conv": roofline_conv,
            "conv_mode": CONV_MODES.get(mode, "?"), "conv_mode_irnet": CONV_MODES.get(mode_irn, "?")}
    if a.config == 2:
        counts = [int(k.size) for k in out["keys"]]
        line["e2e"]["d2h_bytes_per_step"] = int(sum(counts) * (128 * 128 + H * W) * 4)
    if a.config == 5:
        dets = [d for d in out["detections"] if d is not None]
        line["e2e"]["d2h_bytes_per_step"] = int(sum(d["mask"].size + d["score"].size * 4 for d in dets))
        line["instances"] = {"images_with_detections": len(dets), "detections": int(sum(len(d["score"]) for d in dets)),
                             "walk_channels": int(sum(len(k) for k in out["keys"]))}
        if have_rw:
            line["walk"] = {"fused": bool(L.irn_rw_last_was_fused()), "step_us": 1e3 * step_ms.value, "iters": n_it.value}

    # ---- context + parity on a bounded sample (rank 0, single-GPU runs of the default config only)
    if rank == 0 and world == 1 and a.config == 3:
        if not a.no_eager_baseline:
            try:
                line["torch_eager_baseline"] = eager_baseline(dev, 8)
                if conv_ms:
                    line["torch_eager_baseline"]["ours_conv_path_ms_per_image"] = conv_ms / B
            except Exception as e:   # context only: never fail the bench over it
                line["torch_eager_baseline"] = {"error": repr(e)[:200]}
        if not a.no_cpu_baseline:
            line["cpu_baseline"], line["parity"] = cpu_baseline_and_parity(out["labels"], ids, a.parity_images)
    if rank == 0:
        out_stream.write(json.dumps(line) + "\n")
        out_stream.flush()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
