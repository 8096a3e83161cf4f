"""Generate the golden fixtures in this directory by running the UNMODIFIED reference
(/root/reference, imported through oracle/refshim.py) on seeded synthetic inputs.

Run in the build container only:   python tests/golden/make_golden.py [--big]
(`--big` adds the 128x128 / exp_times=8 random-walk case: several minutes of CPU sgemm.)

The fixtures pin the oracle (tests/test_oracle_golden.py) and, on the GPU box, the CUDA path
(tests/test_gpu_*.py).  Nothing here runs on the GPU box.
"""
import argparse
import hashlib
import json
import os
import shutil
import sys
import tempfile
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import refshim  # noqa: E402
from irn_b200 import synth  # noqa: E402

RW_CASES = [  # (name, h, w, C, exp_times, edge kind, seed)
    ("16x16_c2_e0_uniform", 16, 16, 2, 0, "uniform", 0),
    ("16x16_c2_e8_uniform", 16, 16, 2, 8, "uniform", 0),
    ("20x28_c3_e4_sigmoid4", 20, 28, 3, 4, "sigmoid4", 1),
    ("24x21_c1_e8_bimodal", 24, 21, 1, 8, "bimodal", 2),
    ("33x47_c5_e6_low", 33, 47, 5, 6, "low", 3),
    ("40x40_c2_e8_bimodal", 40, 40, 2, 8, "bimodal", 4),
    ("64x64_c2_e8_bimodal", 64, 64, 2, 8, "bimodal", 5),
]
RW_BIG = ("128x128_c2_e8_bimodal", 128, 128, 2, 8, "bimodal", 6)


def sha_path_index(pi):
    h = hashlib.sha256()
    for p in pi.path_indices:
        h.update(np.ascontiguousarray(p, dtype=np.int64).tobytes())
    h.update(np.ascontiguousarray(pi.src_indices, dtype=np.int64).tobytes())
    h.update(np.ascontiguousarray(pi.dst_indices, dtype=np.int64).tobytes())
    h.update(np.ascontiguousarray(pi.search_dst, dtype=np.int64).tobytes())
    return h.hexdigest()


def gen_path_index(ref_indexing):
    out = {}
    for radius, size in [(5, (133, 138)), (5, (21, 26)), (5, (29, 31)), (10, (128, 128)), (3, (12, 17)), (2, (9, 9))]:
        pi = ref_indexing.PathIndex(radius, size)
        out["r%d_%dx%d" % (radius, size[0], size[1])] = {
            "radius": radius, "size": list(size), "sha256": sha_path_index(pi),
            "group_shapes": [list(p.shape) for p in pi.path_indices],
            "search_dst": np.asarray(pi.search_dst).tolist(),
            "src_head": pi.src_indices[:5].tolist(), "dst_head": pi.dst_indices[:, :3].tolist() if radius <= 5 else None,
        }
    json.dump(out, open(os.path.join(HERE, "path_index.json"), "w"), indent=0)
    print("path_index.json", {k: v["sha256"][:12] for k, v in out.items()})


def gen_rw(ref_indexing, case):
    name, h, w, C, et, kind, seed = case
    edge = synth.edge_map(h, w, kind, seed)
    x = synth.seeds(C, h, w, seed)
    with torch.no_grad():
        rw = ref_indexing.propagate_to_edge(torch.from_numpy(x), torch.from_numpy(edge), radius=5, beta=10, exp_times=et).numpy()
    np.savez_compressed(os.path.join(HERE, "rw_%s.npz" % name), x=x, edge=edge, rw=rw.astype(np.float32),
                        beta=10, exp_times=et, radius=5)
    print("rw", name, rw.shape, float(rw.max()))


def gen_affinity(ref_indexing):
    h, w, r = 12, 17, 5
    edge = synth.edge_map(h, w, "uniform", 7)
    pi = ref_indexing.PathIndex(r, (h + r, w + 2 * r))
    ep = torch.nn.functional.pad(torch.from_numpy(edge), (r, r, 0, r), value=1.0)
    aff = ref_indexing.edge_to_affinity(ep[None], pi.path_indices).numpy()   # [1, 34, (h+1)*(w+2)]
    np.savez_compressed(os.path.join(HERE, "affinity_12x17.npz"), edge=edge, aff=aff)
    print("affinity", aff.shape)


def gen_to_affinity(ref_indexing):
    """The reference's AffinityDisplacementLoss.to_affinity (net/resnet50_irn.py:162-175), forward and autograd backward, called
    UNBOUND on a stub that carries only what the method reads (the path-index buffers): constructing the real module would build
    a ResNet-50 for nothing."""
    from net import resnet50_irn as ref_irn
    out = {}
    for tag, r, h, w, B, kind, seed in (("r10", 10, 32, 36, 1, "sigmoid4", 3), ("r5", 5, 24, 31, 3, "uniform", 5), ("r10b", 10, 30, 30, 2, "bimodal", 9)):
        pi = ref_indexing.PathIndex(r, (h, w))
        stub = types.SimpleNamespace(n_path_lengths=len(pi.path_indices),
                                     _buffers={ref_irn.AffinityDisplacementLoss.path_indices_prefix + str(i): torch.from_numpy(p)
                                               for i, p in enumerate(pi.path_indices)})
        edge = np.stack([synth.edge_map(h, w, kind, seed + b) for b in range(B)])                # [B,1,h,w] like sigmoid(edge_out)
        e = torch.from_numpy(edge).requires_grad_(True)
        aff = ref_irn.AffinityDisplacementLoss.to_affinity(stub, e)
        g = torch.from_numpy(np.random.RandomState(seed).standard_normal(tuple(aff.shape)).astype(np.float32))
        aff.backward(g)
        out[tag + "_edge"], out[tag + "_aff"] = edge, aff.detach().numpy()
        out[tag + "_grad_edge"] = e.grad.numpy()       # for grad_aff = RandomState(seed).standard_normal(aff.shape) as float32
        out[tag + "_radius"], out[tag + "_seed"] = r, seed
        print("to_affinity", tag, tuple(aff.shape), float(np.abs(e.grad.numpy()).max()))
    np.savez_compressed(os.path.join(HERE, "to_affinity.npz"), **out)


def gen_reference_live(ref_indexing):
    """A second, independent record of the reference's outputs on a few of the inputs above (PathIndex, edge_to_affinity,
    one random walk, to_affinity forward and gradient), computed afresh rather than read back from the fixtures:
    tests/test_reference_live.py holds the fixtures to it."""
    from net import resnet50_irn as ref_irn
    out = {"path_sha": sha_path_index(ref_indexing.PathIndex(5, (21, 26)))}
    h, w, r = 12, 17, 5
    pi = ref_indexing.PathIndex(r, (h + r, w + 2 * r))
    ep = torch.nn.functional.pad(torch.from_numpy(synth.edge_map(h, w, "uniform", 7)), (r, r, 0, r), value=1.0)
    out["aff_sha"] = hashlib.sha256(np.ascontiguousarray(ref_indexing.edge_to_affinity(ep[None], pi.path_indices).numpy()).tobytes()).hexdigest()
    name, hh, ww, C, et, kind, seed = RW_CASES[1]
    with torch.no_grad():
        rw = ref_indexing.propagate_to_edge(torch.from_numpy(synth.seeds(C, hh, ww, seed)), torch.from_numpy(synth.edge_map(hh, ww, kind, seed)),
                                            radius=5, beta=10, exp_times=et)
    out["rw_name"], out["rw"] = name, rw.numpy().astype(np.float32)
    r, h, w, B, kind, seed = 5, 24, 31, 3, "uniform", 5          # case "r5" of gen_to_affinity
    pi = ref_indexing.PathIndex(r, (h, w))
    stub = types.SimpleNamespace(n_path_lengths=len(pi.path_indices),
                                 _buffers={ref_irn.AffinityDisplacementLoss.path_indices_prefix + str(i): torch.from_numpy(p) for i, p in enumerate(pi.path_indices)})
    e = torch.from_numpy(np.stack([synth.edge_map(h, w, kind, seed + b) for b in range(B)])).requires_grad_(True)
    aff = ref_irn.AffinityDisplacementLoss.to_affinity(stub, e)
    aff.backward(torch.from_numpy(np.random.RandomState(seed).standard_normal(tuple(aff.shape)).astype(np.float32)))
    out["toaff_sha"] = hashlib.sha256(np.ascontiguousarray(aff.detach().numpy()).tobytes()).hexdigest()
    out["toaff_grad"] = e.grad.numpy()
    np.savez_compressed(os.path.join(HERE, "reference_live.npz"), **out)
    print("reference_live", {k: getattr(v, "shape", v) for k, v in out.items()})


def gen_nets():
    import net.resnet50_cam as rcam
    import net.resnet50_irn as rirn
    sd = synth.cam_state_dict()
    cam = rcam.CAM()
    cam.load_state_dict(sd, strict=True)
    cam.eval()
    out = {}
    for i, (H, W) in enumerate([(64, 64), (80, 112), (256, 256)]):
        x = synth.normalize_image(synth.image(100 + i, H, W))
        x = np.stack([x, x[..., ::-1].copy()])
        with torch.no_grad():
            y = cam(torch.from_numpy(x)).numpy()
        out["x%d" % i] = x.astype(np.float32)
        out["y%d" % i] = y
        print("cam", (H, W), y.shape, float(y.max()))
    np.savez_compressed(os.path.join(HERE, "cam_forward.npz"), **out)

    sd2 = synth.irn_state_dict()
    irn = rirn.EdgeDisplacement()
    irn.load_state_dict(sd2, strict=False)
    irn.eval()
    out = {}
    for i, (H, W) in enumerate([(96, 128), (250, 333), (512, 512)]):
        x = synth.normalize_image(synth.image(200 + i, H, W))
        x = np.stack([x, x[..., ::-1].copy()])
        with torch.no_grad():
            e, d = irn(torch.from_numpy(x))
        if (H, W) != (512, 512):
            out["x%d" % i] = x.astype(np.float32)   # the 512 input is regenerated from the seed (3 MB otherwise)
        out["edge%d" % i] = e.numpy()
        out["dp%d" % i] = d.numpy()
        print("irn", (H, W), e.shape, d.shape)
    np.savez_compressed(os.path.join(HERE, "irn_forward.npz"), **out)
    return cam, irn


def load_nets():
    import net.resnet50_cam as rcam
    import net.resnet50_irn as rirn
    cam = rcam.CAM()
    cam.load_state_dict(synth.cam_state_dict(), strict=True)
    cam.eval()
    irn = rirn.EdgeDisplacement()
    irn.load_state_dict(synth.irn_state_dict(), strict=False)
    irn.eval()
    return cam, irn


def gen_steps(cam, irn):
    """Drive the reference's own step._work loops over a tiny synthetic VOC tree."""
    from PIL import Image
    import voc12.dataloader as vd
    import step.make_cam
    import step.make_sem_seg_labels
    import step.make_ins_seg_labels
    import imageio

    def safe_list(path):   # numpy-2 safe replacement for load_img_name_list (voc12/dataloader.py:58-62)
        return np.array([int(l.strip().replace("_", "")) for l in open(path) if l.strip()], dtype=np.int64)
    vd.load_img_name_list = safe_list

    # torch's default collate turns size=(H,W) into [tensor([H]), tensor([W])]; with numpy >= 1.25 the
    # reference's `[..., :orig_img_size[0], ...]` on np.asarray(pack['size']) (shape (2,1)) no longer
    # converts to an index (step/make_sem_seg_labels.py:29,43).  Version shim only: hand it plain ints.
    from torch.utils.data import DataLoader as _DL
    from torch.utils.data._utils.collate import default_collate

    def _collate(batch):
        out = default_collate(batch)
        out["size"] = (int(batch[0]["size"][0]), int(batch[0]["size"][1]))
        return out

    def _loader(ds, **kw):
        return _DL(ds, collate_fn=_collate, **kw)
    for m in (step.make_cam, step.make_sem_seg_labels, step.make_ins_seg_labels):
        m.DataLoader = _loader

    tmp = tempfile.mkdtemp(prefix="irn_golden_")
    try:
        os.makedirs(os.path.join(tmp, "JPEGImages"))
        ids = ["2007_000032", "2007_000039", "2007_000063"]
        sizes = [(96, 128), (121, 90), (75, 100)]
        for i, (name, (H, W)) in enumerate(zip(ids, sizes)):
            Image.fromarray(synth.image(300 + i, H, W)).save(os.path.join(tmp, "JPEGImages", name + ".jpg"), quality=95)
        lst = os.path.join(tmp, "list.txt")
        open(lst, "w").write("\n".join(ids) + "\n")
        args = types.SimpleNamespace(num_workers=0, cam_out_dir=os.path.join(tmp, "cam"), sem_seg_out_dir=os.path.join(tmp, "sem"),
                                     ins_seg_out_dir=os.path.join(tmp, "ins"), beta=10, exp_times=8,
                                     sem_seg_bg_thres=0.25, ins_seg_bg_thres=0.25)
        for d in (args.cam_out_dir, args.sem_seg_out_dir, args.ins_seg_out_dir):
            os.makedirs(d)

        # the reference prints progress with `iter % (len(databin)//20)` -> ZeroDivisionError for < 20 images (SURVEY D9);
        # run the loops with process_id=1 != n_gpus-1 so that branch is skipped, data bin passed as index 1.
        ds = vd.VOC12ClassificationDatasetMSF(lst, voc12_root=tmp, scales=(1.0, 0.5, 1.5, 2.0))
        with torch.no_grad():
            step.make_cam._work(1, cam, [None, ds], args)
        ds1 = vd.VOC12ClassificationDatasetMSF(lst, voc12_root=tmp, scales=(1.0,))
        with torch.no_grad():
            step.make_sem_seg_labels._work(1, irn, [None, ds1], args)
            step.make_ins_seg_labels._work(1, irn, [None, ds1], args)

        out = {}
        for i, name in enumerate(ids):
            out["img%d" % i] = np.asarray(Image.open(os.path.join(tmp, "JPEGImages", name + ".jpg")))
            out["label%d" % i] = vd.cls_labels_dict[int(name.replace("_", ""))]
            cd = np.load(os.path.join(args.cam_out_dir, name + ".npy"), allow_pickle=True).item()
            out["cam_keys%d" % i] = cd["keys"].numpy()
            out["cam_cam%d" % i] = cd["cam"].numpy()
            out["cam_high%d" % i] = cd["high_res"]
            out["sem%d" % i] = np.asarray(Image.open(os.path.join(args.sem_seg_out_dir, name + ".png")))
            ins = np.load(os.path.join(args.ins_seg_out_dir, name + ".npy"), allow_pickle=True).item()
            out["ins_score%d" % i] = np.asarray(ins["score"], np.float32)
            out["ins_mask%d" % i] = np.packbits(ins["mask"].astype(bool), axis=-1)
            out["ins_mask_shape%d" % i] = np.asarray(ins["mask"].shape)
            out["ins_class%d" % i] = np.asarray(ins["class"])
            print("steps", name, cd["cam"].shape, out["sem%d" % i].shape, ins["mask"].shape, np.unique(out["sem%d" % i]))
        out["ids"] = np.array(ids)
        np.savez_compressed(os.path.join(HERE, "steps.npz"), **out)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def gen_steps512(cam, irn):
    """The benchmark's size: ONE 512x512 synthetic image through the reference's own three `_work` loops (4-scale CAM at
    256/512/768/1024 inputs, EdgeDisplacement, the dense 16384^2 walk squared 8 times -- minutes of CPU sgemm -- for the
    sem-seg AND the ins-seg step).  Forward hooks / a wrapper around propagate_to_edge record the intermediate tensors
    (per-scale CAMs, edge, dp, walk outputs) without touching the reference's code.  The image is stored losslessly
    (PNG bytes under the .jpg name: PIL sniffs the format) so tests regenerate it from the seed."""
    from PIL import Image
    import voc12.dataloader as vd
    import step.make_cam
    import step.make_sem_seg_labels
    import step.make_ins_seg_labels
    from misc import indexing as ref_indexing

    def safe_list(path):
        return np.array([int(l.strip().replace("_", "")) for l in open(path) if l.strip()], dtype=np.int64)
    vd.load_img_name_list = safe_list
    from torch.utils.data import DataLoader as _DL
    from torch.utils.data._utils.collate import default_collate

    def _collate(batch):
        out = default_collate(batch)
        out["size"] = (int(batch[0]["size"][0]), int(batch[0]["size"][1]))
        return out

    def _loader(ds, **kw):
        return _DL(ds, collate_fn=_collate, **kw)
    for m in (step.make_cam, step.make_sem_seg_labels, step.make_ins_seg_labels):
        m.DataLoader = _loader

    name, seed = "2007_000170", 512      # a train_aug id whose real label has two classes
    label = vd.cls_labels_dict[int(name.replace("_", ""))]
    assert label.sum() >= 2, label
    tmp = tempfile.mkdtemp(prefix="irn_golden512_")
    rec = {"cam_scales": [], "walks": [], "irn": []}
    h1 = cam.register_forward_hook(lambda m, i, o: rec["cam_scales"].append((tuple(i[0].shape), o.detach().numpy().copy())))
    h2 = irn.register_forward_hook(lambda m, i, o: rec["irn"].append((o[0].detach().numpy().copy(), o[1].detach().numpy().copy())))
    orig = ref_indexing.propagate_to_edge

    def spy(x, edge, **kw):
        out = orig(x, edge, **kw)
        rec["walks"].append((tuple(x.shape), out.detach().numpy().copy()))
        return out
    ref_indexing.propagate_to_edge = spy
    try:
        os.makedirs(os.path.join(tmp, "JPEGImages"))
        Image.fromarray(synth.image(seed, 512, 512)).save(os.path.join(tmp, "JPEGImages", name + ".jpg"), format="PNG")
        lst = os.path.join(tmp, "list.txt")
        open(lst, "w").write(name + "\n")
        args = types.SimpleNamespace(num_workers=0, cam_out_dir=os.path.join(tmp, "cam"), sem_seg_out_dir=os.path.join(tmp, "sem"),
                                     ins_seg_out_dir=os.path.join(tmp, "ins"), beta=10, exp_times=8,
                                     sem_seg_bg_thres=0.25, ins_seg_bg_thres=0.25)
        for d in (args.cam_out_dir, args.sem_seg_out_dir, args.ins_seg_out_dir):
            os.makedirs(d)
        ds = vd.VOC12ClassificationDatasetMSF(lst, voc12_root=tmp, scales=(1.0, 0.5, 1.5, 2.0))
        with torch.no_grad():
            step.make_cam._work(1, cam, [None, ds], args)
        ds1 = vd.VOC12ClassificationDatasetMSF(lst, voc12_root=tmp, scales=(1.0,))
        import time
        with torch.no_grad():
            t0 = time.time()
            step.make_sem_seg_labels._work(1, irn, [None, ds1], args)
            print("sem-seg loop %.0f s" % (time.time() - t0), flush=True)
            t0 = time.time()
            step.make_ins_seg_labels._work(1, irn, [None, ds1], args)
            print("ins-seg loop %.0f s" % (time.time() - t0), flush=True)
        out = {"name": np.array(name), "seed": np.array(seed), "label": label}
        for shp, y in rec["cam_scales"]:
            out["camscale_%d" % shp[-1]] = y            # keyed by the input width: 512, 256, 768, 1024
        cd = np.load(os.path.join(args.cam_out_dir, name + ".npy"), allow_pickle=True).item()
        out["cam_keys"] = cd["keys"].numpy()
        out["cam_cam"] = cd["cam"].numpy()
        out["cam_high_s4"] = np.ascontiguousarray(cd["high_res"][:, 1::4, 2::4])     # every 4th pixel (rows 1::4, cols 2::4) of the full-res maps
        out["cam_high_max"] = cd["high_res"].reshape(cd["high_res"].shape[0], -1).max(1)
        out["edge"], out["dp"] = rec["irn"][0]
        assert np.array_equal(rec["irn"][0][0], rec["irn"][1][0])
        out["walk_sem"] = rec["walks"][0][1]
        out["walk_ins"] = rec["walks"][1][1]
        out["walk_ins_in_shape"] = np.asarray(rec["walks"][1][0])
        out["sem"] = np.asarray(Image.open(os.path.join(args.sem_seg_out_dir, name + ".png")))
        ins = np.load(os.path.join(args.ins_seg_out_dir, name + ".npy"), allow_pickle=True).item()
        out["ins_score"] = np.asarray(ins["score"], np.float32)
        out["ins_mask"] = np.packbits(ins["mask"].astype(bool), axis=-1)
        out["ins_mask_shape"] = np.asarray(ins["mask"].shape)
        out["ins_class"] = np.asarray(ins["class"])
        print("steps512", name, {k: getattr(v, "shape", None) for k, v in out.items()})
        np.savez_compressed(os.path.join(HERE, "steps512.npz"), **out)
    finally:
        h1.remove()
        h2.remove()
        ref_indexing.propagate_to_edge = orig
        shutil.rmtree(tmp, ignore_errors=True)


def gen_instance_fns():
    import step.make_ins_seg_labels as rins
    out = {}
    for i, (h, w, n) in enumerate([(40, 52, 3), (128, 128, 4), (33, 29, 2)]):
        dp = synth.displacement(h, w, n, seed=i)
        cen = rins.find_centroids_with_refinement(dp.copy())
        inst = rins.cluster_centroids(cen, dp)
        out["dp%d" % i] = dp
        out["centroids%d" % i] = cen
        out["instances%d" % i] = np.packbits(inst, axis=-1)
        out["instances_shape%d" % i] = np.asarray(inst.shape)
        print("centroids", (h, w), cen.shape, inst.shape)
    np.savez_compressed(os.path.join(HERE, "instance_fns.npz"), **out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--big", action="store_true")
    ap.add_argument("--only", default="")
    a = ap.parse_args()
    refshim.install()
    os.chdir(refshim.REF)          # voc12/dataloader.py:24 loads 'voc12/cls_labels.npy' relative to cwd
    torch.manual_seed(0)
    from misc import indexing as ref_indexing
    only = set(a.only.split(",")) if a.only else None

    def want(k):
        return only is None or k in only
    if want("path"):
        gen_path_index(ref_indexing)
    if want("aff"):
        gen_affinity(ref_indexing)
    if want("toaff"):
        gen_to_affinity(ref_indexing)
    if want("rw"):
        for c in RW_CASES:
            gen_rw(ref_indexing, c)
    if a.big:
        gen_rw(ref_indexing, RW_BIG)
    if want("live"):
        gen_reference_live(ref_indexing)
    if want("inst"):
        gen_instance_fns()
    if want("nets") or want("steps"):
        cam, irn = gen_nets()
        if want("steps"):
            gen_steps(cam, irn)
    if only is not None and "steps512" in only:      # minutes of CPU: only on request
        gen_steps512(*load_nets())


if __name__ == "__main__":
    main()
