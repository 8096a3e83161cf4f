"""The three label-generation steps end to end through their reference-compatible entry points
(`step.<name>.run(args)` with `--cam_network irn_b200.cam --irn_network irn_b200.irn`) on a tiny synthetic VOC tree,
against what the unmodified reference produced for the same files (tests/golden/steps.npz)."""
import os
import types

import numpy as np
import pytest
import torch
from PIL import Image

from conftest import golden_path, check_detections, unpack_masks, record
from irn_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def voc_tree(tmp_path_factory, cuda_dev):
    g = np.load(golden_path("steps.npz"))
    root = tmp_path_factory.mktemp("voc")
    os.makedirs(root / "JPEGImages")
    ids = [str(s) for s in g["ids"]]
    labels = {}
    for i, name in enumerate(ids):
        # the decoded pixels the reference saw, stored losslessly (PIL sniffs the format, the .jpg suffix is only a name)
        Image.fromarray(g["img%d" % i]).save(root / "JPEGImages" / (name + ".jpg"), format="PNG")
        labels[int(name.replace("_", ""))] = g["label%d" % i]
    np.save(root / "cls_labels.npy", labels, allow_pickle=True)
    (root / "list.txt").write_text("\n".join(ids) + "\n")
    for d in ("sess", "cam", "sem", "ins"):
        os.makedirs(root / d)
    torch.save(synth.cam_state_dict(), root / "sess" / "res50_cam.pth.pth")
    torch.save(synth.irn_state_dict(), root / "sess" / "res50_irn.pth")
    args = types.SimpleNamespace(
        num_workers=0, voc12_root=str(root), train_list=str(root / "list.txt"), infer_list=str(root / "list.txt"),
        cam_network="irn_b200.cam", irn_network="irn_b200.irn", cam_scales=(1.0, 0.5, 1.5, 2.0),
        cam_weights_name=str(root / "sess" / "res50_cam.pth"), irn_weights_name=str(root / "sess" / "res50_irn.pth"),
        cam_out_dir=str(root / "cam"), sem_seg_out_dir=str(root / "sem"), ins_seg_out_dir=str(root / "ins"),
        beta=10, exp_times=8, sem_seg_bg_thres=0.25, ins_seg_bg_thres=0.25, synthetic=0)
    from irn_b200.voc12 import dataloader
    dataloader._cls_labels["voc12/cls_labels.npy"] = labels     # the reference loads this file from the cwd at import time
    return g, ids, args


def test_make_cam_outputs(voc_tree):
    g, ids, args = voc_tree
    from irn_b200.step import make_cam
    make_cam.run(args)
    for i, name in enumerate(ids):
        d = np.load(os.path.join(args.cam_out_dir, name + ".npy"), allow_pickle=True).item()
        assert set(d) == {"keys", "cam", "high_res"}
        assert isinstance(d["cam"], torch.Tensor) and isinstance(d["high_res"], np.ndarray)   # SURVEY.md D6
        assert np.array_equal(d["keys"].numpy(), g["cam_keys%d" % i])
        assert np.abs(d["cam"].numpy() - g["cam_cam%d" % i]).max() < 1e-4      # max-normalised: absolute = relative to 1
        assert np.abs(d["high_res"] - g["cam_high%d" % i]).max() < 1e-4


def test_make_cam_host_pyramid_identical(voc_tree):
    """--device_pyramid False (PIL pyramids built by the loader, the reference's data path) writes the same bytes."""
    g, ids, args = voc_tree
    from irn_b200.step import make_cam
    host_args = types.SimpleNamespace(**vars(args))
    host_args.device_pyramid = False
    host_args.cam_out_dir = os.path.join(os.path.dirname(args.cam_out_dir), "cam_host")
    os.makedirs(host_args.cam_out_dir, exist_ok=True)
    make_cam.run(host_args)
    make_cam.run(args)
    for name in ids:
        a = np.load(os.path.join(args.cam_out_dir, name + ".npy"), allow_pickle=True).item()
        b = np.load(os.path.join(host_args.cam_out_dir, name + ".npy"), allow_pickle=True).item()
        assert np.array_equal(a["keys"].numpy(), b["keys"].numpy())
        assert np.array_equal(a["cam"].numpy(), b["cam"].numpy()) and np.array_equal(a["high_res"], b["high_res"])


def test_make_sem_seg_labels_outputs(voc_tree):
    g, ids, args = voc_tree
    from irn_b200.step import make_sem_seg_labels
    make_sem_seg_labels.run(args)
    for i, name in enumerate(ids):
        lab = np.asarray(Image.open(os.path.join(args.sem_seg_out_dir, name + ".png")))
        ref = g["sem%d" % i]
        assert lab.dtype == np.uint8 and lab.shape == ref.shape
        dis = float((lab != ref).mean())
        record("make_sem_seg_labels_vs_reference_png", image=name, disagreement=dis)
        # the oracle's exact-operator walk itself sits 2e-3 from the reference's fp32 dense walk on these images
        # (tests/test_oracle_golden.py); boundary pixels flip at 1e-5 float noise
        assert dis < 2.5e-3, "label disagreement %g" % dis


def test_make_ins_seg_labels_outputs(voc_tree):
    """Against the dicts the reference's own loop saved: detection count and order, classes, scores (1e-4), masks."""
    g, ids, args = voc_tree
    from irn_b200.step import make_ins_seg_labels
    make_ins_seg_labels.run(args)
    for i, name in enumerate(ids):
        d = np.load(os.path.join(args.ins_seg_out_dir, name + ".npy"), allow_pickle=True).item()
        ref_mask = unpack_masks(g, str(i))
        assert set(d) == {"score", "mask", "class"}
        assert d["mask"].dtype == bool and d["mask"].shape[1:] == ref_mask.shape[1:]
        worst = check_detections(d, g["ins_score%d" % i], ref_mask, g["ins_class%d" % i], score_tol=1e-4, pixel_tol=2.5e-3)
        record("make_ins_seg_labels_vs_reference", image=name, detections=len(d["score"]), reference_detections=len(g["ins_score%d" % i]),
               worst_mask_disagreement=worst, score_err=float(np.abs(np.sort(d["score"])[::-1][:3] - np.sort(g["ins_score%d" % i])[::-1][:3]).max()))


def _copy_args(args, root, tag, **over):
    a = types.SimpleNamespace(**vars(args))
    for k in ("cam_out_dir", "sem_seg_out_dir", "ins_seg_out_dir"):
        d = os.path.join(root, tag + "_" + k)
        os.makedirs(d, exist_ok=True)
        setattr(a, k, d)
    for k, v in over.items():
        setattr(a, k, v)
    return a


def _same_tree(a_dir, b_dir, names, kind):
    for n in names:
        if kind == "png":
            assert np.array_equal(np.asarray(Image.open(os.path.join(a_dir, n + ".png"))), np.asarray(Image.open(os.path.join(b_dir, n + ".png")))), n
            continue
        a = np.load(os.path.join(a_dir, n + ".npy"), allow_pickle=True).item()
        b = np.load(os.path.join(b_dir, n + ".npy"), allow_pickle=True).item()
        assert set(a) == set(b)
        for k in a:
            x, y = (v.numpy() if isinstance(v, torch.Tensor) else np.asarray(v) for v in (a[k], b[k]))
            assert type(a[k]) is type(b[k]) and x.dtype == y.dtype and np.array_equal(x, y), (n, k)


def test_batched_steps_write_the_same_files(voc_tree, tmp_path):
    """--step_batch 16 (buckets of equally-sized images through the batched pipeline, writer threads) against
    --step_batch 1 (the reference's one-image loop): identical files, byte for byte, for all three steps.  Synthetic 64x96
    images so that buckets really hold several images."""
    _, _, args = voc_tree
    from irn_b200.step import make_cam, make_sem_seg_labels, make_ins_seg_labels
    from irn_b200.step import _common
    names = ["2007_%06d" % i for i in range(5)]
    real = _common.make_dataset

    def small(a, list_path, scales, cam_dir=None):
        from irn_b200.voc12 import dataloader
        if _common.step_batch(a) == 1:
            cam_dir = None          # the one-image loop reads the stored CAMs itself, like the reference
        return dataloader.SyntheticMSF(5, size=(64, 96), scales=scales, decode_only=_common.device_pyramid(a), cam_dir=cam_dir)
    _common.make_dataset = small
    try:
        one = _copy_args(args, str(tmp_path), "b1", synthetic=5, step_batch=1, exp_times=5)
        many = _copy_args(args, str(tmp_path), "b16", synthetic=5, step_batch=3, exp_times=5)
        for a in (one, many):
            make_cam.run(a)
            make_sem_seg_labels.run(a)
            make_ins_seg_labels.run(a)
    finally:
        _common.make_dataset = real
    _same_tree(one.cam_out_dir, many.cam_out_dir, names, "npy")
    _same_tree(one.sem_seg_out_dir, many.sem_seg_out_dir, names, "png")
    _same_tree(one.ins_seg_out_dir, many.ins_seg_out_dir, names, "npy")


_SPAWN_CHILD = """
import os, sys, types, pickle
sys.path.insert(0, {root!r})
import torch
from irn_b200.step import make_cam, make_sem_seg_labels, make_ins_seg_labels
args = pickle.load(open({args!r}, 'rb'))
make_cam.run(args); make_sem_seg_labels.run(args); make_ins_seg_labels.run(args)
"""


def test_spawn_branch_matches_single_gpu(voc_tree, tmp_path):
    """The reference's multi-GPU seam (step/make_cam.py:67-74: stride split + torch.multiprocessing.spawn, one process per
    GPU) on every visible GPU, byte-compared with the same run restricted to one GPU (SURVEY.md section 4)."""
    import pickle
    import subprocess
    import sys
    from conftest import ROOT
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    _, _, args = voc_tree
    names = ["2007_%06d" % i for i in range(6)]
    runs = {}
    for tag, visible in (("multi", None), ("single", "0")):
        a = _copy_args(args, str(tmp_path), tag, synthetic=6, step_batch=2, exp_times=5, num_workers=0)
        pickle.dump(a, open(tmp_path / (tag + ".pkl"), "wb"))
        env = dict(os.environ, PYTHONPATH=ROOT)
        if visible is not None:
            env["CUDA_VISIBLE_DEVICES"] = visible
        r = subprocess.run([sys.executable, "-c", _SPAWN_CHILD.format(root=ROOT, args=str(tmp_path / (tag + ".pkl")))], env=env,
                           capture_output=True, text=True, timeout=900, cwd=str(tmp_path))
        assert r.returncode == 0, r.stderr[-3000:]
        runs[tag] = a
    _same_tree(runs["multi"].cam_out_dir, runs["single"].cam_out_dir, names, "npy")
    _same_tree(runs["multi"].sem_seg_out_dir, runs["single"].sem_seg_out_dir, names, "png")
    _same_tree(runs["multi"].ins_seg_out_dir, runs["single"].ins_seg_out_dir, names, "npy")


def test_run_sample_cli_synthetic(tmp_path, cuda_dev):
    """`python run_sample.py --synthetic N` (reference flag names, default output dirs) writes the three result trees."""
    import subprocess
    import sys
    from conftest import ROOT
    env = dict(os.environ, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "run_sample.py"), "--synthetic", "2", "--num_workers", "0", "--exp_times", "6"],
                       cwd=tmp_path, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    for i in range(2):
        name = "2007_%06d" % i
        d = np.load(tmp_path / "result" / "cam" / (name + ".npy"), allow_pickle=True).item()
        assert d["cam"].shape[1:] == (128, 128) and d["high_res"].shape[1:] == (512, 512)
        lab = np.asarray(Image.open(tmp_path / "result" / "sem_seg" / (name + ".png")))
        assert lab.shape == (512, 512) and lab.dtype == np.uint8
        ins = np.load(tmp_path / "result" / "ins_seg" / (name + ".npy"), allow_pickle=True).item()
        assert set(ins) == {"score", "mask", "class"} and ins["mask"].shape[1:] == (512, 512)
