"""Generate tests/golden/*.npz from the UNMODIFIED reference (build container only).

Run:  python -m oracle.make_golden        (needs /root/reference; no GPU)

The reference has no tests or golden vectors of its own (SURVEY.md section 4), so these
fixtures are what pins parity: they are produced by the reference's own
``embedding.UniDirsEmbed`` / ``model.OccupancyMap`` / ``render_rays`` /
``loss.step_batch_loss`` driven exactly like train.py:181-182,293-326
(functorch ``combine_state_for_ensemble`` + ``vmap`` + ``torch.optim.AdamW``),
and by ``vmap.sceneObject.get_training_samples`` (vmap.py:319-459).
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import _refload  # noqa: E402
from oracle import vmap_oracle as vo  # noqa: E402
from oracle import sampler_oracle as so  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def _np(t):
    return t.detach().cpu().numpy().copy()


def reference_step_case(name, n_obj, hidden, n_rays, n_samples, scale, n_cam2surf, seed,
                        n_steps=0, kill_depth_obj=None):
    model, embedding, render_rays, loss = _refload.load("model", "embedding", "render_rays", "loss")
    from functorch import combine_state_for_ensemble, vmap

    torch.manual_seed(seed)
    e1, e2 = vo.emb_sizes(5)
    fcs, pes = [], []
    for _ in range(n_obj):                      # trainer.py:27-33
        fc = model.OccupancyMap(e1, e2, hidden_size=hidden)
        fc.apply(model.init_weights)
        fcs.append(fc)
        pes.append(embedding.UniDirsEmbed(max_deg=5, scale=scale))
    batch = vo.synthetic_batch(n_obj, n_rays, n_samples, seed=seed + 100, n_cam2surf=n_cam2surf)
    if kill_depth_obj is not None:              # exercise the any-empty early-out
        batch["mask_depth"][kill_depth_obj] = False

    opt = torch.optim.AdamW([torch.zeros(1, requires_grad=True)], lr=1e-3, weight_decay=0.013)  # train.py:67
    fc_model, fc_param, fc_buffer = combine_state_for_ensemble(fcs)       # utils.py:31
    [p.requires_grad_() for p in fc_param]
    opt.add_param_group({"params": fc_param})
    pe_model, pe_param, pe_buffer = combine_state_for_ensemble(pes)
    [p.requires_grad_() for p in pe_param]
    opt.add_param_group({"params": pe_param})

    out = {"scale": np.float32(scale), "hidden": np.int32(hidden), "n_cam2surf": np.int32(n_cam2surf)}
    for k, v in batch.items():
        out["in_" + k] = _np(v)
    fc_names = [n for n, _ in fcs[0].named_parameters()]
    assert tuple(fc_names) == vo.FC_KEYS, fc_names
    for n, p in zip(fc_names, fc_param):
        out["p0_" + n] = _np(p)
    out["p0_" + vo.PE_KEY] = _np(pe_param[0])

    def fwd_loss():
        emb = vmap(pe_model)(pe_param, pe_buffer, batch["pcs"])           # train.py:293
        alpha, col = vmap(fc_model)(fc_param, fc_buffer, emb)             # train.py:294
        l, _ = loss.step_batch_loss(alpha, col, batch["gt_depth"], batch["gt_colour"],
                                    batch["sem"], batch["mask_depth"], batch["z"])   # train.py:303
        return emb, alpha, col, l

    emb, alpha, col, l = fwd_loss()
    out["emb_obj0_ray0"] = _np(emb[0, 0])
    out["alpha"] = _np(alpha)
    out["colour"] = _np(col)
    occ = render_rays.occupancy_activation(alpha.squeeze(-1))
    term = render_rays.occupancy_to_termination(occ, is_batch=True)
    depth = render_rays.render(term, batch["z"])
    out["r_depth"] = _np(depth)
    out["r_var"] = _np(render_rays.render(term, (batch["z"] - depth[..., None]) ** 2))
    out["r_colour"] = _np(render_rays.render(term[..., None], col, dim=-2))
    out["r_opacity"] = _np(term.sum(-1))
    out["loss0"] = _np(l)
    l.backward()
    for n, p in zip(fc_names, fc_param):
        out["g0_" + n] = _np(p.grad)
    out["g0_" + vo.PE_KEY] = _np(pe_param[0].grad)
    losses = [float(l)]
    if n_steps:
        opt.step()
        opt.zero_grad(set_to_none=True)
        for n, p in zip(fc_names, fc_param):
            out["p1_" + n] = _np(p)
        out["p1_" + vo.PE_KEY] = _np(pe_param[0])
        for _ in range(n_steps - 1):
            _, _, _, l = fwd_loss()
            losses.append(float(l))
            l.backward()
            opt.step()
            opt.zero_grad(set_to_none=True)
        for n, p in zip(fc_names, fc_param):
            out[f"p{n_steps}_" + n] = _np(p)
        out[f"p{n_steps}_" + vo.PE_KEY] = _np(pe_param[0])
        _, _, _, l = fwd_loss()
        losses.append(float(l))
    out["losses"] = np.asarray(losses, dtype=np.float64)
    out["n_steps"] = np.int32(n_steps)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(name, "loss0", float(out["loss0"]), "losses", losses)


def reference_sampler_case(name, seed, n_kf, n_frames, n_samples, n1, W=64, H=48, KF=8):
    vmap_mod = _refload.load("vmap")
    g = torch.Generator().manual_seed(seed)
    rgbs = torch.randint(0, 256, (KF, W, H, 4), generator=g).to(torch.uint8)
    rgbs[..., 3] = (torch.rand(KF, W, H, generator=g) * 3).long().clamp(0, 2).to(torch.uint8)
    depth = torch.rand(KF, W, H, generator=g) * 4 + 0.5
    depth[torch.rand(KF, W, H, generator=g) < 0.15] = 0.0
    twc = torch.eye(4).repeat(KF, 1, 1)
    ang = torch.rand(KF, generator=g) * 0.6
    twc[:, 0, 0], twc[:, 0, 2] = torch.cos(ang), torch.sin(ang)
    twc[:, 2, 0], twc[:, 2, 2] = -torch.sin(ang), torch.cos(ang)
    twc[:, :3, 3] = torch.rand(KF, 3, generator=g) - 0.5
    bbox = torch.empty(KF, 4)
    bbox[:, 0] = torch.randint(0, W // 2, (KF,), generator=g).float()
    bbox[:, 1] = bbox[:, 0] + torch.randint(4, W // 2, (KF,), generator=g).float()
    bbox[:, 2] = torch.randint(0, H // 2, (KF,), generator=g).float()
    bbox[:, 3] = bbox[:, 2] + torch.randint(4, H // 2, (KF,), generator=g).float()
    rays = so.camera_ray_dirs(W, H, 60.0, 60.0, W / 2 - 0.5, H / 2 - 0.5)
    latest = [n_kf - 2, n_kf - 1] if n_kf >= 2 else [0]

    obj = object.__new__(vmap_mod.sceneObject)          # skip __init__ (builds a Trainer / open3d)
    obj.n_keyframes = n_kf
    obj.data_device = "cpu"
    obj.lastest_kf_queue = list(latest)
    obj.bbox, obj.rgbs_batch, obj.depth_batch, obj.t_wc_batch = bbox, rgbs, depth, twc
    obj.n_bins_cam2surface, obj.n_bins = n1, 9
    obj.surface_eps, obj.stop_eps = 0.1, 0.05
    obj.min_bound, obj.max_bound = 0.0, 8.0
    obj.this_obj, obj.other_obj, obj.unknown_obj = 1, 0, 2
    obj.obj_center = torch.tensor(0.0)
    torch.manual_seed(seed + 1)
    o_rgb, o_depth, o_valid, o_lab, o_pcs, o_z = obj.get_training_samples(n_frames, n_samples, rays)
    np.savez_compressed(
        os.path.join(OUT, name + ".npz"),
        rgbs_batch=_np(rgbs), depth_batch=_np(depth), t_wc_batch=_np(twc), bbox=_np(bbox), rays_dir=_np(rays),
        n_kf=np.int32(n_kf), latest=np.asarray(latest, dtype=np.int64), n_frames=np.int32(n_frames),
        n_samples=np.int32(n_samples), n1=np.int32(n1), seed=np.int64(seed + 1),
        o_rgb=_np(o_rgb), o_depth=_np(o_depth), o_valid=_np(o_valid), o_lab=_np(o_lab),
        o_pcs=_np(o_pcs), o_z=_np(o_z))
    print(name, "pcs", tuple(o_pcs.shape), "valid", int(o_valid.sum()))


def reference_config_case():
    """Attribute bag of the reference's Config for the two shipped Replica room0 files."""
    import json
    cfg_mod = _refload.load("cfg")
    out = {}
    for tag, rel in (("vMAP", "configs/Replica/config_replica_room0_vMAP.json"),
                     ("iMAP", "configs/Replica/config_replica_room0_iMAP.json")):
        path = os.path.join(_refload.REF_ROOT, rel)
        c = cfg_mod.Config(path)
        attrs = {k: (v.tolist() if hasattr(v, "tolist") else v) for k, v in vars(c).items()}
        out[tag] = {"raw": json.load(open(path)), "attrs": attrs}
    json.dump(out, open(os.path.join(OUT, "config_room0.json"), "w"), indent=1, sort_keys=True)
    print("config_room0", sorted(out["vMAP"]["attrs"])[:5], "...")


def reference_ingest_case(name, W, H, n_inst, seed, depth_scale=1000.0):
    """Run the reference's OWN data loader (dataset.Replica.__getitem__, dataset.py:80-141) on a synthetic
    Replica-format directory written under a scratch folder of this repo: the golden holds the instance /
    class images it read and the bbox_dict / relabelled instance image it returned."""
    import shutil
    import tempfile
    import types

    import cv2
    import numpy as np

    from oracle import ingest_oracle as io

    dataset = _refload.load("dataset")
    inst, cls = io.synthetic_instance_frame(W, H, n_inst, seed)
    root = tempfile.mkdtemp(prefix="_ds_", dir=os.path.dirname(os.path.abspath(__file__)))
    try:
        for d in ("rgb", "depth", "semantic_instance", "semantic_class"):
            os.makedirs(os.path.join(root, d))
        rng = np.random.default_rng(seed)
        # files are stored [H][W]; the loader transposes to [W][H] (dataset.py:87-91)
        cv2.imwrite(os.path.join(root, "rgb", "rgb_0.png"), rng.integers(0, 255, (H, W, 3), dtype=np.uint8))
        cv2.imwrite(os.path.join(root, "depth", "depth_0.png"), rng.integers(500, 4000, (H, W)).astype(np.uint16))
        cv2.imwrite(os.path.join(root, "semantic_instance", "semantic_instance_0.png"), inst.T.astype(np.uint16))
        cv2.imwrite(os.path.join(root, "semantic_class", "semantic_class_0.png"), cls.T.astype(np.uint16))
        np.savetxt(os.path.join(root, "traj_w_c.txt"), np.eye(4).reshape(1, 16), delimiter=" ")
        cfg = types.SimpleNamespace(imap_mode=False, dataset_dir=root, depth_scale=depth_scale, max_depth=8.0)
        ds = dataset.Replica(cfg)
        sample = ds[0]
        bbox_dict = {int(k): np.asarray(v).astype(np.int64) for k, v in sample["bbox_dict"].items()}
        obj = np.asarray(sample["obj"]).astype(np.int32)
        ids = np.array(sorted(bbox_dict), dtype=np.int64)
        np.savez_compressed(os.path.join(OUT, name + ".npz"), inst=inst.astype(np.int16), cls=cls.astype(np.int16),
                            background_cls=np.array(ds.background_cls_list, dtype=np.int64),
                            bbox_scale=np.float64(ds.bbox_scale), ids=ids,
                            bboxes=np.stack([bbox_dict[int(i)] for i in ids]), obj=obj.astype(np.int16))
        print(name, "instances in frame", len(np.unique(inst)), "kept", len(ids))
    finally:
        shutil.rmtree(root, ignore_errors=True)


def reference_enlarge_table():
    """utils.enlarge_bbox on every extent 1..1300 at the scales the repo ships / plausible ones: pins the
    float32 truncation of int(0.5*scale*extent) when the extent is a torch int64 scalar (dataset.py:121)."""
    import numpy as np
    import torch
    utils = _refload.load("utils")
    scales = [0.2, 0.1, 0.5, 1.0, 0.3, 1.5]
    ext = np.arange(1, 1301)
    margins = np.zeros((len(scales), ext.size), dtype=np.int64)
    for si, sc in enumerate(scales):
        for ei, e in enumerate(ext):
            # big canvas so clipping does not hide the margin; both axes share the extent
            r = utils.enlarge_bbox([torch.tensor(2000), torch.tensor(2000), torch.tensor(2000 + int(e)),
                                    torch.tensor(2000 + int(e))], scale=sc, w=10000, h=10000)
            margins[si, ei] = 0 if r is None else 2000 - r[0]
    np.savez_compressed(os.path.join(OUT, "ingest_enlarge_table.npz"), scales=np.array(scales), extents=ext,
                        margins=margins)
    print("ingest_enlarge_table", margins[:, [9, 10, 99, 1199]].tolist())


# ---- the sweep pinned by tests/test_oracle_live_reference.py ------------------------------------------------------
# Parameter lists are the tests' own; each case is keyed by its seed.
SWEEP_STEP = [(1, 32, 17, 6, 2.0, 1, 21), (5, 32, 9, 10, 2.0, 1, 22), (2, 64, 13, 14, 5.0, 5, 23),
              (1, 128, 8, 10, 5.0, 5, 24), (3, 32, 1, 10, 2.0, 1, 25)]
SWEEP_SAMPLER = [(31, 7, 9, 11, 1), (32, 3, 6, 5, 5), (33, 1, 4, 7, 1), (34, 8, 20, 3, 1), (35, 4, 5, 16, 5)]
SWEEP_KEYFRAMES = [(3, 6, 40, 1), (1, 4, 25, 2), (5, 8, 60, 3)]
SWEEP_INGEST = [(96, 64, 9, 41), (200, 150, 25, 42), (64, 96, 5, 43)]
SWEEP_SAMPLE = 128          # stored elements per gradient / parameter tensor (a fixed, seeded sample)
SWEEP_STEPS = 2


def sweep_step_case(n_obj, hidden, n_rays, n_samples, scale, n1, seed, n_steps=SWEEP_STEPS):
    """The reference's functorch step (train.py:293-326) from ``vo.init_params(n_obj, hidden, seed=seed)``: loss and
    gradients of the first step, the losses of ``n_steps`` AdamW steps and the parameters after them.  Gradients and
    final parameters are stored as a seeded sample of elements plus the full tensor's norm, concatenated over
    ``vo.ALL_KEYS`` (``count`` elements per tensor, flat indices ``idx`` into its [n_obj, *shape] stack)."""
    model, embedding, loss = _refload.load("model", "embedding", "loss")
    from functorch import combine_state_for_ensemble, vmap
    e1, e2 = vo.emb_sizes(5)
    fcs = [model.OccupancyMap(e1, e2, hidden_size=hidden) for _ in range(n_obj)]
    pes = [embedding.UniDirsEmbed(max_deg=5, scale=scale) for _ in range(n_obj)]
    init = vo.init_params(n_obj, hidden, seed=seed)
    batch = vo.synthetic_batch(n_obj, n_rays, n_samples, seed=seed + 100, n_cam2surf=n1)
    opt = torch.optim.AdamW([torch.zeros(1, requires_grad=True)], lr=1e-3, weight_decay=0.013)        # train.py:67
    fc_model, fc_param, fc_buffer = combine_state_for_ensemble(fcs)                                    # utils.py:31
    pe_model, pe_param, pe_buffer = combine_state_for_ensemble(pes)
    names = [n for n, _ in fcs[0].named_parameters()]
    assert tuple(names) == vo.FC_KEYS, names
    with torch.no_grad():
        for n, p in zip(names, fc_param):
            p.copy_(init[n])
        pe_param[0].copy_(init[vo.PE_KEY])
    for p in list(fc_param) + list(pe_param):
        p.requires_grad_()
    opt.add_param_group({"params": fc_param}); opt.add_param_group({"params": pe_param})
    tensors = dict(zip(names, fc_param), **{vo.PE_KEY: pe_param[0]})

    def fwd_loss():
        emb = vmap(pe_model)(pe_param, pe_buffer, batch["pcs"])                                        # train.py:293
        alpha, col = vmap(fc_model)(fc_param, fc_buffer, emb)                                          # train.py:294
        return loss.step_batch_loss(alpha, col, batch["gt_depth"], batch["gt_colour"], batch["sem"],
                                    batch["mask_depth"], batch["z"])[0]                                # train.py:303
    l0 = fwd_loss()
    l0.backward()
    grads = {k: t.grad.detach().clone() for k, t in tensors.items()}
    losses = [float(l0)]
    for s in range(n_steps):
        opt.step(); opt.zero_grad(set_to_none=True)
        l = fwd_loss(); losses.append(float(l))
        if s + 1 < n_steps:
            l.backward()
    out = {"losses": np.asarray(losses, dtype=np.float64)}
    for k, v in batch.items():
        out["in_" + k] = _np(v)
    rng = np.random.default_rng(seed)
    cols = {"count": [], "idx": [], "g": [], "p": [], "norms": [], "init_sum": []}
    for k in vo.ALL_KEYS:
        g, p = grads[k].reshape(-1), tensors[k].detach().reshape(-1)
        idx = np.arange(g.numel()) if g.numel() <= SWEEP_SAMPLE else np.sort(rng.choice(g.numel(), SWEEP_SAMPLE, replace=False))
        cols["count"].append(idx.size); cols["idx"].append(idx)
        cols["g"].append(_np(g[idx])); cols["p"].append(_np(p[idx]))
        cols["norms"].append([float(g.double().norm()), float(p.double().norm())])
        cols["init_sum"].append(float(init[k].double().sum()))
    out["count"] = np.asarray(cols["count"], dtype=np.int32)
    out["idx"] = np.concatenate(cols["idx"]).astype(np.int32)
    out["g"], out["p"] = np.concatenate(cols["g"]), np.concatenate(cols["p"])
    out["norms"], out["init_sum"] = np.asarray(cols["norms"]), np.asarray(cols["init_sum"])
    return out


def sweep_sampler_inputs(seed, W=56, H=40, KF=8):
    """Keyframe buffers of one sampler case, drawn from ``seed`` (rgbs, depth, t_wc, bbox, rays_dir)."""
    g = torch.Generator().manual_seed(seed)
    rgbs = torch.randint(0, 256, (KF, W, H, 4), generator=g).to(torch.uint8)
    rgbs[..., 3] = (torch.rand(KF, W, H, generator=g) * 3).long().clamp(0, 2).to(torch.uint8)
    depth = torch.rand(KF, W, H, generator=g) * 4 + 0.5
    depth[torch.rand(KF, W, H, generator=g) < 0.15] = 0.0
    twc = torch.eye(4).repeat(KF, 1, 1)
    twc[:, :3, 3] = torch.rand(KF, 3, generator=g) - 0.5
    bbox = torch.empty(KF, 4)
    bbox[:, 0] = torch.randint(0, W // 2, (KF,), generator=g).float()
    bbox[:, 1] = bbox[:, 0] + torch.randint(4, W // 2, (KF,), generator=g).float()
    bbox[:, 2] = torch.randint(0, H // 2, (KF,), generator=g).float()
    bbox[:, 3] = bbox[:, 2] + torch.randint(4, H // 2, (KF,), generator=g).float()
    return rgbs, depth, twc, bbox, so.camera_ray_dirs(W, H, 60.0, 60.0, W / 2 - 0.5, H / 2 - 0.5)


def sweep_sampler_case(seed, n_kf, n_frames, n_samples, n1):
    """sceneObject.get_training_samples (vmap.py:319-459) on ``sweep_sampler_inputs(seed)`` after
    ``torch.manual_seed(seed + 1)``."""
    vmap_mod = _refload.load("vmap")
    rgbs, depth, twc, bbox, rays = sweep_sampler_inputs(seed)
    obj = object.__new__(vmap_mod.sceneObject)          # skip __init__ (builds a Trainer / open3d)
    obj.n_keyframes, obj.data_device = n_kf, "cpu"
    obj.lastest_kf_queue = [n_kf - 2, n_kf - 1] if n_kf >= 2 else [0]
    obj.bbox, obj.rgbs_batch, obj.depth_batch, obj.t_wc_batch = bbox, rgbs, depth, twc
    obj.n_bins_cam2surface, obj.n_bins, obj.surface_eps, obj.stop_eps = n1, 9, 0.1, 0.05
    obj.min_bound, obj.max_bound = 0.0, 8.0
    obj.this_obj, obj.other_obj, obj.unknown_obj = 1, 0, 2
    obj.obj_center = torch.tensor(0.0)
    torch.manual_seed(seed + 1)
    res = obj.get_training_samples(n_frames, n_samples, rays)
    out = {k: _np(v) for k, v in zip(("rgb", "depth", "valid", "lab", "pcs", "z"), res)}
    out["inputs_sum"] = np.asarray([float(rgbs.double().sum()), float(depth.double().sum()),
                                    float(twc.double().sum()), float(bbox.double().sum())])
    return out


def sweep_keyframe_frame(seed, fid, W=6, H=5):
    g = torch.Generator().manual_seed(1000 * seed + fid)
    return (torch.randint(0, 255, (W, H, 3), dtype=torch.uint8, generator=g), torch.rand(W, H, generator=g),
            torch.randint(0, 3, (W, H), dtype=torch.uint8, generator=g), torch.tensor([0., float(fid % W), 0., float(fid % H)]),
            torch.eye(4) * (fid + 1))


def sweep_keyframe_case(kf_step, buf, n_frames_seen, seed, W=6, H=5):
    """sceneObject.append_keyframe / prune_keyframe (vmap.py:208-268) fed ``sweep_keyframe_frame(seed, fid)`` for
    fid = 1 .. n_frames_seen - 1 with ``random.seed(fid)`` before each: the bookkeeping after every frame, and for each
    buffer slot in use the id of the frame whose rgb / mask / depth / pose / bbox it holds."""
    import random
    ref_mod = _refload.load("vmap")
    frames = [sweep_keyframe_frame(seed, fid, W, H) for fid in range(n_frames_seen)]
    rgb, depth, mask, bbox, T = frames[0]
    ref = object.__new__(ref_mod.sceneObject)               # the reference __init__ builds a Trainer / needs open3d
    ref.n_keyframes, ref.kf_pointer, ref.keyframe_buffer_size = 1, None, buf
    ref.kf_id_dict, ref.kf_buffer_full, ref.frame_cnt, ref.lastest_kf_queue = _refload._Bidict({0: 0}), False, 0, []
    ref.keyframe_step, ref.rgb_idx, ref.state_idx = kf_step, slice(0, 3), slice(3, 4)
    ref.bbox = torch.empty(buf, 4); ref.rgbs_batch = torch.empty(buf, W, H, 4, dtype=torch.uint8)
    ref.depth_batch = torch.empty(buf, W, H); ref.t_wc_batch = torch.empty(buf, 4, 4)
    ref.bbox[0] = bbox; ref.rgbs_batch[0, :, :, :3] = rgb; ref.rgbs_batch[0, :, :, 3:4] = mask[..., None]
    ref.depth_batch[0] = depth; ref.t_wc_batch[0] = T

    def holds(k, f):
        rgb, depth, mask, bbox, T = f
        return (torch.equal(ref.rgbs_batch[k, :, :, :3], rgb) and torch.equal(ref.rgbs_batch[k, :, :, 3], mask)
                and torch.equal(ref.depth_batch[k], depth) and torch.equal(ref.t_wc_batch[k], T)
                and torch.equal(ref.bbox[k], bbox))
    states = []
    for fid in range(1, n_frames_seen):
        random.seed(fid); ref.append_keyframe(*frames[fid], fid)
        n = max(ref.n_keyframes, (ref.kf_pointer or 0) + 1)
        slots = [next(f for f in range(fid + 1) if holds(k, frames[f])) for k in range(n)]
        states.append({"n_keyframes": ref.n_keyframes, "kf_pointer": ref.kf_pointer,
                       "lastest_kf_queue": list(ref.lastest_kf_queue), "frame_cnt": ref.frame_cnt,
                       "kf_id_dict": sorted([int(a), int(b)] for a, b in dict(ref.kf_id_dict).items()),
                       "kf_buffer_full": bool(ref.kf_buffer_full), "slot_frames": slots})
    return states


def sweep_module_surface():
    """state_dict keys / shapes of OccupancyMap (hidden 32, 128, 256) and UniDirsEmbed, the embedding's direction
    table and scale, and cameraInfo's ray cache (model.py:17-52, embedding.py:44-80, vmap.py:494-524)."""
    import json
    import types
    ref_model, ref_emb, ref_vmap = _refload.load("model", "embedding", "vmap")
    surf = {f"occupancy_h{h}": [[k, list(v.shape)] for k, v in ref_model.OccupancyMap(87, 42, hidden_size=h).state_dict().items()]
            for h in (32, 128, 256)}
    pe = ref_emb.UniDirsEmbed(max_deg=5, scale=2.0)
    surf["unidirs"] = list(pe.state_dict())
    json.dump(surf, open(os.path.join(OUT, "sweep_module_surface.json"), "w"), indent=1)
    cfg = types.SimpleNamespace(data_device="cpu", W=37, H=23, fx=31.5, fy=29.25, cx=18.0, cy=11.5)
    np.savez_compressed(os.path.join(OUT, "sweep_module_surface.npz"), b_layer=_np(pe.B_layer.weight),
                        scale=np.float32(float(pe.scale)), rays_dir_cache=_np(ref_vmap.cameraInfo(cfg).rays_dir_cache))


def sweep():
    """tests/golden/sweep_*: what the reference computes for every case of tests/test_oracle_live_reference.py."""
    import json
    steps = {}
    for case in SWEEP_STEP:
        steps.update({f"s{case[-1]}_{k}": v for k, v in sweep_step_case(*case).items()})
    np.savez_compressed(os.path.join(OUT, "sweep_step.npz"), **steps)
    samples = {}
    for case in SWEEP_SAMPLER:
        samples.update({f"s{case[0]}_{k}": v for k, v in sweep_sampler_case(*case).items()})
    np.savez_compressed(os.path.join(OUT, "sweep_sampler.npz"), **samples)
    kf = {f"s{case[-1]}": sweep_keyframe_case(*case) for case in SWEEP_KEYFRAMES}
    json.dump(kf, open(os.path.join(OUT, "sweep_keyframes.json"), "w"), separators=(",", ":"))
    sweep_module_surface()
    for W, H, n_inst, seed in SWEEP_INGEST:
        reference_ingest_case(f"sweep_ingest_s{seed}", W=W, H=H, n_inst=n_inst, seed=seed)


def main():
    os.makedirs(OUT, exist_ok=True)
    sweep()
    reference_ingest_case("ingest_small", W=160, H=120, n_inst=14, seed=21)
    reference_ingest_case("ingest_replica_size", W=1200, H=680, n_inst=40, seed=22)
    reference_enlarge_table()
    reference_config_case()
    # vMAP object ensemble (room0_vMAP.json: H=32, scale 2, 1+9 samples), 3 AdamW steps
    reference_step_case("step_vmap_h32", n_obj=3, hidden=32, n_rays=24, n_samples=10, scale=2.0,
                        n_cam2surf=1, seed=1, n_steps=3)
    # background model shape (H=128, scale 5, 5+9 samples) as a 1-object ensemble
    reference_step_case("step_bg_h128", n_obj=1, hidden=128, n_rays=16, n_samples=14, scale=5.0,
                        n_cam2surf=5, seed=2, n_steps=0)
    # any-empty-mask early-out (render_rays.py:68-73): object 1 has no valid depth
    reference_step_case("step_emptymask_h32", n_obj=2, hidden=32, n_rays=12, n_samples=10, scale=2.0,
                        n_cam2surf=1, seed=3, n_steps=1, kill_depth_obj=1)
    reference_sampler_case("sampler_obj", seed=10, n_kf=6, n_frames=12, n_samples=8, n1=1)
    reference_sampler_case("sampler_bg", seed=11, n_kf=5, n_frames=10, n_samples=6, n1=5)
    reference_sampler_case("sampler_2kf", seed=12, n_kf=2, n_frames=6, n_samples=8, n1=1)


if __name__ == "__main__":
    main()
