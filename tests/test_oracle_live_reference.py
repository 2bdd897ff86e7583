"""Oracle vs the UNMODIFIED reference modules over a sweep of shapes / seeds.  What the reference computed for every
case -- through the same harness train.py uses (functorch vmap over combine_state_for_ensemble, loss.step_batch_loss,
torch.optim.AdamW), its sampler, keyframe policy, module classes and data loader -- is stored in tests/golden/sweep_*
(``oracle/make_golden.py`` regenerates it); the inputs are rebuilt here from the same seeds and checked against
fingerprints of the ones the reference was given."""
import json
import os
import types

import numpy as np
import pytest
import torch

from oracle import make_golden as mg
from oracle import vmap_oracle as vo
from tests._util import GOLDEN, rel_l2


def _golden(name):
    return np.load(os.path.join(GOLDEN, name))


@pytest.mark.parametrize("n_obj,hidden,n_rays,n_samples,scale,n1,seed", [
    (1, 32, 17, 6, 2.0, 1, 21), (5, 32, 9, 10, 2.0, 1, 22), (2, 64, 13, 14, 5.0, 5, 23), (1, 128, 8, 10, 5.0, 5, 24),
    (3, 32, 1, 10, 2.0, 1, 25)])
def test_oracle_matches_live_reference_step(n_obj, hidden, n_rays, n_samples, scale, n1, seed):
    """Gradients of the first step and parameters after two AdamW steps: relative L2 error over a fixed sample of
    elements of every tensor, and the whole tensor's norm, within the same bounds."""
    g = _golden("sweep_step.npz")
    ref = {k[len(f"s{seed}_"):]: g[k] for k in g.files if k.startswith(f"s{seed}_")}
    n_steps, l_ref = mg.SWEEP_STEPS, ref["losses"].tolist()
    init = vo.init_params(n_obj, hidden, seed=seed)
    np.testing.assert_allclose([float(init[k].double().sum()) for k in vo.ALL_KEYS], ref["init_sum"], rtol=1e-12,
                               err_msg="vo.init_params no longer draws the parameters the reference started from")
    batch = {k: torch.from_numpy(ref["in_" + k]) for k in ("pcs", "z", "gt_depth", "gt_colour", "sem", "mask_depth")}
    ends = np.cumsum(ref["count"])

    def check(mine, col, tol):
        for i, k in enumerate(vo.ALL_KEYS):
            sl = slice(ends[i] - ref["count"][i], ends[i])
            flat = mine[k].detach().reshape(-1)
            assert rel_l2(flat[torch.from_numpy(ref["idx"][sl]).long()], ref[col][sl]) < tol, k
            n_ref = ref["norms"][i, 0 if col == "g" else 1]
            assert abs(float(flat.double().norm()) - n_ref) <= tol * n_ref, k

    orc = vo.OracleEnsemble(init, scale)
    loss, grads = orc.grads(batch)
    assert abs(float(loss) - l_ref[0]) <= 2e-6 * abs(l_ref[0]) + 1e-7
    check(grads, "g", 2e-5)
    orc = vo.OracleEnsemble(init, scale)            # fresh optimiser state / no leftover .grad
    losses = [float(orc.step(batch)) for _ in range(n_steps)]
    for a, b in zip(losses, l_ref[:n_steps]):
        assert abs(a - b) <= 5e-6 * abs(b) + 1e-7
    check(orc.params, "p", 2e-6)


@pytest.mark.parametrize("seed,n_kf,n_frames,n_samples,n1", [(31, 7, 9, 11, 1), (32, 3, 6, 5, 5), (33, 1, 4, 7, 1),
                                                             (34, 8, 20, 3, 1), (35, 4, 5, 16, 5)])
def test_sampler_oracle_matches_live_reference(seed, n_kf, n_frames, n_samples, n1):
    """sceneObject.get_training_samples (vmap.py:319-459) vs oracle/sampler_oracle.py with the reference's RNG
    call order reproduced: integer outputs and z bit-exact."""
    from oracle import sampler_oracle as so
    g = _golden("sweep_sampler.npz")
    ref = {k[len(f"s{seed}_"):]: g[k] for k in g.files if k.startswith(f"s{seed}_")}
    rgbs, depth, twc, bbox, rays = mg.sweep_sampler_inputs(seed)
    np.testing.assert_allclose([float(t.double().sum()) for t in (rgbs, depth, twc, bbox)], ref["inputs_sum"],
                               rtol=1e-12, err_msg="the sampler inputs differ from the ones the reference was given")
    latest = [n_kf - 2, n_kf - 1] if n_kf >= 2 else [0]
    cfg = so.SamplerCfg(n_bins_cam2surface=n1)
    torch.manual_seed(seed + 1)
    rnd = so.draw_randoms_reference_order(None, n_kf, latest, n_frames, n_samples, bbox, rgbs, depth, cfg)
    rgb, dep, valid, lab, pcs, z = so.sample_from_randoms(rnd, rgbs, depth, twc, bbox, rays, cfg)
    for name, t in (("rgb", rgb), ("depth", dep), ("valid", valid), ("lab", lab), ("z", z)):
        assert np.array_equal(t.numpy(), ref[name]) and t.dtype == torch.from_numpy(ref[name]).dtype, name
    np.testing.assert_allclose(pcs.numpy(), ref["pcs"], rtol=0, atol=1e-6)


@pytest.mark.parametrize("kf_step,buf,n_frames_seen,seed", [(3, 6, 40, 1), (1, 4, 25, 2), (5, 8, 60, 3)])
def test_keyframe_policy_matches_live_reference(kf_step, buf, n_frames_seen, seed, monkeypatch):
    """vmap_b200.vmap.sceneObject.append_keyframe / prune_keyframe vs the reference's (vmap.py:208-268), fed the same
    frames and the same ``random`` stream: slot choice, keyframe count, latest queue, id map and buffer contents."""
    import random
    from vmap_b200 import vmap as vm
    states = json.load(open(os.path.join(GOLDEN, "sweep_keyframes.json")))[f"s{seed}"]
    assert len(states) == n_frames_seen - 1
    monkeypatch.setattr(vm.trainer_mod, "Trainer", lambda cfg: types.SimpleNamespace())
    cfg = types.SimpleNamespace(do_bg=False, data_device="cpu", training_device="cpu", obj_scale=2.0, bg_scale=5.0,
                                hidden_feature_size=32, hidden_feature_size_bg=128, n_bins_cam2surface=1,
                                n_bins_cam2surface_bg=5, keyframe_step=kf_step, keyframe_step_bg=kf_step, min_depth=0.0,
                                max_depth=8.0, n_bins=9, n_unidir_funcs=5, surface_eps=0.1, stop_eps=0.05,
                                keyframe_buffer_size=buf)
    frames = [mg.sweep_keyframe_frame(seed, fid) for fid in range(n_frames_seen)]
    mine = vm.sceneObject(cfg, 7, *frames[0], 0)
    for fid, ref in zip(range(1, n_frames_seen), states):
        random.seed(fid); mine.append_keyframe(*frames[fid], fid)
        assert mine.n_keyframes == ref["n_keyframes"] and mine.kf_pointer == ref["kf_pointer"], fid
        assert mine.lastest_kf_queue == ref["lastest_kf_queue"] and mine.frame_cnt == ref["frame_cnt"]
        assert sorted([a, b] for a, b in dict(mine.kf_id_dict).items()) == ref["kf_id_dict"]
        assert mine.kf_buffer_full == ref["kf_buffer_full"]
        assert max(mine.n_keyframes, (mine.kf_pointer or 0) + 1) == len(ref["slot_frames"])
        for k, f in enumerate(ref["slot_frames"]):
            rgb, depth, mask, bbox, T = frames[f]
            assert torch.equal(mine.rgbs_batch[k, :, :, :3], rgb) and torch.equal(mine.rgbs_batch[k, :, :, 3], mask), (fid, k)
            assert torch.equal(mine.depth_batch[k], depth) and torch.equal(mine.t_wc_batch[k], T), (fid, k)
            assert torch.equal(mine.bbox[k], bbox), (fid, k)


def test_module_surface_matches_live_reference():
    """state_dict keys / shapes of OccupancyMap and UniDirsEmbed, the icosahedron directions, and cameraInfo's ray cache
    against the reference classes (model.py:17-52, embedding.py:44-80, vmap.py:494-524)."""
    from vmap_b200 import embedding as my_emb, model as my_model, vmap as my_vmap
    surf = json.load(open(os.path.join(GOLDEN, "sweep_module_surface.json")))
    arr = _golden("sweep_module_surface.npz")
    for hidden in (32, 128, 256):
        a = my_model.OccupancyMap(87, 42, hidden_size=hidden).state_dict()
        assert [[k, list(v.shape)] for k, v in a.items()] == surf[f"occupancy_h{hidden}"]
    pa = my_emb.UniDirsEmbed(max_deg=5, scale=2.0)
    assert list(pa.state_dict()) == surf["unidirs"]
    assert np.array_equal(pa.B_layer.weight.detach().numpy(), arr["b_layer"]) and float(pa.scale) == float(arr["scale"])
    cfg = types.SimpleNamespace(data_device="cpu", W=37, H=23, fx=31.5, fy=29.25, cx=18.0, cy=11.5)
    assert np.array_equal(my_vmap.cameraInfo(cfg).rays_dir_cache.numpy(), arr["rays_dir_cache"])


@pytest.mark.parametrize("W,H,n_inst,seed", [(96, 64, 9, 41), (200, 150, 25, 42), (64, 96, 5, 43)])
def test_ingest_oracle_matches_live_reference_loader(W, H, n_inst, seed):
    """oracle/ingest_oracle.replica_frame vs dataset.Replica.__getitem__ (dataset.py:80-141), which read the instance /
    class images of ``synthetic_instance_frame(W, H, n_inst, seed)`` from a Replica-format directory."""
    from oracle import ingest_oracle as io
    g = _golden(f"sweep_ingest_s{seed}.npz")
    inst, cls = io.synthetic_instance_frame(W, H, n_inst, seed)
    assert np.array_equal(inst, g["inst"]) and np.array_equal(cls, g["cls"])
    bbox_dict, obj = io.replica_frame(inst, cls, set(g["background_cls"].tolist()), float(g["bbox_scale"]))
    assert {k: v.tolist() for k, v in bbox_dict.items()} == dict(zip(g["ids"].tolist(), g["bboxes"].tolist()))
    assert np.array_equal(obj, g["obj"].astype(np.int32))
