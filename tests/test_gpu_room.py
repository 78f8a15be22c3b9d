"""Room driver (configs[4]): sharding over ranks renders every window exactly once, and a window rendered inside a
multi-window launch equals the same window rendered alone."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def test_room_shards_cover_all_windows_and_batches_are_independent(cuda_device):
    from spsg_b200 import room as R, synthetic as S
    dims = (64, 96, 128)
    room = R.synthetic_room_sdf(dims, cuda_device, seed=5)
    predict = R.synthetic_predictor(room)
    kw = dict(views_per_chunk=2, width=96, height=64, max_num_locs_per_sample=200000, keep_images=True)
    whole = R.render_room(predict, dims, cuda_device, chunks_per_launch=4, **kw)
    assert whole["windows"] == 3 * 4 and whole["rendered_windows"] > 0
    assert whole["label_hist"].sum() == whole["rays"]
    # two "ranks" run one after the other on this GPU: together they render what one rank renders
    parts = [R.render_room(predict, dims, cuda_device, chunks_per_launch=3, rank=r, world=2, **kw) for r in range(2)]
    assert parts[0]["rendered_windows"] + parts[1]["rendered_windows"] == whole["rendered_windows"]
    np.testing.assert_array_equal(parts[0]["label_hist"] + parts[1]["label_hist"], whole["label_hist"])
    got = {w: img for p in parts for (w, img) in p["images"]}
    for w, img in whole["images"]:
        assert torch.equal(got[w], img), "window %s differs between launch groupings" % (w,)
    # something was actually hit and labelled
    assert whole["label_hist"][:S.NUM_CLASSES].sum() > 0.1 * whole["rays"]


def test_room_windows_match_looped_reference_calls(cuda_device):
    """Every window / view label image of the room driver against the compiled reference extension: the window's voxels
    from the literal `torch.nonzero` sparsification, one reference call per view (the reference renders one view per chunk
    and call), labels by the literal argmax(cat(render, ones)) of train.py:749-752."""
    from oracle import ref_driver
    from spsg_b200 import room as R, synthetic as S
    if not ref_driver.available(pinned=True):
        pytest.skip("oracle/_ref not built (run __graft_entry__.build() where /root/reference exists)")
    dims, F, w, h = (64, 96, 128), 3, 96, 64
    room = R.synthetic_room_sdf(dims, cuda_device, seed=3)
    predict = R.synthetic_predictor(room)
    got = R.render_room(predict, dims, cuda_device, views_per_chunk=F, chunks_per_launch=4, width=w, height=h,
                        max_num_locs_per_sample=200000, keep_images=True)
    chunk_dims = (dims[0], 64, 64)
    view_np, intr_np = R.window_views(F, chunk_dims)
    view = torch.from_numpy(view_np).to(cuda_device)
    intr = torch.from_numpy(intr_np).to(cuda_device)
    ref = ref_driver.RefRaycaster(1, chunk_dims, w, h, S.DEPTH_MIN, S.DEPTH_MAX, S.THRESH_SAMPLE_DIST, S.RAY_INCREMENT,
                                  200000, 64, device=cuda_device, pinned=True)
    hist = np.zeros(S.NUM_CLASSES + 1)
    images = dict(got["images"])
    assert len(images) == got["rendered_windows"] > 6
    for (y0, x0), labels in images.items():
        locs3, sdf, color, sem = predict(y0, x0, (64, 64))
        locs = torch.cat([locs3, torch.zeros(locs3.shape[0], 1, dtype=torch.long, device=cuda_device)], 1).contiguous()
        normal = torch.zeros(locs.shape[0], 3, device=cuda_device)  # the semantic rendering does not depend on the normals
        for f in range(F):
            _, _, _, r_sem = ref.forward(locs, sdf, color, normal, sem, view[f:f + 1].contiguous(), intr[f:f + 1].contiguous())
            cat = torch.cat((r_sem, torch.ones(r_sem.shape[:-1] + (1,), device=cuda_device)), dim=-1)
            want = torch.max(cat, dim=-1)[1].to(torch.uint8)[0].cpu()
            assert torch.equal(labels[f], want), "window %s view %d: %d label pixels differ" % (
                (y0, x0), f, int((labels[f] != want).sum()))
            hist += np.bincount(want.reshape(-1).numpy(), minlength=S.NUM_CLASSES + 1)
    np.testing.assert_array_equal(hist, got["label_hist"])
