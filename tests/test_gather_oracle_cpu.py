"""The float64 gather oracle (tests/gather_oracle.py) on hand-built renderings and tables: no GPU needed."""
import numpy as np
import pytest
import torch

from tests import gather_oracle as O

NINF = -np.inf


def _scene():
    """One image 2 x 4 of three voxels (ids in the normal payload), one miss; voxel 3 is never hit."""
    n = 4
    rng = np.random.default_rng(0)
    vals_color = rng.random((n, 3), dtype=np.float32)
    vals_sem = rng.standard_normal((n, 14)).astype(np.float32)
    nrm = O.voxel_normals(n)
    vox = np.array([[0, 0, 1, -1], [2, 0, 1, 1]])
    hit = vox >= 0
    color = np.where(hit[..., None], vals_color[np.maximum(vox, 0)], NINF).astype(np.float32)[None]
    normal = np.where(hit[..., None], nrm[np.maximum(vox, 0)], NINF).astype(np.float32)[None]
    sem = np.where(hit[..., None], vals_sem[np.maximum(vox, 0)], NINF).astype(np.float32)[None]
    depth = np.where(hit, 3.0, NINF).astype(np.float32)[None]
    return n, vals_color, vals_sem, color, depth, normal, sem, vox


def test_pixel_map_from_payload_ids():
    n, vals_color, vals_sem, color, depth, normal, sem, vox = _scene()
    got = O.pixel_map(color, depth, normal, sem, vals_color, vals_sem)
    assert np.array_equal(got, vox.reshape(1, -1))
    bad = color.copy()
    bad[0, 1, 2, 0] = np.nextafter(bad[0, 1, 2, 0], np.float32(2))
    with pytest.raises(AssertionError, match="colour"):
        O.pixel_map(bad, depth, normal, sem, vals_color, vals_sem)
    bad = sem.copy()
    bad[0, 0, 3, 5] = 0.0  # a miss with a finite value
    with pytest.raises(AssertionError, match="miss"):
        O.pixel_map(color, depth, normal, bad, vals_color, vals_sem)


def _tables(max_pix=4, num=None, mapping=None):
    n, vals_color, vals_sem, color, depth, normal, sem, _ = _scene()
    vox = O.pixel_map(color, depth, normal, sem, vals_color, vals_sem)
    if num is None:
        num = np.array([3, 3, 1, 0], np.int32)
    if mapping is None:
        mapping = np.full((n, max_pix), -7, np.int32)
        mapping[0, :3] = [5, 0, 1][:max_pix]
        mapping[1, :3] = [7, 2, 6][:max_pix]
        mapping[2, :1] = [4]
    return O.check_tables(vox, mapping, num, np.zeros(n, np.int64), 1), n


def test_tables_counts_and_entries():
    tab, n = _tables()
    assert list(tab.cnt) == [3, 3, 1, 0] and tab.overflow.size == 0
    with pytest.raises(AssertionError, match="mapping3dto2d_num"):
        _tables(num=np.array([3, 2, 1, 0], np.int32))
    m = np.full((n, 4), -7, np.int32)
    m[0, :3], m[1, :3], m[2, 0] = [5, 0, 0], [7, 2, 6], 4
    with pytest.raises(AssertionError, match="twice"):
        _tables(mapping=m)
    m[0, :3] = [5, 0, 2]  # pixel 2 belongs to voxel 1
    with pytest.raises(AssertionError, match="another voxel"):
        _tables(mapping=m)


def test_overflowing_voxel_averages_the_table_subset():
    tab, n = _tables(max_pix=2)
    assert list(tab.cnt) == [2, 2, 1, 0] and list(tab.overflow) == [0, 1]
    G = np.zeros((8, 21))
    G[:, 17] = np.arange(8) * 10.0
    g = O.gather(tab, G)
    assert g.want[0, 17] == (50 + 0) / 2 and g.want[1, 17] == (70 + 20) / 2 and g.want[2, 17] == 40
    assert g.want[3].tolist() == [0.0] * 21 and g.bound[3].tolist() == [0.0] * 21


def test_known_means_and_mutations_fail():
    tab, n = _tables()
    rng = np.random.default_rng(3)
    G = (rng.choice([-1, 1], (8, 21)) * 10.0 ** rng.uniform(-6, 3, (8, 21))).astype(np.float32).astype(np.float64)
    g = O.gather(tab, G)
    want0 = (G[5] + G[0] + G[1]) / 3
    np.testing.assert_allclose(g.want[0], want0, rtol=1e-15)
    exact = g.want.astype(np.float32)
    O.compare(exact, g, "exact")
    # mean with the normaliser off by one, and a dropped pixel: outside the bound
    wrong = exact.copy()
    wrong[0] = (want0 * 3 / 4).astype(np.float32)
    with pytest.raises(AssertionError, match="outside their bound"):
        O.compare(wrong, g, "cnt+1")
    wrong = exact.copy()
    wrong[1] = ((G[7] + G[2]) / 3).astype(np.float32)
    with pytest.raises(AssertionError, match="outside their bound"):
        O.compare(wrong, g, "dropped")
    wrong = exact.copy()
    wrong[3, 4] = np.float32(1e-30)  # a row nothing hit must be exactly 0
    with pytest.raises(AssertionError):
        O.compare(wrong, g, "unhit")
    wrong = exact.copy()
    wrong[2, 0] = np.nan
    with pytest.raises(AssertionError, match="NaN"):
        O.compare(wrong, g, "nan")
    assert bool((g.bound <= 1e-5 * g.mag + 1e-40).all())


def test_near_tie_detection():
    one = np.float32(1.0)
    mid = (1.0 + float(np.nextafter(one, np.float32(2)))) / 2
    x = np.array([mid, mid + 2.0 ** -60, 1.0, 1.0 + 2.0 ** -26, mid - 2.0 ** -40])
    tie = O.near_tie(x, np.full(5, 2.0 ** -50))
    assert tie.tolist() == [True, True, False, False, False]


def test_deterministic_emulation_is_sequential_fp32():
    """Two views of one voxel: the fp32 emulation adds the per-view means in view order."""
    n = 1
    vox = np.array([[0, 0, 0], [0, -1, -1]])
    mapping = np.array([[0, 1, 2], [0, -1, -1]], np.int32)
    tab = O.check_tables(vox, mapping, np.array([3, 1], np.int32), np.zeros(n, np.int64), 2)
    G = np.zeros((6, 21))
    G[:3, 0] = [1.0, 1.0, 2.0 ** -30]
    G[3, 0] = 2.0 ** -25
    g = O.gather(tab, G, deterministic=True)
    y0 = np.float32((1.0 + 1.0 + 2.0 ** -30) * float(np.float32(1.0 / 3)))
    assert g.exact[0, 0] == np.float32(y0 + np.float32(2.0 ** -25))
    assert g.exact[0, 1] == 0.0 and not g.ties[0, 1]


def test_fused_grads_match_autograd_of_literal_losses():
    """fused_pixel_grads against torch autograd (float64) of oracle/losses_ref.py, on renderings without ties."""
    from oracle import losses_ref as R
    rng = np.random.default_rng(7)
    I, H, W = 2, 5, 6
    hit = rng.random((I, H, W)) < 0.7
    depth = np.where(hit, rng.uniform(10, 60, (I, H, W)), NINF).astype(np.float32)
    color = np.where(hit[..., None], rng.random((I, H, W, 3)), NINF).astype(np.float32)
    sem = np.where(hit[..., None], rng.standard_normal((I, H, W, 14)) * 30, NINF).astype(np.float32)
    td = (rng.random((I, 1, H, W)) * 1.2).astype(np.float32)
    td[rng.random(td.shape) < 0.2] = 0.0
    tc = rng.random((I, H, W, 3)).astype(np.float32)
    wc = (rng.random((I, 1, H, W)) + 0.5).astype(np.float32)
    wc[0, 0, 0, :3] = 0.0
    label = rng.integers(0, 15, (I, H, W, 1)).astype(np.uint8)
    cw = (rng.random(14) + 0.1).astype(np.float32)
    cw[3] = 0.0
    vs, weights, scale = 0.02, (0.5, 1.5, 0.8), 1.75
    up = [rng.standard_normal(s).astype(np.float32) for s in ((I, H, W, 3), (I, H, W), (I, H, W, 3), (I, H, W, 14))]
    up[2] = None
    G, mag, bnd, (vals, vb) = O.fused_pixel_grads(color, depth, sem, td, tc, wc, label, cw, vs, weights, scale, up)

    t = lambda a: torch.from_numpy(a).double()
    c, d, s = (t(a).requires_grad_(True) for a in (color, depth, sem))
    terms = [R.depth_l1_loss(d, t(td), vs), R.compute_2dcolor_loss(c, t(tc), t(wc)),
             R.semantic_2d_ce_loss(s, torch.from_numpy(label), t(cw))]
    obj = scale * sum(w * x for w, x in zip(weights, terms))
    obj = obj + (c * t(up[0])).masked_fill(c == NINF, 0).sum() + (d * t(up[1])).masked_fill(d == NINF, 0).sum() + \
        (s * t(up[3])).masked_fill(s == NINF, 0).sum()
    obj.backward()
    want = O.route(s.grad.numpy(), c.grad.numpy(), d.grad.numpy(), np.zeros((I * H * W, 3)))
    h = hit.reshape(-1)  # the gather reads hit pixels only
    np.testing.assert_allclose(G[h], want[h], rtol=1e-6, atol=1e-12)
    for k, x in enumerate(terms):
        assert abs(vals[k] - float(x.detach())) <= 1e-6 * abs(float(x.detach()))
    assert bool((bnd <= 1e-4 * mag + 1e-30).all()) and bool((vb[3] <= 1e-5 * abs(vals[3])))
