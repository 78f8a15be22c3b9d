"""Randomised sweep of per-view normals (SPSG_FLAG_VIEW_NORMALS) against per-view single calls;
tests/test_gpu_view_normals.py runs a seeded slice under pytest and uses the same case runner.

Each case renders a random soup (B = 1-8 chunks, F = 1-5 views, random cameras, N, max_pixels_per_voxel and flags) with an
(N,F,3) normal payload encoding (v + 1, f + 0.5, -0.25), some rows zero, and checks:
  * image b*F + f's four renderings are bit-identical to a single-view launch with cameras view[f::F] and payload
    normals[:, f], and its registration counts to that launch's;
  * colour, depth, semantic and the counts are bit-identical to the shared-normals (N,3) render of the same cameras;
  * backward (plain through autograd, fused, fused + upstream images; atomics or deterministic): d_normal[:, f] is the
    single-view backward of view f's normal gradient bit for bit, except for voxels whose table overflowed and for counted
    near-ties of the final rounding (as tests/gather_oracle.py counts them: the pixels are summed in registration order);
    colour, depth and semantic are bit-identical to the shared-mode backward on the same tables (deterministic) or within
    2^-20 of its largest entry per channel (float atomics).
usage: python tests/fuzz_view_normals.py [cases] [seed]"""
import ctypes
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import numpy as np
import torch

from spsg_b200 import _native as N
from tests import fuzz_gather as FZ
from tests import gather_oracle as O
from tests.common import hit_image_from_mapping

NINF = -float("inf")
VARIANTS = ("plain", "fused", "fused_up")


def view_payload(n, F, dev, rng, zero_frac=0.05):
    """(N,F,3) fp32: row (v, f) = (v + 1, f + 0.5, -0.25), a random fraction of the rows zero (rendered as -inf)."""
    assert n < (1 << 24)
    p = np.empty((n, F, 3), np.float32)
    p[:, :, 0] = np.arange(1, n + 1, dtype=np.float32)[:, None]
    p[:, :, 1] = np.arange(F, dtype=np.float32)[None, :] + 0.5
    p[:, :, 2] = -0.25
    p[rng.random((n, F)) < zero_frac] = 0.0
    return torch.from_numpy(p).to(dev)


def raycasters(dev, B, F, dims, w, h, n, max_pix=64, det=False, flags=0, dmin=0.0, dmax=150.0, inc=0.9):
    """(F-view module, single-view module) with the same buffers' geometry."""
    m = FZ.raycaster(dev, B, F, dims, w, h, n, dmin, dmax, inc, max_pix, det, flags)
    s = FZ.raycaster(dev, B, 1, dims, w, h, n, dmin, dmax, inc, max_pix, False, flags)
    return m, s


def _per_view(x, B, F, f):
    """Images b*F + f of an (I, ...) tensor."""
    return x.reshape((B, F) + tuple(x.shape[1:]))[:, f]


def _bits_equal(a, b):
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def _native_backward(m, p, n, planes=None, fused=None):
    """The C ABI backward on m's tables and workspace, in the mode ``p.flags`` says, into fresh buffers.
    planes: plain gradient images (colour, depth, normal, semantic); fused: (tg, loss_out, grad_scale, upstream planes)."""
    dev = m.image_depth.device
    q = N.Params.from_buffer_copy(p)
    q.flags &= ~N.SPSG_FLAG_GRADS_CLEARED
    nv = q.views_per_chunk if q.flags & N.SPSG_FLAG_VIEW_NORMALS else 1
    d = [torch.full((n, c), float("nan"), device=dev) for c in (3, 1, 3 * nv, 14)]
    ws = m.workspace.ws
    st = torch.cuda.current_stream(dev).cuda_stream
    tables = (N.ptr(m.sparse_mapping), N.ptr(m.mapping3dto2d), N.ptr(m.mapping3dto2d_num))
    outs = tuple(N.ptr(x) for x in d)
    if fused is None:
        N.check(N.lib.spsg_raycast_backward(ctypes.byref(q), *(N.ptr(g) for g in planes), *tables, *outs, N.ptr(ws),
                                            ws.numel(), st))
    else:
        tg, loss_out, scale, up = fused
        ups = N.UpstreamGrads(*(N.ptr(g) for g in up)) if up is not None else None
        N.check(N.lib.spsg_raycast_backward_loss_upstream(
            ctypes.byref(q), N.ptr(m.image_color), N.ptr(m.image_depth), N.ptr(m.image_semantic), ctypes.byref(tg),
            N.ptr(loss_out), N.ptr(scale), ctypes.byref(ups) if ups is not None else None, *tables, *outs, N.ptr(ws),
            ws.numel(), st))
    return d


def _normal_ties(m, t, n, B, F, f, gn, cnt):
    """Near-tie entries (N,3) of view f's normal means (gather_oracle.gather's rule): the kernel sums each (voxel, view)'s
    pixels in double precision in registration order, which differs between the two launches."""
    I, H, W = gn.shape[0], gn.shape[1], gn.shape[2]
    vox = hit_image_from_mapping(m.mapping3dto2d, m.mapping3dto2d_num, t["locs"], I, H, W, F)
    vf = _per_view(vox, B, F, f).reshape(-1)
    g = _per_view(gn, B, F, f).reshape(-1, 3).double()
    hit = vf >= 0
    S = torch.zeros(n, 3, dtype=torch.float64, device=gn.device).index_add_(0, vf[hit], g[hit])
    A = torch.zeros(n, 3, dtype=torch.float64, device=gn.device).index_add_(0, vf[hit], g[hit].abs())
    S, A, c = S.cpu().numpy(), A.cpu().numpy(), cnt.cpu().numpy().astype(np.float64)[:, None]
    live = c > 0
    inv = np.where(live, (1.0 / np.where(live, c, 1.0)).astype(np.float32).astype(np.float64), 0.0)
    x = S * inv
    delta = 2 * c * 2.0 ** -53 * A * inv + 2.0 ** -51 * np.abs(x)
    return torch.from_numpy(live & O.near_tie(x, delta)).to(gn.device)


def check_case(dev, t, n, B, F, view, intr, m, s, variant="plain", seed=0, backward=True, what=""):
    """One case (module docstring).  Returns (overflowed rows, near-tie entries excluded)."""
    from spsg_b200 import losses as L
    rng = np.random.default_rng(seed)
    locs, sdf, col, sem = t["locs"], t["sdf"], t["color"], t["semantic"]
    P = view_payload(n, F, dev, rng)
    I = B * F
    det = bool(m.flags & N.SPSG_FLAG_DETERMINISTIC_GRADS)
    # today's shared-normals render of the same cameras
    with torch.no_grad():
        sh = [o.clone() for o in m(locs, sdf, col, P[:, 0].contiguous(), sem, view, intr)]
    num_sh = m.mapping3dto2d_num[:F * n].clone()
    # per-view render (its tables stay in m for the backward)
    p = tg = loss_out = scale = up = None
    if variant == "plain":
        ls = [x.clone().requires_grad_(True) for x in (sdf, col, P, sem)]
        out = m(locs, *ls, view, intr)
        pv = [o.detach().clone() for o in out]
    else:
        tgt, _ = FZ.fused_targets(sh, rng, dev, tuple(bool(x) for x in rng.random(3) < 0.7))
        targets = (tgt["images_depth"], tgt["images_color"], tgt["weight_color"], tgt["target2d_label"],
                   tgt["weight_semantic_class"], 0.02, (0.5, 1.5, 0.8))
        p, tg, loss_out = L.fused_forward(m, locs, sdf, col, P, sem, view, intr, targets, n > 0)
        assert p.flags & N.SPSG_FLAG_VIEW_NORMALS, what
        pv = [x[:I].clone() for x in (m.image_color, m.image_depth, m.image_normal, m.image_semantic)]
    num_pv = m.mapping3dto2d_num[:F * n].clone()
    for k, plane in ((0, "colour"), (1, "depth"), (3, "semantic")):
        assert _bits_equal(pv[k], sh[k]), "%s: %s differs from the shared-normals render" % (what, plane)
    assert torch.equal(num_pv, num_sh), "%s: registration counts differ from the shared-normals render" % what
    nrm = pv[2]
    fin = nrm[..., 1] != NINF
    img_view = (torch.arange(I, device=dev) % F).float()[:, None, None] + 0.5
    assert bool((nrm[..., 1] == img_view)[fin].all()), "%s: a pixel shows another view's normal row" % what
    # gradients of the per-view route
    if backward:
        if variant == "plain":
            planes = FZ.upstream_grads([o.shape for o in out], dev, seed)
            torch.autograd.backward(out, planes)
            got = [x.grad for x in ls]  # sdf, colour, normal (N,F,3), semantic
            gn = planes[2]
            p = N.make_params(m.width, m.height, 0, 0, 0, 0, m.dims3d[2], m.dims3d[1], m.dims3d[0], B, F,
                              m.mapping3dto2d.shape[1], n, m.flags | N.SPSG_FLAG_VIEW_NORMALS)
            same = _native_backward(m, p, n, planes=(planes[0], planes[1], planes[2], planes[3]))
        else:
            scale = torch.tensor(float(rng.choice([1.0, 0.37, 3.0])), device=dev)
            if variant == "fused_up":
                up = FZ.upstream_grads([x.shape for x in pv], dev, seed + 1)
            L.fused_backward(m, p, tg, loss_out, scale, n > 0, up)
            g = L._voxel_grads(m, p, n)
            got = [x.clone() for x in (g[0], g[1], g[2], g[3])]
            gn = up[2] if up is not None else torch.zeros_like(pv[2])
            same = None
        assert tuple(got[2].shape) == (n, F, 3), "%s: normal gradient shape %s" % (what, tuple(got[2].shape))
        # shared mode on the same tables: colour, depth and semantic
        q = N.Params.from_buffer_copy(p)
        q.flags &= ~N.SPSG_FLAG_VIEW_NORMALS
        if same is None:
            same = _native_backward(m, q, n, fused=(tg, loss_out, scale, up))
        else:
            same = _native_backward(m, q, n, planes=(planes[0], planes[1], planes[2], planes[3]))
        for a, b, name in ((got[1], same[0], "colour"), (got[0], same[1], "depth"), (got[3], same[3], "semantic")):
            if det or F == 1:
                assert _bits_equal(a, b), "%s: %s gradient differs from the shared-mode backward" % (what, name)
            else:
                tol = 2.0 ** -20 * float(b.abs().max()) if b.numel() else 0.0
                err = float((a - b).abs().max()) if b.numel() else 0.0
                assert err <= tol, "%s: %s gradient %g off the shared-mode backward (bound %g)" % (what, name, err, tol)
    # single-view launches, view by view
    overflow = ties = 0
    max_pix = m.mapping3dto2d.shape[1]
    for f in range(F):
        Pf = P[:, f].contiguous().requires_grad_(backward)
        so = s(locs, sdf, col, Pf, sem, view[f::F].contiguous(), intr[f::F].contiguous())
        for k, plane in enumerate(("colour", "depth", "normal", "semantic")):
            assert _bits_equal(so[k], _per_view(pv[k], B, F, f)), \
                "%s: view %d %s differs from the single-view launch" % (what, f, plane)
        num_f = num_pv[f * n:(f + 1) * n]
        assert torch.equal(s.mapping3dto2d_num[:n], num_f), "%s: view %d counts differ from the single-view launch" % (what, f)
        if not backward:
            continue
        gn_f = _per_view(gn, B, F, f).contiguous()
        torch.autograd.backward(so[2], gn_f)
        want = Pf.grad
        a = got[2][:, f].contiguous()
        ok_rows = (num_f <= max_pix)[:, None].expand(n, 3)
        overflow += int((num_f > max_pix).sum())
        tie = _normal_ties(m, t, n, B, F, f, gn, num_f.clamp(max=max_pix))
        bad = (a.view(torch.int32) != want.view(torch.int32)) & ~(a == want) & ok_rows & ~tie
        ties += int((tie & ok_rows).sum())
        if bool(bad.any()):
            v, c = [int(x) for x in torch.nonzero(bad)[0]]
            raise AssertionError("%s: view %d d_normal differs from the single-view backward at %d entries (voxel %d "
                                 "channel %d: %r vs %r)" % (what, f, int(bad.sum()), v, c, float(a[v, c]),
                                                              float(want[v, c])))
    return overflow, ties


def draw(rng):
    """One random case."""
    B, F = int(rng.integers(1, 9)), int(rng.integers(1, 6))
    dims = tuple(int(v) for v in rng.integers(6, 61, 3))
    kinds = ["noise", "blocky", "special"]
    specs = [(int(rng.integers(0, 1 << 30)), kinds[int(rng.integers(0, 3))]) for _ in range(B)]
    if B > 1 and rng.random() < 0.2:
        specs[int(rng.integers(0, B))] = None
    w, h = int(rng.integers(1, 97)), int(rng.integers(1, 73))
    flags = [0, 0, N.SPSG_FLAG_SMEM_MAPS, N.SPSG_FLAG_GLOBAL_MAPS, N.SPSG_FLAG_NO_BRICK_SKIP][int(rng.integers(0, 5))]
    return dict(dims=dims, B=B, F=F, specs=specs, keep=int(rng.integers(1, 4000)) if rng.random() < 0.3 else None, w=w,
                h=h, max_pix=int(rng.choice(FZ.MAX_PIX)), det=bool(rng.random() < 0.5), flags=flags,
                focal=float(rng.uniform(0.5, 1.5)), cam_seed=int(rng.integers(0, 1 << 30)),
                variant=VARIANTS[int(rng.integers(0, 3))])


def run_case(c, dev, seed):
    from tests.test_gpu_adversarial import _cameras
    specs = c["specs"] if any(s is not None for s in c["specs"]) else [(1, "blocky")] + c["specs"][1:]
    t, n = FZ.scene(dev, c["dims"], specs, c["keep"])
    B, F = c["B"], c["F"]
    view = _cameras(c["dims"], B * F, c["cam_seed"], dev)
    intr = FZ.intrinsics(dev, B * F, c["w"], c["h"], c["focal"])
    m, s = raycasters(dev, B, F, c["dims"], c["w"], c["h"], n, c["max_pix"], c["det"], c["flags"])
    what = "case %s" % {k: v for k, v in c.items() if k != "specs"}
    return check_case(dev, t, n, B, F, view, intr, m, s, c["variant"], seed, True, what)


def run(cases=100, seed0=0, dev=None):
    """Returns the number of mismatching cases."""
    dev = dev or torch.device("cuda", 0)
    bad = overflow = ties = 0
    t0 = time.time()
    for k in range(cases):
        rng = np.random.default_rng(seed0 * 100003 + k)
        c = draw(rng)
        try:
            ov, ti = run_case(c, dev, seed0 * 100003 + k)
            overflow += ov > 0
            ties += ti
        except AssertionError as e:
            bad += 1
            print("MISMATCH case %d: %s" % (k, e), flush=True)
    print("%d cases, %d with a pixel-table overflow, %d near-tie entries excluded, %d mismatching, %.1f s"
          % (cases, overflow, ties, bad, time.time() - t0))
    return bad


if __name__ == "__main__":
    sys.exit(1 if run(int(sys.argv[1]) if len(sys.argv) > 1 else 100, int(sys.argv[2]) if len(sys.argv) > 2 else 0) else 0)
