"""Randomised sweep of the producer glue on float32 / bfloat16 heads in NCDHW, NDHWC and channel-slice layouts against the
literal expressions (rows of torch.nonzero, head[idx].float(), autograd of it), bit for bit.

    python tests/fuzz_head_formats.py --cases 2000 --seed 0
"""
import argparse
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SPECIALS = [float("nan"), float("inf"), -float("inf"), 0.0, -0.0]


def literal_locs(sdf, truncation, empty=None):
    mask = torch.abs(sdf.detach()[:, 0]) < truncation
    if empty is not None:
        mask = mask & ~empty[:, 0]
    locs = torch.nonzero(mask)
    return torch.cat([locs[:, 1:], locs[:, :1]], 1)


def literal_gather(head, locs):
    return head[locs[:, -1], :, locs[:, 0], locs[:, 1], locs[:, 2]].float()


def bits(t):
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32)


def same_bits(a, b):
    """bit-identical, except that a NaN only has to be a NaN in the other tensor too (its payload is not compared)"""
    a, b = a.contiguous(), b.contiguous()
    na, nb = torch.isnan(a), torch.isnan(b)
    return torch.equal(na, nb) and torch.equal(bits(a)[~na], bits(b)[~nb])


def same_values(a, b):
    """equal values (-0 == +0), NaN where the other has NaN"""
    return torch.equal(torch.isnan(a), torch.isnan(b)) and torch.equal(a.nan_to_num(0.0), b.nan_to_num(0.0))


def make_head(values, layout, dtype, channels, g):
    """values (B,C,Dz,Dy,Dx) float32 on the device -> a head of `dtype` in `layout` holding them (rounded)"""
    v = values.to(dtype)
    if layout == "ncdhw":
        return v.contiguous()
    if layout == "ndhwc":
        return v.contiguous(memory_format=torch.channels_last_3d)
    # a channel slice of a wider tensor, NCDHW or NDHWC
    B, C = v.shape[:2]
    extra = int(torch.randint(1, 6, (1,), generator=g))
    lo = int(torch.randint(0, extra + 1, (1,), generator=g))
    wide = torch.randn(B, C + extra, *v.shape[2:], device=v.device).to(dtype)
    if layout == "slice_ndhwc":
        wide = wide.contiguous(memory_format=torch.channels_last_3d)
    wide[:, lo:lo + C] = v
    return wide[:, lo:lo + C]


def one_case(g, dev):
    from spsg_b200 import sparsify
    B = int(torch.randint(1, 9, (1,), generator=g))
    dz, dy, dx = (int(torch.randint(1, 24, (1,), generator=g)) for _ in range(3))
    dtype = torch.bfloat16 if torch.rand(1, generator=g) < 0.6 else torch.float32
    T = float(torch.rand(1, generator=g) * 3.0 + 0.01)
    sdf = (torch.randn(B, 1, dz, dy, dx, generator=g) * 3.0)
    flat = sdf.view(-1)
    k = max(1, flat.numel() // 20)
    pos = torch.randint(0, flat.numel(), (k,), generator=g)
    choice = torch.randint(0, len(SPECIALS) + 3, (k,), generator=g)
    tb = float(torch.tensor(T).to(dtype).float())                      # the truncation in the head's dtype
    step = 2.0 ** (torch.floor(torch.log2(torch.tensor(tb))).item() - (7 if dtype == torch.bfloat16 else 23))
    for p, c in zip(pos.tolist(), choice.tolist()):
        if c < len(SPECIALS):
            flat[p] = SPECIALS[c]
        else:  # exactly the (rounded) truncation and one ulp of the head's dtype either side, either sign
            flat[p] = (tb + step * (c - len(SPECIALS) - 1)) * (1 if p % 2 else -1)
    sdf_layout = ["ncdhw", "ndhwc", "slice_ndhwc"][int(torch.randint(0, 3, (1,), generator=g))]
    sdf = make_head(sdf.to(dev), sdf_layout, dtype, 1, g)
    empty = (torch.rand(B, 1, dz, dy, dx, generator=g) < 0.3).to(dev) if torch.rand(1, generator=g) < 0.5 else None
    got = sparsify.sparse_locs(sdf, T, empty)
    want = literal_locs(sdf, T, empty)
    if got.shape != want.shape or not torch.equal(got, want):
        return 1, "rows"
    locs = want
    heads = []
    for _ in range(int(torch.randint(1, 7, (1,), generator=g))):
        C = [1, 3, 14, 19, 2, 5][int(torch.randint(0, 6, (1,), generator=g))]
        vals = torch.randn(B, C, dz, dy, dx, generator=g).to(dev)
        vals.view(-1)[::53] = float("nan")
        layout = ["ncdhw", "ndhwc", "slice_ncdhw", "slice_ndhwc"][int(torch.randint(0, 4, (1,), generator=g))]
        hdt = torch.bfloat16 if torch.rand(1, generator=g) < 0.6 else torch.float32
        heads.append(make_head(vals, layout, hdt, C, g))
    mine = [h.detach().requires_grad_(True) for h in heads]
    ref = [h.detach().clone().requires_grad_(True) for h in heads]
    out = sparsify.gather_dense(locs, *mine)
    out = out if isinstance(out, tuple) else (out,)
    want_v = [literal_gather(h, locs) for h in ref]
    for a, b in zip(out, want_v):
        if a.dtype != torch.float32 or not torch.equal(bits(a), bits(b)):
            return 1, "values"
    ws = [torch.randn(b.shape, generator=g).to(dev) for b in want_v]
    for w in ws:
        if w.numel():
            w.view(-1)[0] = -0.0
    ga = torch.autograd.grad(sum((a * w).sum() for a, w in zip(out, ws)), mine)
    gb = torch.autograd.grad(sum((b * w).sum() for b, w in zip(want_v, ws)), ref)
    for h, a, b in zip(heads, ga, gb):
        if a.dtype != h.dtype:
            return 1, "grad dtype"
        if h.dtype == torch.float32 and h.is_contiguous():  # the original scatter: equal values (it keeps -0 as -0)
            if not same_values(a, b):
                return 1, "grads"
        elif not same_bits(a, b):
            return 1, "grads"
        if h.shape[1] > 1 and h.stride(1) == 1 and not a.is_contiguous(memory_format=torch.channels_last_3d):
            return 1, "grad layout"
    return 0, None


def fuzz_run(cases, seed0=0, dev=None, verbose=False):
    dev = dev or torch.device("cuda", 0)
    bad = 0
    for i in range(cases):
        g = torch.Generator().manual_seed(seed0 * 100003 + i)
        torch.manual_seed(seed0 * 100003 + i)
        b, what = one_case(g, dev)
        if b and verbose:
            print("case %d (seed %d): %s mismatch" % (i, seed0, what))
        bad += b
    return bad


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", type=int, default=500)
    ap.add_argument("--seed", type=int, default=0)
    a = ap.parse_args()
    n = fuzz_run(a.cases, a.seed, verbose=True)
    print("fuzz_head_formats: %d cases, %d mismatching" % (a.cases, n))
    sys.exit(1 if n else 0)
