"""Per-voxel normals of the predicted sparse SDF: drop-in for the reference's ``loss.compute_normals_sparse``
(torch/loss.py:285-306, with ``compute_normals_dense`` :261-267), the producer of the raycaster's ``vals_normals``
(train.py:542) -- SURVEY.md section 8(f) rank 1.

The reference scatters the sparse values into a zero-filled dense volume, takes three slice differences, pads with -inf,
gathers back at the voxels, rotates chunk by chunk in a Python loop of 3x3 matmuls and normalises (about 15 kernels, two
dense temporaries and a boolean-mask sync per chunk).  Here it is one voxel-index build plus ONE gather kernel, and its
backward (the second gradient path into the SDF, SURVEY.md section 3.1) is two gather kernels without atomics.  No CPU path.

    normals = compute_normals_sparse(sdf_locs, sdf_vals, dims, transform=None)

``sdf_locs`` (N,4) int64 rows (z,y,x,chunk), sorted by chunk as ``torch.nonzero`` produces them (the reference
concatenates its result chunk by chunk, so for unsorted input its rows would come back permuted; sorted input is the only
case it is used with); ``sdf_vals`` (N,1) float32; ``dims`` (Dz,Dy,Dx); ``transform`` (B,4,4) grid->camera (the inverse view
matrix, train.py:544) or None.  Returns (N,3) float32.  Matches the reference within fp32 rounding (the 3x3 products are
summed in a fixed order here, in cuBLAS's order there).

    normals = compute_normals_sparse(sdf_locs, sdf_vals, dims, transform, views_per_chunk=F)

is the payload of a render with F views per chunk and per-view normals: ``transform`` (B*F,4,4), one per image in image
order (``inverse(view_matrix)``); returns (N,F,3), row (v, f) rotated by image ``chunk(v)*F + f``'s transform -- what F
calls with ``transform[f::F]`` give, bit for bit, with the central differences taken once.
"""
import torch
from torch.autograd import Function

from . import _native as N
from . import raycast_rgbd_cuda as rc


class _NormalsSparse(Function):
    @staticmethod
    def forward(ctx, sdf_locs, sdf_vals, transform, dims, num_chunks, views=1):
        rc._check_input(sdf_locs, "sdf_locs")
        rc._check_input(sdf_vals, "sdf_vals")
        rc._check_dtype(sdf_locs, torch.int64, "sdf_locs")
        rc._check_dtype(sdf_vals, torch.float32, "sdf_vals")
        if transform is not None:
            rc._check_input(transform, "transform")
            rc._check_dtype(transform, torch.float32, "transform")
            if transform.shape[0] < num_chunks * views or tuple(transform.shape[1:]) != (4, 4):
                if views > 1:
                    raise RuntimeError("transform must be (B*F,4,4) with B*F >= %d images" % (num_chunks * views))
                raise RuntimeError("transform must be (B,4,4) with B >= %d chunks" % num_chunks)
        n = sdf_locs.shape[0]
        if sdf_locs.dim() != 2 or sdf_locs.shape[1] != 4 or sdf_vals.numel() != n:
            raise RuntimeError("sdf_locs must be (N,4) and sdf_vals (N,1)")
        dev = sdf_vals.device
        index = torch.empty((num_chunks, dims[0], dims[1], dims[2]), dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            if views == 1:
                out = torch.empty((n, 3), dtype=torch.float32, device=dev)
                N.check(N.lib.spsg_normals_forward(N.ptr(sdf_locs), n, N.ptr(sdf_vals), N.ptr(transform), N.ptr(index),
                                                   num_chunks, dims[0], dims[1], dims[2], N.ptr(out), rc._stream(dev)))
            else:
                out = torch.empty((n, views, 3), dtype=torch.float32, device=dev)
                N.check(N.lib.spsg_normals_forward_views(N.ptr(sdf_locs), n, N.ptr(sdf_vals), N.ptr(transform), views,
                                                         N.ptr(index), num_chunks, dims[0], dims[1], dims[2], N.ptr(out),
                                                         rc._stream(dev)))
        ctx.save_for_backward(sdf_locs, sdf_vals, index)
        ctx.transform, ctx.dims, ctx.num_chunks, ctx.views = transform, dims, num_chunks, views
        return out

    @staticmethod
    def backward(ctx, grad_out):
        sdf_locs, sdf_vals, index = ctx.saved_tensors
        n = sdf_locs.shape[0]
        dev = sdf_vals.device
        grad_out = grad_out.contiguous().to(torch.float32)
        scratch = torch.empty((n, 3), dtype=torch.float32, device=dev)
        d_sdf = torch.empty_like(sdf_vals)
        dims = ctx.dims
        with torch.cuda.device(dev):
            if ctx.views == 1:
                N.check(N.lib.spsg_normals_backward(N.ptr(sdf_locs), n, N.ptr(sdf_vals), N.ptr(ctx.transform),
                                                    N.ptr(index), ctx.num_chunks, dims[0], dims[1], dims[2],
                                                    N.ptr(grad_out), N.ptr(scratch), N.ptr(d_sdf), rc._stream(dev)))
            else:
                N.check(N.lib.spsg_normals_backward_views(N.ptr(sdf_locs), n, N.ptr(sdf_vals), N.ptr(ctx.transform),
                                                          ctx.views, N.ptr(index), ctx.num_chunks, dims[0], dims[1],
                                                          dims[2], N.ptr(grad_out), N.ptr(scratch), N.ptr(d_sdf),
                                                          rc._stream(dev)))
        return None, d_sdf, None, None, None, None


def compute_normals_sparse(sdf_locs, sdf_vals, dims, transform=None, num_chunks=None, views_per_chunk=1):
    """Reference signature (loss.py:285) plus ``num_chunks``: the reference reads ``sdf_locs[-1, -1] + 1`` back from the
    device (loss.py:287, a host synchronisation); pass ``num_chunks`` (or a ``transform``, whose first dimension gives
    it) to avoid that.  ``views_per_chunk`` F > 1: per-view normals (N,F,3) for a render with F views per chunk;
    ``transform`` (B*F,4,4) is then required."""
    if not sdf_vals.is_cuda:
        raise RuntimeError("compute_normals_sparse needs CUDA tensors: this implementation has no CPU path")
    dims = (int(dims[0]), int(dims[1]), int(dims[2]))
    views = int(views_per_chunk)
    if views < 1:
        raise RuntimeError("views_per_chunk must be >= 1")
    if views > 1 and transform is None:
        raise RuntimeError("per-view normals need a (B*F,4,4) transform")
    if num_chunks is None:
        if transform is not None:
            num_chunks = int(transform.shape[0]) // views
        elif sdf_locs.shape[0] > 0:
            num_chunks = int(sdf_locs[-1, -1].item()) + 1  # loss.py:287
        else:
            num_chunks = 1
    sdf_vals_c = sdf_vals.contiguous()
    if transform is not None:
        transform = transform.contiguous()
    if views == 1:
        return _NormalsSparse.apply(sdf_locs.contiguous(), sdf_vals_c, transform, dims, int(num_chunks))
    return _NormalsSparse.apply(sdf_locs.contiguous(), sdf_vals_c, transform, dims, int(num_chunks), views)
