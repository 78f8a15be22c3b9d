"""Dense generator heads -> the raycaster's sparse inputs (reference ``torch/train.py:494-509``; SURVEY.md section 8(f)
rank 1).

The reference builds the voxel list and its payloads with PyTorch indexing::

    locs = torch.nonzero((torch.abs(output_sdf.detach()[:, 0]) < args.truncation) & ~empty[:, 0])    # train.py:495
    locs = torch.cat([locs[:, 1:], locs[:, :1]], 1)                                                    # :498
    output_sdf = [locs, output_sdf[locs[:, -1], :, locs[:, 0], locs[:, 1], locs[:, 2]]]                # :499
    output_color = [locs, output_color[locs[:, -1], :, locs[:, 0], locs[:, 1], locs[:, 2]]]            # :505
    output_semantic = output_semantic[locs[:, -1], :, locs[:, 0], locs[:, 1], locs[:, 2]]              # :508

``sparse_locs`` returns the same ``locs`` (same rows, same order, int64, columns z, y, x, b) from one ordered stream
compaction, and ``gather_dense`` the same values for any number of heads from fused gather launches, with the matching
backward (zero-filled dense gradient + scatter).  No CPU path.

Heads may be float32 or bfloat16 (a generator under ``torch.autocast(dtype=torch.bfloat16)``), NCDHW- or
NDHWC-contiguous (a generator in ``torch.channels_last_3d``) or channel slices of either: they are read where they are.
Gathered values are always float32; the gradient of a head has its dtype and, for channel-adjacent (NDHWC) heads, NDHWC
strides.  float32 NCDHW-contiguous heads take the original gather / scatter calls.  Any other dtype raises.
"""

import ctypes

import torch
from torch.autograd import Function

from . import _native as N
from . import raycast_rgbd_cuda as rc

_MAX_PAYLOADS = 4
_HEAD_DTYPES = (torch.float32, torch.bfloat16)


def _check_head_dtype(t, name):
    if t.dtype not in _HEAD_DTYPES:
        raise RuntimeError("%s must be float32 or bfloat16, got %s" % (name, t.dtype))


def _prepare(sdf, empty):
    """-> (sdf, empty, key): the (B,Dz,Dy,Dx) SDF as the compaction reads it, and what identifies the caller's tensor"""
    if sdf.dim() == 5:
        if sdf.shape[1] != 1:
            raise RuntimeError("sdf must have one channel")
        sdf = sdf[:, 0]
    if sdf.dim() != 4:
        raise RuntimeError("sdf must be (B,Dz,Dy,Dx) or (B,1,Dz,Dy,Dx)")
    sdf = sdf.detach()
    if not isinstance(sdf, torch.Tensor) or not sdf.is_cuda:
        raise RuntimeError("sdf must be a CUDA tensor")
    _check_head_dtype(sdf, "sdf")
    key = (sdf.data_ptr(), tuple(sdf.shape), sdf.stride(), sdf.dtype, sdf._version)
    if not sdf.is_contiguous():
        sdf = sdf.contiguous()  # a channel slice of a wider head: its one channel, packed for the 16-byte loads
    if empty is not None:
        if empty.dim() == 5:
            empty = empty[:, 0]
        if empty.shape != sdf.shape:
            raise RuntimeError("empty must have the shape of sdf")
        if empty.dtype not in (torch.bool, torch.uint8):
            raise RuntimeError("empty must be a bool (or uint8) mask")
        rc._check_input(empty, "empty")
    if sdf.data_ptr() % 16:
        sdf = sdf.clone()  # the kernels read 16-byte vectors
    if empty is not None and empty.data_ptr() % 8:
        empty = empty.clone()
    return sdf, empty, key


class CountedLocs:
    """Step 1 of the compaction done ahead of time (``count_locs``): ``n`` rows will come out; the per-tile offsets wait in
    a scratch buffer of their own until ``sparse_locs(..., counted=this)`` writes the rows."""

    def __init__(self, sdf, empty, truncation, scratch, n, key):
        self.sdf, self.empty, self.truncation, self.scratch, self.n = sdf, empty, float(truncation), scratch, n
        self.key = key


def count_locs(sdf, truncation, empty=None):
    """How many voxels ``sparse_locs`` will return (one host synchronisation, the one ``torch.nonzero`` has), keeping the
    work done: pass the result as ``counted=`` to ``sparse_locs`` / ``sparsify_predictions`` later.  Lets a training step
    decide early (train.py:524-529) and build the rows late -- after other renders on the same raycaster -- so that
    ``raycaster=`` still feeds the prediction render directly."""
    sdf, empty, key = _prepare(sdf, empty)
    dev = sdf.device
    cells = sdf.numel()
    if cells == 0:
        return CountedLocs(sdf, empty, truncation, None, 0, key)
    count = N.lib.spsg_sparsify_count if sdf.dtype == torch.float32 else N.lib.spsg_sparsify_count_bf16
    with rc.device_guard(dev):
        scratch = torch.empty(max(int(N.lib.spsg_sparsify_scratch_bytes(cells)), 256), dtype=torch.uint8, device=dev)
        total = torch.empty(1, dtype=torch.int64, device=dev)
        N.check(count(N.ptr(sdf), N.ptr(empty), cells, float(truncation), N.ptr(scratch), scratch.numel(), N.ptr(total),
                      rc._stream(dev)))
        n = int(total.item())  # the host needs N to size the outputs (torch.nonzero synchronises for the same reason)
    return CountedLocs(sdf, empty, truncation, scratch, n, key)


def sparse_locs(sdf, truncation, empty=None, raycaster=None, counted=None):
    """``locs`` (N,4) int64 rows (z, y, x, b) of the voxels with ``|sdf| < truncation`` (and ``~empty``), in
    ``torch.nonzero`` order.  sdf / empty: (B,Dz,Dy,Dx) or (B,1,Dz,Dy,Dx); empty is a bool mask or None.  A bfloat16
    sdf is compared as torch compares it with a Python scalar: ``truncation`` rounded to bfloat16 first.

    ``raycaster`` (a ``RaycastRGBD`` over the same grid): the pass that writes ``locs`` also writes the raycaster's voxel
    index (``sparse_mapping``) and dense SDF brick for these rows, so the forward that renders the returned tensor with
    the SDF values gathered from ``sdf`` skips its own fill and index passes (nothing goes through int64 ``locs`` twice).
    The caller's promise: the ``vals_sdf`` passed with these ``locs`` are ``gather_dense(locs, sdf)``.
    ``counted``: the result of ``count_locs`` on the same (unmodified) tensors."""
    if counted is None:
        counted = count_locs(sdf, truncation, empty)
    else:
        _, _, key = _prepare(sdf, empty)
        if key != counted.key or float(truncation) != counted.truncation:
            raise RuntimeError("counted= belongs to another sdf tensor / truncation (or the tensor was modified since)")
    sdf, empty, n, scratch = counted.sdf, counted.empty, counted.n, counted.scratch
    dev = sdf.device
    B, dz, dy, dx = sdf.shape
    if sdf.numel() == 0:
        return torch.zeros(0, 4, dtype=torch.int64, device=dev)
    with rc.device_guard(dev):
        stream = rc._stream(dev)
        locs = torch.empty(n, 4, dtype=torch.int64, device=dev)
        bf16 = sdf.dtype == torch.bfloat16
        if raycaster is not None and _feeds(raycaster, sdf, n):
            m = raycaster
            # the workspace of the forward to come, sized for the most views the module renders (the brick sits at its start)
            # and for the mode that forward will run in (deterministic mode needs more)
            flags = rc.with_torch_mode(m.flags) & (N.SPSG_FLAG_DETERMINISTIC | N.SPSG_FLAG_ALL_PIXELS)
            p = N.make_params(m.width, m.height, m.depth_min, m.depth_max, m.thresh_sample_dist, m.ray_increment,
                              m.dims3d[2], m.dims3d[1], m.dims3d[0], m.batch_size, m.max_num_frames,
                              rc.table_shape(m.mapping3dto2d, m.mapping3dto2d_num, flags)[1], n, flags)
            ws = m.workspace.get(dev, N.workspace_bytes(p))
            indexed = N.lib.spsg_sparsify_locs_indexed_bf16 if bf16 else N.lib.spsg_sparsify_locs_indexed
            N.check(indexed(N.ptr(sdf), N.ptr(empty), B, dz, dy, dx, float(truncation),
                            N.ptr(scratch), N.ptr(locs), n, N.ptr(m.sparse_mapping), N.ptr(ws), stream))
            m.workspace.mark_prebuilt(locs)
        else:
            write = N.lib.spsg_sparsify_locs_bf16 if bf16 else N.lib.spsg_sparsify_locs
            N.check(write(N.ptr(sdf), N.ptr(empty), B, dz, dy, dx, float(truncation), N.ptr(scratch), N.ptr(locs), n,
                          stream))
    return locs


def _feeds(m, sdf, n):
    """can the index + brick of raycaster ``m`` be written for this head: same grid, same device, rows within its buffers"""
    ws = getattr(m, "workspace", None)
    return (ws is not None and n > 0 and tuple(sdf.shape) == (m.batch_size,) + tuple(m.dims3d) and
            m.sparse_mapping.device == sdf.device and tuple(m.sparse_mapping.shape) == tuple(sdf.shape) and
            n * m.max_num_frames <= rc.table_shape(m.mapping3dto2d, m.mapping3dto2d_num, m.flags)[0])


def _payload_array(dense, sparse):
    arr = (N.DensePayload * len(dense))()
    for k, (d, s) in enumerate(zip(dense, sparse)):
        arr[k] = N.DensePayload(d.data_ptr(), s.data_ptr(), d.shape[1], 0)
    return arr


def _run(fn, dense, sparse, locs, shape):
    dev = locs.device
    B, dz, dy, dx = shape
    with rc.device_guard(dev):
        for k0 in range(0, len(dense), _MAX_PAYLOADS):
            d, s = dense[k0:k0 + _MAX_PAYLOADS], sparse[k0:k0 + _MAX_PAYLOADS]
            N.check(fn(_payload_array(d, s), len(d), N.ptr(locs), locs.shape[0], B, dz, dy, dx, rc._stream(dev)))


def _head_array(dense, sparse):
    arr = (N.DenseHead * len(dense))()
    for k, (d, s) in enumerate(zip(dense, sparse)):
        extent = d.untyped_storage().nbytes() // d.element_size() - d.storage_offset()
        arr[k] = N.DenseHead(d.data_ptr(), s.data_ptr(), (ctypes.c_int64 * 5)(*d.stride()), extent, d.shape[1],
                             N.SPSG_DTYPE_BF16 if d.dtype == torch.bfloat16 else N.SPSG_DTYPE_F32)
    return arr


def _run_strided(fn, dense, sparse, locs, shape):
    dev = locs.device
    B, dz, dy, dx = shape
    with rc.device_guard(dev):
        for k0 in range(0, len(dense), _MAX_PAYLOADS):
            d, s = dense[k0:k0 + _MAX_PAYLOADS], sparse[k0:k0 + _MAX_PAYLOADS]
            N.check(fn(_head_array(d, s), len(d), N.ptr(locs), locs.shape[0], B, dz, dy, dx, rc._stream(dev)))


def _original_route(t):
    """float32 NCDHW-contiguous heads take spsg_dense_gather / spsg_dense_scatter, as they always did"""
    return t.dtype == torch.float32 and t.is_contiguous()


def _grad_format(t):
    """(dtype, memory format) of head t's gradient: its dtype; NDHWC when its channels are adjacent (an NDHWC head or a
    channel slice of one), else NCDHW"""
    return t.dtype, torch.channels_last_3d if t.shape[1] > 1 and t.stride(1) == 1 else torch.contiguous_format


class _GatherDense(Function):
    @staticmethod
    def forward(ctx, locs, *dense):
        shape = (dense[0].shape[0],) + tuple(dense[0].shape[2:])
        for t in dense:
            if not t.is_cuda:
                raise RuntimeError("dense head must be a CUDA tensor")
            _check_head_dtype(t, "dense head")
            if t.dim() != 5 or (t.shape[0],) + tuple(t.shape[2:]) != shape:
                raise RuntimeError("dense heads must be (B,C,Dz,Dy,Dx) tensors over the same grid")
        rc._check_input(locs, "locs")
        rc._check_dtype(locs, torch.int64, "locs")
        n = locs.shape[0]
        out = tuple(torch.empty(n, t.shape[1], device=t.device) for t in dense)
        orig = [k for k, t in enumerate(dense) if _original_route(t)]
        strided = [k for k, t in enumerate(dense) if not _original_route(t)]
        if orig:
            _run(N.lib.spsg_dense_gather, [dense[k] for k in orig], [out[k] for k in orig], locs, shape)
        if strided:
            _run_strided(N.lib.spsg_dense_gather_strided, [dense[k] for k in strided], [out[k] for k in strided], locs,
                         shape)
        ctx.locs, ctx.shape = locs, shape
        ctx.channels = tuple(t.shape[1] for t in dense)
        ctx.grad_formats = tuple(None if _original_route(t) else _grad_format(t) for t in dense)
        return out

    @staticmethod
    def backward(ctx, *grads):
        locs, shape = ctx.locs, ctx.shape
        B, dz, dy, dx = shape
        need = ctx.needs_input_grad[1:]
        idx = [k for k, nd in enumerate(need) if nd]
        sparse = {k: grads[k].to(torch.float32).contiguous() if grads[k] is not None
                  else torch.zeros(locs.shape[0], ctx.channels[k], device=locs.device) for k in idx}
        out = [None] * len(need)
        orig = [k for k in idx if ctx.grad_formats[k] is None]
        strided = [k for k in idx if ctx.grad_formats[k] is not None]
        for k in orig:
            out[k] = torch.empty(B, ctx.channels[k], dz, dy, dx, device=locs.device)
        for k in strided:
            dtype, fmt = ctx.grad_formats[k]
            out[k] = torch.empty(B, ctx.channels[k], dz, dy, dx, dtype=dtype, device=locs.device, memory_format=fmt)
        if orig:
            _run(N.lib.spsg_dense_scatter, [out[k] for k in orig], [sparse[k] for k in orig], locs, shape)
        if strided:
            _run_strided(N.lib.spsg_dense_scatter_strided, [out[k] for k in strided], [sparse[k] for k in strided], locs,
                         shape)
        return (None,) + tuple(out)


def gather_dense(locs, *dense):
    """``head[locs[:, -1], :, locs[:, 0], locs[:, 1], locs[:, 2]].float()`` for every head (B,C,Dz,Dy,Dx) -> (N,C) float32,
    one fused launch per four heads; differentiable with respect to the heads.  float32 or bfloat16 heads, NCDHW, NDHWC
    or channel slices of either, are read where they are."""
    if not dense:
        return ()
    out = _GatherDense.apply(locs, *dense)
    return out if len(dense) > 1 else out[0]


def sparsify_predictions(output_sdf, truncation, empty=None, *heads, raycaster=None, counted=None):
    """train.py:494-509 in one call: ``(locs, sdf_values, *head_values)`` for the dense SDF head (B,1,Dz,Dy,Dx) and any
    further heads (colour, semantics, a one-hot target volume, ...).  ``raycaster`` / ``counted``: see ``sparse_locs`` --
    the rows feed that raycaster's next forward directly."""
    locs = sparse_locs(output_sdf, truncation, empty, raycaster=raycaster, counted=counted)
    vals = gather_dense(locs, output_sdf, *heads)
    if not heads:
        vals = (vals,)
    return (locs,) + tuple(vals)
