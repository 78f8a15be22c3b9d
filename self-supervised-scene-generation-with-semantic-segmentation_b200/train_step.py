"""The 2D view-guided training step (BASELINE.json configs[3]; reference ``torch/train.py:399-757``) on this package's ops.

The reference's step is: generator forward (``train.py:465``) -> dense 3D losses (``:476-493``) -> sparsification of the
predicted SDF / colour / semantic heads (``:494-509``) -> per-voxel normals (``:542-544``) -> three raycasts of the same
camera set -- the input scan (``:556-578``), the target chunk whose rendered semantics become the 2D labels (``:581-622``)
and the prediction (``:626-632``) -- -> depth L1 / colour L1 / 2D semantic cross-entropy (``:635-643, 744-746``) ->
``loss.backward()``, ``optimizer.step()`` (``:756-757``).

``ViewGuidedTrainStep`` runs exactly that data flow with every op between the generator's dense heads and the scalar loss
replaced by this package's CUDA ops: ordered stream compaction + fused gathers (``sparsify``), the sparse normals kernel
(``normals``), the persistent raycast kernel, its label render (``RaycastRGBD.render_labels``) and the raycast with the
three 2D losses fused into its epilogue (``losses.render_with_2d_losses``).  The generator and the dense 3D losses are the
caller's (the reference's own ``model.Generator`` / ``loss`` module in bench.py and the tests): they are stock PyTorch and
outside the hot path (SURVEY.md section 8).  Data parallelism is ``torch.nn.parallel.DistributedDataParallel`` around the
generator: its gradient all-reduce is the step's only collective (SURVEY.md section 8(e)).  No CPU path.
"""
import contextlib

import torch

from . import losses, normals, sparsify
from .raycast_rgbd import RaycastRGBD


def prepare_generator(model):
    """The generator laid out for B200: parameters (and with them every activation cuDNN produces) in
    ``torch.channels_last_3d`` (NDHWC).  The reference's ``Generator`` is a Conv3d + BatchNorm3d U-Net with 10-100 channels on
    128x64x64 volumes; in the default NCDHW layout cuDNN brackets its tensor-core kernels with layout transposes, in NDHWC it
    does not: forward + backward of a batch of 8 takes 196 ms instead of 332 ms (same TF32 convolutions, same loss to the
    last printed digit; ``tools/gen_layout_probe.py``).  Nothing in the model changes.  Call before wrapping in DDP."""
    return model.to(memory_format=torch.channels_last_3d)


class ViewGuidedTrainStep:
    """One training iteration past ``num_iters_geo_only`` with the 2D semantic branch (``--pred_3d_semantic ''``)
    (``train.py:740-747``), with or without image-space terms such as the reference's GAN and VGG style losses.

    model       generator with the reference's call signature ``model(inputs, mask, pred_sdf=[..], pred_color=..,
                pred_semantic=..) -> (occ, sdf, colour, semantic)`` dense heads (``model.py:345``); may be DDP-wrapped
    loss_util   module providing the reference's dense 3D losses (``loss.compute_targets``, ``compute_dense_geo_weights``,
                ``compute_geo_occ_loss``, ``compute_geo_loss``; loss.py:8-146)
    image_loss  None (GAN and style terms off), or a callable ``image_loss(pred, input2d) -> scalar`` added to the loss:
                ``pred`` = the prediction's ``(color, depth, normal, semantic)`` renderings, differentiable (their
                gradients are gathered into the voxels by the fused backward); ``input2d`` = the input scan's (I,6,H,W)
                conditioning ``cat(colour * 2 - 1, normal)`` with misses set to 0, channels first, as in train.py:556-578,
                or None with ``render_input=False``.  ``pred`` are the raycaster's buffers, valid until the next step.
                The discriminator, its own update and the exact form of the GAN / style terms are the caller's: this
                step only adds what ``image_loss`` returns.  Its value is recorded in ``self.last["image_loss"]``.
    autocast_bf16  run the generator forward and the dense 3D losses under ``torch.autocast("cuda", dtype=torch.bfloat16)``.
                The bfloat16 heads (NDHWC with ``prepare_generator``) go to the producer glue as they are; from the voxel
                payloads on (normals, the three raycasts, the 2D losses, ``image_loss``) everything stays float32.  No
                gradient scaler: bfloat16 has float32's exponent range.  False: the float32 step.
    max_pixels_per_voxel  the raycaster's voxel -> pixel table width (64, the reference's): a (voxel, view)'s gradient is
                the mean over the first that many of its pixels.  None: over all of them, without the table
                (``RaycastRGBD(..., max_pixels_per_voxel=None)``; at B = 8, F = 1 and the default row bound that drops a
                1.31 GB allocation).
    num_classes the semantic label set's size C (14, the reference's; e.g. 20 for ScanNet, 41 for NYU40): the generator's
                semantic head has C channels, ``sample["semantics"]`` holds labels 0..C (C = unlabeled) and ``class_weight``
                C weights.  The raycaster and the 2D labels are C wide.
    """

    def __init__(self, model, loss_util, batch_size, dims3d, width, height, class_weight, voxelsize=0.02, truncation=3.0,
                 weight_occ_loss=1.0, weight_sdf_loss=0.1, weight_depth_loss=1.0, weight_color_loss=1.0,
                 weight_semantic_loss=0.1, weight_surf_geo=1.0, weight_missing_geo=5.0, logweight_sdf=True,
                 max_num_locs_per_sample=640000, views_per_chunk=1, render_input=True, device=None, image_loss=None,
                 autocast_bf16=False, max_pixels_per_voxel=64, num_classes=14):
        self.model, self.loss_util = model, loss_util
        self.image_loss = image_loss
        self.autocast_bf16 = autocast_bf16
        self.batch_size, self.dims3d, self.width, self.height = batch_size, tuple(dims3d), width, height
        self.voxelsize, self.truncation = voxelsize, truncation
        self.w = dict(occ=weight_occ_loss, sdf=weight_sdf_loss, depth=weight_depth_loss, color=weight_color_loss,
                      semantic=weight_semantic_loss)
        self.weight_surf_geo, self.weight_missing_geo, self.logweight_sdf = weight_surf_geo, weight_missing_geo, logweight_sdf
        self.class_weight = class_weight
        self.views = views_per_chunk
        self.num_classes = num_classes
        self.render_input = render_input
        ray_increment = 0.3 * truncation            # train.py:134
        thresh_sample_dist = 50.5 * ray_increment   # train.py:135
        self.raycaster = RaycastRGBD(batch_size, self.dims3d, width, height, depth_min=0.1 / voxelsize,
                                     depth_max=6.0 / voxelsize, thresh_sample_dist=thresh_sample_dist,
                                     ray_increment=ray_increment, max_num_frames=views_per_chunk,
                                     max_num_locs_per_sample=max_num_locs_per_sample,
                                     max_pixels_per_voxel=max_pixels_per_voxel, device=device, num_classes=num_classes)
        self.last = {}

    def _normals(self, locs, vals, transform):
        """train.py:542-544: the voxels' normals in the camera frame of the image that renders them.  With several views
        per chunk that is one normal per (voxel, view): ``transform`` holds one (4,4) per image, (N,F,3) comes back."""
        if self.views == 1:
            return normals.compute_normals_sparse(locs, vals, self.dims3d, transform=transform)
        return normals.compute_normals_sparse(locs, vals, self.dims3d, transform=transform, views_per_chunk=self.views)

    def _target_labels(self, target_for_sdf, target_for_colors, target_for_semantics, view_matrix, intrinsics, transform):
        """train.py:581-622: render the target chunk, its semantics become the per-pixel labels.  The reference renders
        colours, normals and a one-hot semantic image and takes its argmax (train.py:590-616); each pixel's label is that
        of its hit voxel (C where the ray misses, or the voxel is unlabeled), which the label render writes directly.  The
        target colours and the cameras' ``transform`` are not needed for that."""
        locs, vals = sparsify.sparsify_predictions(target_for_sdf, self.truncation)
        sem = sparsify.gather_dense(locs, target_for_semantics.float())
        voxel_labels = sem[:, 0].to(torch.uint8).contiguous()
        return self.raycaster.render_labels(locs, vals, voxel_labels, view_matrix, intrinsics)  # (I,H,W) uint8

    def _render_input(self, inputs, view_matrix, intrinsics, transform):
        """train.py:556-578: the input scan's colour / normal rendering (the discriminator's conditioning; with no
        ``image_loss`` nothing reads it, it only keeps the step's work like the reference's).  Returns the raycaster's
        buffers, which the next render overwrites.  Its normals come from the sparse
        normals kernel (absent neighbours count as 0), where the reference uses `loss.compute_normals` on the dense input
        volume (truncated neighbours count as +-truncation): the two differ at the rim of the input's band."""
        locs, vals, cols = sparsify.sparsify_predictions(inputs[:, :1].contiguous(), self.truncation, None,
                                                         inputs[:, 1:4].contiguous())
        input_normals = self._normals(locs, vals, transform)
        raycast_color, _, raycast_normal, _ = self.raycaster(locs, vals, cols, input_normals, None, view_matrix, intrinsics)
        return raycast_color, raycast_normal

    @staticmethod
    def _conditioning(raycast_color, raycast_normal):
        """train.py:556-578 (baseline/ref_train_step.py:85-91): (I,6,H,W) = cat(colour * 2 - 1, normal), misses -> 0."""
        miss = -float("inf")
        color = torch.where(raycast_color == miss, torch.zeros_like(raycast_color), raycast_color * 2 - 1)
        normal = torch.where(raycast_normal == miss, torch.zeros_like(raycast_normal), raycast_normal)
        return torch.cat([color, normal], 3).permute(0, 3, 1, 2).contiguous()

    def __call__(self, sample, optimizer=None):
        """sample: dict with the reference dataloader's keys (scene_dataloader.py / data_util.py:862-902), all on the
        device: input (B,4,Dz,Dy,Dx), mask (B,1,..), sdf (B,1,..), known (B,1,..) bool or None, colors (B,Dz,Dy,Dx,3) uint8,
        semantics (B,1,Dz,Dy,Dx) labels 0..14, images_color (I,3,H,W), images_depth (I,H,W), view_matrix (I,4,4),
        images_intrinsic (I,4); I = B * views_per_chunk.  Returns the total loss (after backward / optimizer step when an
        optimizer is given)."""
        lu, T = self.loss_util, self.truncation
        inputs, mask, known = sample["input"], sample["mask"], sample.get("known")
        target_for_sdf, target_for_colors = lu.compute_targets(sample["sdf"], T, True, known, sample["colors"])
        target_for_semantics = sample["semantics"]
        if optimizer is not None:
            optimizer.zero_grad(set_to_none=True)
        dense_region = (torch.autocast("cuda", dtype=torch.bfloat16) if self.autocast_bf16 else contextlib.nullcontext())
        with dense_region:
            output_occ, output_sdf, output_color, output_semantic = self.model(
                inputs, mask, pred_sdf=[True, True], pred_color=True, pred_semantic=True)      # train.py:465
            # ---- dense 3D losses (train.py:476-493), the caller's functions
            input_occ = torch.abs(inputs[:, :1]) < (T - 0.01)
            weight = lu.compute_dense_geo_weights(target_for_sdf, input_occ, T, self.weight_surf_geo,
                                                  self.weight_missing_geo)
            empty = torch.sigmoid(output_occ.detach()) < 0.5
            weight[empty] = 0
            loss_occ = lu.compute_geo_occ_loss(target_for_sdf, output_occ, known, weight, T)
            loss_sdf = lu.compute_geo_loss(target_for_sdf, None, output_sdf, known, weight, self.logweight_sdf)
            loss = self.w["occ"] * loss_occ + self.w["sdf"] * loss_sdf
        # ---- dense heads -> sparse raycaster inputs (train.py:494-509)
        # (counted first, written after the other two renders of the step: the rows then feed the prediction render
        # directly -- voxel index and SDF brick written with them, see sparsify.sparse_locs)
        counted = sparsify.count_locs(output_sdf, T, empty)
        n = counted.n
        self.last = dict(num_locs=n, loss_occ=loss_occ.detach(), loss_sdf=loss_sdf.detach())
        if 0 < n <= self.raycaster.get_max_num_locs_per_sample() * self.batch_size:          # train.py:524-529
            view_matrix, intrinsics = sample["view_matrix"], sample["images_intrinsic"]
            transform = torch.inverse(view_matrix)                    # train.py:544, one per image (I = B * F)
            input2d = None
            if self.render_input:
                input_color, input_normal = self._render_input(inputs, view_matrix, intrinsics, transform)
                if self.image_loss is not None:  # now: the two renders below overwrite these buffers
                    input2d = self._conditioning(input_color, input_normal)
            with torch.no_grad():
                target2d_label = self._target_labels(target_for_sdf, target_for_colors, target_for_semantics,
                                                     view_matrix, intrinsics, transform)
            locs, sdf_vals, color_vals, sem_vals = sparsify.sparsify_predictions(
                output_sdf, T, empty, output_color, output_semantic, raycaster=self.raycaster, counted=counted)
            output_normals = self._normals(locs, sdf_vals, transform)
            color = (color_vals + 1) * 0.5                                                     # train.py:623
            # prediction raycast + depth L1 + colour L1 + 2D semantic CE (train.py:626-643, 744-746), one kernel pair
            total2d, terms, pred = losses.render_with_2d_losses(
                self.raycaster, locs, sdf_vals, color, output_normals, sem_vals, view_matrix, intrinsics,
                images_depth=sample["images_depth"], images_color=sample["images_color"].permute(0, 2, 3, 1),
                target2d_label=target2d_label, weight_semantic_class=self.class_weight, voxelsize=self.voxelsize,
                weight_depth_loss=self.w["depth"], weight_color_loss=self.w["color"],
                weight_semantic_loss=self.w["semantic"], differentiable_images=self.image_loss is not None)
            loss = loss + total2d
            self.last.update(terms2d=terms.detach())
            if self.image_loss is not None:
                loss_image = self.image_loss(pred, input2d)
                loss = loss + loss_image
                self.last.update(image_loss=loss_image.detach())
        if optimizer is not None:
            loss.backward()                                                                    # train.py:756
            optimizer.step()                                                                   # train.py:757
        return loss.detach()

    def validate(self, sample):
        """The 2D branch of train.py ``test()`` (:870-1275; the losses of :1088-1090, :1193-1196): the step's forward and
        losses without training.  Under ``torch.no_grad()``: the generator forward and dense 3D losses as in ``__call__``,
        the target labels, then the prediction's depth / colour / semantic terms and its confusion matrix against the target
        labels from one ``losses.evaluate_2d`` call -- no input render, normals, ``image_loss`` or backward.  Returns the
        weighted total; ``self.last`` holds ``num_locs``, ``loss_occ``, ``loss_sdf`` and, when the prediction is rendered,
        ``terms2d`` and ``confusion`` ((C+1, C+1) int64, see ``losses.semantic_metrics``).  No parameter's ``.grad`` is
        touched; the generator's train / eval mode is the caller's."""
        lu, T = self.loss_util, self.truncation
        with torch.no_grad():
            inputs, mask, known = sample["input"], sample["mask"], sample.get("known")
            target_for_sdf, target_for_colors = lu.compute_targets(sample["sdf"], T, True, known, sample["colors"])
            dense_region = (torch.autocast("cuda", dtype=torch.bfloat16) if self.autocast_bf16 else contextlib.nullcontext())
            with dense_region:
                output_occ, output_sdf, output_color, output_semantic = self.model(
                    inputs, mask, pred_sdf=[True, True], pred_color=True, pred_semantic=True)
                input_occ = torch.abs(inputs[:, :1]) < (T - 0.01)
                weight = lu.compute_dense_geo_weights(target_for_sdf, input_occ, T, self.weight_surf_geo,
                                                      self.weight_missing_geo)
                empty = torch.sigmoid(output_occ) < 0.5
                weight[empty] = 0
                loss_occ = lu.compute_geo_occ_loss(target_for_sdf, output_occ, known, weight, T)
                loss_sdf = lu.compute_geo_loss(target_for_sdf, None, output_sdf, known, weight, self.logweight_sdf)
                loss = self.w["occ"] * loss_occ + self.w["sdf"] * loss_sdf
            counted = sparsify.count_locs(output_sdf, T, empty)
            n = counted.n
            self.last = dict(num_locs=n, loss_occ=loss_occ, loss_sdf=loss_sdf)
            if 0 < n <= self.raycaster.get_max_num_locs_per_sample() * self.batch_size:
                view_matrix, intrinsics = sample["view_matrix"], sample["images_intrinsic"]
                target2d_label = self._target_labels(target_for_sdf, target_for_colors, sample["semantics"], view_matrix,
                                                     intrinsics, None)
                locs, sdf_vals, color_vals, sem_vals = sparsify.sparsify_predictions(
                    output_sdf, T, empty, output_color, output_semantic, raycaster=self.raycaster, counted=counted)
                total2d, terms, confusion, _ = losses.evaluate_2d(
                    self.raycaster, locs, sdf_vals, (color_vals + 1) * 0.5, sem_vals, view_matrix, intrinsics,
                    images_depth=sample["images_depth"], images_color=sample["images_color"].permute(0, 2, 3, 1),
                    target2d_label=target2d_label, weight_semantic_class=self.class_weight, voxelsize=self.voxelsize,
                    weight_depth_loss=self.w["depth"], weight_color_loss=self.w["color"],
                    weight_semantic_loss=self.w["semantic"])
                loss = loss + total2d
                self.last.update(terms2d=terms, confusion=confusion)
        return loss
