"""Drop-in mirrors of the reference's loss-side classes on the warp output (SURVEY.md 8f row f4): the similarity classes of
src/liftreg/layers/losses.py (NCCLoss; NGFLoss, defined here from first principles) and the subspace loss of
src/liftreg/losses/SubspaceLoss.py.

`NCCLoss` is what `losses/SubspaceLoss.py:12` instantiates by its dotted name ('layers.losses.NCCLoss') and what
`networks/RegistrationNet.py:210-212` uses as the validation score; both call it on the warp output.  The reference
module itself cannot be imported without `mermaid` (it imports mermaid.finite_differences at the top); this class needs
only the native library."""
import math

import torch
import torch.nn as nn

from . import ops


class NCCLoss(nn.Module):
    """1 - mean_b NCC(input_b, target_b), reference layers/losses.py:14-29; one fused pass instead of ~10 kernels."""

    def forward(self, input, target):
        loss = ops.ncc_loss(input.reshape(input.shape[0], -1), target.reshape(target.shape[0], -1))
        assert not torch.isnan(loss), 'NCC loss is Nan.'          # losses.py:27
        return loss


class LocalNCCLoss(nn.Module):
    """1 - mean local NCC of VoxelMorph's NCC(win=window) form (ops.local_ncc_loss): the squared correlation of each
    window x window x window neighbourhood, zero padding.  Not in the reference; select it with
    `SubspaceLoss(opt, sim=LocalNCCLoss())` or by its dotted name (`sim_class = "liftreg_b200.losses.LocalNCCLoss"`)."""

    def __init__(self, window=9, eps=1e-5):
        super().__init__()
        self.window = int(window)
        self.eps = float(eps)

    def forward(self, input, target):
        return ops.local_ncc_loss(input, target, self.window, self.eps)


class NGFLoss(nn.Module):
    """1 - mean normalized gradient field similarity (ops.ngf_loss): the squared cosine of the angle between the image
    gradients, regularised by eps, so only edge alignment counts and intensity changes between the images do not.  The
    reference's layers/losses.py names an NGFLoss that is not in its tree, so parity is unpinned.  Select it with
    `SubspaceLoss(opt, sim=NGFLoss())` or by its dotted name (`sim_class = "liftreg_b200.losses.NGFLoss"`); it needs no
    arguments, as `losses/SubspaceLoss.py:12` instantiates it."""

    def __init__(self, eps=1.0, boundary="linear"):
        super().__init__()
        self.eps = float(eps)
        self.boundary = boundary

    def forward(self, input, target):
        return ops.ngf_loss(input, target, self.eps, self.boundary)


class MILoss(nn.Module):
    """-mean_b mutual information of the Parzen joint histogram (ops.mi_loss; Mattes et al. 2003, elastix's default
    metric) over a fixed value range, so a non-linear intensity relation between the images (saturated HU windows,
    density change of the lung between breathing phases) is not penalised.  Not in the reference, so parity is
    unpinned.  Select it with `SubspaceLoss(opt, sim=MILoss())` or by its dotted name
    (`sim_class = "liftreg_b200.losses.MILoss"`); it needs no arguments.  Inputs are flattened per item, as NCCLoss."""

    def __init__(self, num_bins=32, value_range=(-1.0, 1.0)):
        super().__init__()
        self.num_bins = int(num_bins)
        self.value_range = (float(value_range[0]), float(value_range[1]))

    def forward(self, input, target):
        return ops.mi_loss(input.reshape(input.shape[0], -1), target.reshape(target.shape[0], -1), self.num_bins,
                           self.value_range)


def sigmoid_decay(ep, static=5, k=5):
    """reference utils/utils.py:93-107: 1 for the first `static` epochs, then k / (k + exp((ep - static) / k))."""
    if ep < static:
        return float(1.)
    ep = ep - static
    return float(k / (k + math.exp(ep / k)))


def _opt(opt, key, default):
    """The reference reads its settings through mermaid's ParameterDict (`opt[(key, default, doc)]`); a plain dict or
    None works here too."""
    if opt is None:
        return default
    try:
        return opt[(key, default, "")]
    except (KeyError, TypeError):
        return opt.get(key, default) if hasattr(opt, "get") else default


class SubspaceLoss(nn.Module):
    """reference losses/SubspaceLoss.py:9-67 (class `loss`): sim_factor * similarity + reg_factor(epoch) * regulariser.

    The similarity is `NCCLoss` (the reference's default sim_class, :12) and the regulariser the fused
    finite-difference kernel (`ops.diffusion_reg`), both differentiable.  `fd_boundary` selects the face rule of
    mermaid's finite differences ("linear" = FD_torch's default).

    Opt key `fold_factor` (default 0, not in the reference): when > 0, `fold_factor * ops.fold_penalty(phi)` is added to
    the total, with phi = params + identity (the model's `disp_field + id_transform`), and reported as "fold_loss".

    Opt keys `dice_factor` (default 0) and `dice_num_labels` (default 2: background and lung mask), not in the reference:
    when dice_factor > 0, `dice_factor * ops.label_dice_loss(phi, input["source_label"], input["target_label"],
    dice_num_labels)` is added to the total and reported as "dice_loss" (label-supervised training; both label maps
    must be in the input).  phi is formed once when both terms are on."""

    def __init__(self, opt=None, sim=None, fd_boundary="linear"):
        super().__init__()
        self.sim_factor = 1.
        self.sim = sim if sim is not None else NCCLoss()
        self.initial_reg_factor = _opt(opt, 'initial_reg_factor', 10)
        self.min_reg_factor = _opt(opt, 'min_reg_factor', 1e-3)
        self.reg_factor_decay_from = _opt(opt, 'reg_factor_decay_from', 10)
        self.fold_factor = _opt(opt, 'fold_factor', 0)
        self.dice_factor = _opt(opt, 'dice_factor', 0)
        self.dice_num_labels = _opt(opt, 'dice_num_labels', 2)
        self.fd_boundary = fd_boundary
        self._identity = {}

    def forward(self, input):
        if self.dice_factor > 0:          # a missing label map fails before any work is done
            labels = input["source_label"], input["target_label"]
        sim_loss = self.sim(input["warped"], input["target"])
        reg_loss = self.compute_reg_loss(input["params"])
        total_loss = self.sim_factor * sim_loss + self.get_reg_factor(input["epoch"]) * reg_loss
        out = {"total_loss": total_loss, "sim_loss": sim_loss.item(), "reg_loss": reg_loss.item()}
        if self.fold_factor > 0 or self.dice_factor > 0:
            phi = self.deformation_map(input["params"])
        if self.fold_factor > 0:
            fold_loss = ops.fold_penalty(phi, self.fd_boundary)
            out["total_loss"] = out["total_loss"] + self.fold_factor * fold_loss
            out["fold_loss"] = fold_loss.item()
        if self.dice_factor > 0:
            dice_loss = ops.label_dice_loss(phi, *labels, self.dice_num_labels)
            out["total_loss"] = out["total_loss"] + self.dice_factor * dice_loss
            out["dice_loss"] = dice_loss.item()
        return out

    def deformation_map(self, disp):
        """the map disp + identity (the model's `disp_field + id_transform`), with the identity cached per shape and device"""
        key = (tuple(disp.shape[2:]), disp.device)
        if key not in self._identity:
            self._identity[key] = ops.identity_map(disp.shape[2:], disp.device)
        return disp + self._identity[key]

    def get_reg_factor(self, epoch):
        """:40-49"""
        return float(max(sigmoid_decay(epoch, static=self.reg_factor_decay_from, k=2) * self.initial_reg_factor,
                         self.min_reg_factor))

    def compute_reg_loss(self, affine_param):
        """:51-67"""
        return ops.diffusion_reg(affine_param, self.fd_boundary)


loss = SubspaceLoss          # the reference's class name inside losses/SubspaceLoss.py
