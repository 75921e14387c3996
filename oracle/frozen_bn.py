"""BatchNorm in evaluation mode under backpropagation ("frozen" BatchNorm), numpy fp64.

Torch7 (THNN / THCUNN BatchNormalization_backward with train == false) differentiates a BatchNorm that normalised with its
running statistics as the fixed per-channel affine it then is:
    gradInput  = gradOutput * gamma * invstd_r,             invstd_r = 1 / sqrt(running_var + eps)
    gradWeight += scale * invstd_r * sum (x - running_mean) * gradOutput
    gradBias   += scale * sum gradOutput
and the running statistics are neither used for a batch mean nor updated.  `bn_backward_eval` states that on NCHW arrays.

`freeze` is the per-module-mode variant of the restated builders (oracle/builders.py): it switches chosen BatchNorm2d modules of
an oracle model to evaluation mode, what bn:evaluate() does inside a Torch7 model in training mode; PyTorch's BatchNorm2d in eval
mode then follows the formulas above under autograd.
"""
import numpy as np
import torch


def bn_forward_eval(x, gamma, beta, running_mean, running_var, eps=1e-5):
    sh = (1, -1, 1, 1)
    invstd = 1.0 / np.sqrt(np.asarray(running_var, np.float64) + eps)
    return (x - np.reshape(running_mean, sh)) * np.reshape(invstd * gamma, sh) + np.reshape(beta, sh)


def bn_backward_eval(x, grad_out, gamma, running_mean, running_var, eps=1e-5, scale=1.0):
    """(gradInput, gradWeight, gradBias) of a BatchNorm in evaluation mode; x, grad_out NCHW"""
    sh = (1, -1, 1, 1)
    invstd = 1.0 / np.sqrt(np.asarray(running_var, np.float64) + eps)
    grad_in = grad_out * np.reshape(np.asarray(gamma, np.float64) * invstd, sh)
    grad_w = scale * invstd * ((x - np.reshape(running_mean, sh)) * grad_out).sum(axis=(0, 2, 3))
    grad_b = scale * grad_out.sum(axis=(0, 2, 3))
    return grad_in, grad_w, grad_b


def batchnorms(model):
    """BatchNorm2d modules of an oracle model in construction order (the order of the product's SpatialBatchNormalization)"""
    return [m for m in model.modules() if isinstance(m, torch.nn.BatchNorm2d)]


def freeze(model, which):
    """evaluation mode for the BatchNorm2d modules of `model` whose construction index is in `which` (the rest keeps its mode)"""
    bns = batchnorms(model)
    for i in which:
        bns[i].eval()
    return [bns[i] for i in which]
