"""State dict (reference key layout, SURVEY.md Appendix A) -> the BN-folded float32 parameter blob that
c4_net_create consumes (layout documented in include/c4b200.h).

Inference always runs in eval() mode (oinkoink/neural/pytorch/model.py:169), so every BatchNorm is an affine map of
its running statistics and folds into the preceding convolution.  The value head's n_fc Linear(42,42) layers have no
activation between them (model.py:83-85), so they are pre-multiplied into one affine map (in float64).
"""
import numpy as np

BN_EPS = 1e-5
MAGIC = 0xC4B2


def _np(sd, k):
    v = sd[k]
    if hasattr(v, "detach"):
        v = v.detach().cpu().numpy()
    return np.asarray(v, dtype=np.float64)


def _fold(sd, conv_w, conv_b, bn):
    w = _np(sd, conv_w)
    scale = _np(sd, bn + ".weight") / np.sqrt(_np(sd, bn + ".running_var") + BN_EPS)
    b = _np(sd, bn + ".bias") - _np(sd, bn + ".running_mean") * scale
    if conv_b is not None:
        b = b + _np(sd, conv_b) * scale
    return w * scale.reshape(-1, *([1] * (w.ndim - 1))), b


def net_shape(sd):
    filters = int(_np(sd, "body.0.0.weight").shape[0])
    n_res = len({k.split(".")[2] for k in sd if k.startswith("body.1.")})
    n_fc = len({k.split(".")[2] for k in sd if k.startswith("value_head.fcN.")})
    return filters, n_res, n_fc


OPERAND_DTYPES = {"fp16": 0, "bf16": 1}


KERNELS = {"auto": 0, "mma": 1, "layers": 2}


def fold_state_dict(sd, operand_dtype="fp16", kernel="auto"):
    """operand_dtype: element type of the tensor-core conv GEMMs (accumulation is always fp32). fp16 is the default
    because bf16 operands miss the 1e-2 parity bound on the reference's trained checkpoint (DESIGN.md)."""
    F, R, n_fc = net_shape(sd)
    # kernel: "auto" = tcgen05/TMEM tower (32 and 64 filters); "mma" forces the mma.sync kernels; "layers" = the
    # layer-by-layer tcgen05 kernels (filters a multiple of 16 in 16..256, 1..40 residual blocks)
    parts = [np.array([MAGIC, F, R, n_fc | (OPERAND_DTYPES[operand_dtype] << 8) | (KERNELS[kernel] << 16)], np.float64)]
    w, b = _fold(sd, "body.0.0.weight", None, "body.0.1")
    parts += [w.reshape(-1), b]
    for i in range(R):
        p = "body.1.%d." % i
        for j in (1, 2):
            w, b = _fold(sd, p + "conv%d.weight" % j, None, p + "batch_norm%d" % j)
            parts += [w.reshape(-1), b]
    w, b = _fold(sd, "value_head.conv1.weight", "value_head.conv1.bias", "value_head.batch_norm")
    parts += [w.reshape(-1), b]
    A = np.eye(42)
    c = np.zeros(42)
    for j in range(n_fc):
        Wj, bj = _np(sd, "value_head.fcN.%d.weight" % j), _np(sd, "value_head.fcN.%d.bias" % j)
        A = Wj @ A
        c = Wj @ c + bj
    parts += [A.reshape(-1), c]
    parts += [_np(sd, "value_head.fc1.weight").reshape(-1), _np(sd, "value_head.fc1.bias").reshape(-1)]
    parts += [_np(sd, "value_head.w1").reshape(-1), _np(sd, "value_head.w2").reshape(-1)]
    w, b = _fold(sd, "policy_head.conv1.weight", "policy_head.conv1.bias", "policy_head.batch_norm")
    parts += [w.reshape(-1), b]
    parts += [_np(sd, "policy_head.fc1.weight").reshape(-1), _np(sd, "policy_head.fc1.bias").reshape(-1)]
    return np.ascontiguousarray(np.concatenate(parts).astype(np.float32))
