"""Training-mode BatchNorm for the CPU oracle.  Test infrastructure.

The ``oracle`` package restates the reference's eval-mode forwards.  The reference's notebooks never call ``.eval()``,
so their BatchNorms normalise with the statistics of each call's batch and update the running buffers;
``batch_statistics()`` runs any oracle forward that way without a second copy of it.  Inside the context every
``batchnorm_eval`` the oracle reaches is ``batchnorm_train``, and the state_dict copies its forwards make
(``cast_state_dict``) hand their updated BatchNorm buffers back to the dict they were made from.  So after
``autovc_forward(sd, ...)`` the caller's ``sd`` holds the updated buffers, in the forward's dtype (an fp64 run keeps
fp64 buffers, and the next fp64 call continues from them).  Outside the context the oracle is untouched.
"""
import contextlib

import torch

BN_BUFFERS = ("running_mean", "running_var", "num_batches_tracked")


def batchnorm_train(sd, prefix, x, eps=1e-5, momentum=0.1):
    """``nn.BatchNorm1d`` in training mode.  x: (B, C, L).

    Normalises with the per-channel mean and biased variance over all B x L values, then updates
    ``running_mean``, ``running_var`` (unbiased variance, factor n / (n - 1)) and ``num_batches_tracked`` in ``sd``;
    ``momentum=None`` is the cumulative average 1 / num_batches_tracked.  The buffers are replaced by new tensors, never
    written in place: the dict may share its tensors with a live module."""
    n = x.numel() // x.shape[1]
    if n <= 1:
        raise ValueError(f"Expected more than 1 value per channel when training, got input size {tuple(x.shape)}")
    mean = x.mean(dim=(0, 2))
    var = x.var(dim=(0, 2), unbiased=False)
    w = sd[prefix + ".weight"].view(1, -1, 1)
    b = sd[prefix + ".bias"].view(1, -1, 1)
    y = (x - mean.view(1, -1, 1)) / torch.sqrt(var.view(1, -1, 1) + eps) * w + b
    count = sd[prefix + ".num_batches_tracked"] + 1
    m = 1.0 / float(count) if momentum is None else momentum
    rm, rv = sd[prefix + ".running_mean"], sd[prefix + ".running_var"]
    sd[prefix + ".running_mean"] = (1 - m) * rm + m * mean.to(rm.dtype)
    sd[prefix + ".running_var"] = (1 - m) * rv + m * (var * (n / (n - 1))).to(rv.dtype)
    sd[prefix + ".num_batches_tracked"] = count
    return y


class _WriteBack(dict):
    """A state_dict copy that passes every BatchNorm buffer assigned to it on to the dict it was copied from (which
    may itself be one of these: a forward that calls another forward copies twice)."""

    def __init__(self, items, source):
        super().__init__(items)
        self._source = source

    def __setitem__(self, key, value):
        super().__setitem__(key, value)
        if key.rsplit(".", 1)[-1] in BN_BUFFERS:
            self._source[key] = value


@contextlib.contextmanager
def batch_statistics(momentum=0.1):
    """Run the oracle's forwards with every BatchNorm in training mode (see the module docstring)."""
    import oracle.adain
    import oracle.adjust
    import oracle.autovc
    import oracle.layers
    import oracle.meta

    cast = oracle.layers.cast_state_dict

    def train(sd, prefix, x, eps=1e-5):
        return batchnorm_train(sd, prefix, x, eps, momentum)

    def cast_back(sd, dtype):
        return _WriteBack(cast(sd, dtype), sd)

    # oracle.layers.conv_bn, oracle.meta.conv_bn_relu and oracle.adain.pre_extract are the only BatchNorm call sites
    patches = [(oracle.layers, "batchnorm_eval", train), (oracle.meta, "batchnorm_eval", train),
               (oracle.adain, "batchnorm_eval", train)]
    patches += [(mod, "cast_state_dict", cast_back) for mod in (oracle.autovc, oracle.meta, oracle.adain, oracle.adjust)]
    saved = [(mod, name, getattr(mod, name)) for mod, name, _ in patches]
    try:
        for mod, name, fn in patches:
            setattr(mod, name, fn)
        yield
    finally:
        for mod, name, fn in saved:
            setattr(mod, name, fn)
