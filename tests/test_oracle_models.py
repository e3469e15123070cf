"""Pins oracle/models.py against golden vectors generated from the imported reference
(oracle/gen_golden.py): forward outputs, the loss through RegressionLossEvaluator.__call__, and
parameter gradients (autograd through the restatement vs the reference's autograd)."""
import numpy as np
import pytest
import torch

from oracle import loss as ol
from oracle import models as om
from oracle.gen_golden import SELECTIONS, seeded_inputs, seeded_out_labels
from oracle.seeded import seeded_state_dict, seeded_tensor, strided_sample

ALL = [list(x) for x in SELECTIONS["all"]]


@pytest.fixture(autouse=True)
def _one_cpu_thread():
    """The golden gradients are fp32.  With many threads the CPU GEMMs split the batch reduction, and a near-zero gradient
    entry can land 4e-4 (relative) away from the golden value on a 16-thread host; one thread keeps the summation order
    fixed whatever the host's core count."""
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(n)


def ff_shapes(D, T, s, hidden, fmt, bn):
    F = T // s
    dims = [(3 * D + 12 + 6 * s + 36) * F] + list(hidden) + [2 * 15 * (F if fmt == "all_frames" else 1)]
    shapes, pos = {}, 0
    for i, (h0, h1) in enumerate(zip(dims[:-1], dims[1:])):
        if bn:
            for n, shp in (("weight", (h0,)), ("bias", (h0,)), ("running_mean", (h0,)), ("running_var", (h0,)),
                           ("num_batches_tracked", ())):
                shapes[f"net.{pos}.{n}"] = shp
            pos += 1
        shapes[f"net.{pos}.weight"] = (h1, h0)
        shapes[f"net.{pos}.bias"] = (h1,)
        pos += 1
        if i < len(dims) - 2:
            pos += 1
    return shapes


FF_CASES = {"sigmoid_all": ("sigmoid", "all_frames", False), "relu_last": ("relu", "last_frame", False),
            "tanh_all": ("tanh", "all_frames", False), "sigmoid_bn": ("sigmoid", "all_frames", True)}


@pytest.mark.parametrize("name", list(FF_CASES))
def test_feedforward_golden(golden, name):
    g = golden("ff.npz")
    act, fmt, bn = FF_CASES[name]
    D, T, s, B, seed, iseed, lseed = (int(v) for v in g[f"{name}/meta"])
    hidden = [int(v) for v in g[f"{name}/hidden"]]
    sd = seeded_state_dict(ff_shapes(D, T, s, hidden, fmt, bn), seed)
    params = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v)
              for k, v in sd.items()}
    F = T // s
    Fo = F if fmt == "all_frames" else 1
    inputs = seeded_inputs(B, F, D, s * 3, iseed)
    _, labels = seeded_out_labels(B, Fo, lseed)
    out = om.feedforward_forward(params, inputs, act, Fo, batchnorm=bn)
    for k, v in out.items():
        np.testing.assert_allclose(v.detach().numpy(), g[f"{name}/out/{k}"], rtol=1e-5, atol=1e-6)
    res = ol.regression_loss(out, labels, *ALL)
    np.testing.assert_allclose(float(res["loss"].detach()), float(g[f"{name}/loss"]), rtol=1e-5)
    res["loss"].backward()
    for k, p in params.items():
        if getattr(p, "grad", None) is not None:
            np.testing.assert_allclose(strided_sample(p.grad).numpy(), g[f"{name}/grad_sample/{k}"], rtol=1e-4, atol=1e-7)


@pytest.mark.parametrize("name", ["sigmoid_b16", "relu_b300"])
def test_feedforward_batchnorm_training_golden(golden, name):
    """Oracle BatchNorm1d in TRAINING mode (batch statistics, running-stat update with the unbiased variance) against the
    imported reference: outputs, loss, every parameter gradient and the updated buffers (tests/golden/ff_bn_train.npz)."""
    g = golden("ff_bn_train.npz")
    act = name.split("_")[0]
    D, T, s, B, seed, iseed, lseed = (int(v) for v in g[f"{name}/meta"])
    hidden = [int(v) for v in g[f"{name}/hidden"]]
    sd = seeded_state_dict(ff_shapes(D, T, s, hidden, "all_frames", True), seed)
    params = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v)
              for k, v in sd.items()}
    F = T // s
    inputs = seeded_inputs(B, F, D, s * 3, iseed)
    _, labels = seeded_out_labels(B, F, lseed)
    stats = {}
    out = om.feedforward_forward(params, inputs, act, F, batchnorm=True, training=True, new_stats=stats)
    for k, v in out.items():
        np.testing.assert_allclose(v.detach().numpy(), g[f"{name}/out/{k}"], rtol=2e-4, atol=2e-5)
    res = ol.regression_loss(out, labels, *ALL)
    np.testing.assert_allclose(float(res["loss"].detach()), float(g[f"{name}/loss"]), rtol=1e-5)
    res["loss"].backward()
    for k, p in params.items():
        if getattr(p, "grad", None) is not None:
            want = g[f"{name}/grad_sample/{k}"]
            # bias-like gradients upstream of a training-mode BatchNorm are sums of cancelling terms (even two fp32 CPU
            # evaluations differ by a few % there, e.g. -7.42e-6 vs -7.66e-6): absolute bar from the companion weight gradient
            scale = np.abs(want).max()
            if k.endswith(".bias"):
                scale = max(scale, np.abs(g[f"{name}/grad_sample/{k[:-4]}weight"]).max())
            np.testing.assert_allclose(strided_sample(p.grad).numpy(), want, rtol=2e-3, atol=2e-4 * scale)
    for k, v in stats.items():
        np.testing.assert_allclose(v.numpy(), g[f"{name}/buffer/{k}"], rtol=1e-5, atol=1e-6)


def groundlink_shapes(D=23, J=12, H=10):
    c = [3 * D + 12 + 3 * J + 6 * H, 128, 128, 256, 256]
    shapes = {}
    for i, pos in enumerate((1, 4, 7, 10)):
        shapes[f"cnn.{pos}.weight"] = (c[i + 1], c[i], 7)
        shapes[f"cnn.{pos}.bias"] = (c[i + 1],)
    for pos in (2, 5):
        shapes[f"fc.{pos}.weight"] = (256, 256)
        shapes[f"fc.{pos}.bias"] = (256,)
    shapes["fc.8.weight"] = (30, 256)
    return shapes


@pytest.mark.parametrize("name,fmt", [("all_t50", "all_frames"), ("last_t20", "last_frame")])
def test_groundlink_golden(golden, name, fmt):
    g = golden("groundlink.npz")
    D, J, H, B, T, seed, iseed, lseed = (int(v) for v in g[f"{name}/meta"])
    sd = seeded_state_dict(groundlink_shapes(D, J, H), seed)
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    inputs = seeded_inputs(B, T, D, H * 3, iseed)
    _, labels = seeded_out_labels(B, T if fmt == "all_frames" else 1, lseed)
    out = om.groundlink_forward(params, inputs, fmt)
    for k, v in out.items():
        np.testing.assert_allclose(v.detach().numpy(), g[f"{name}/out/{k}"], rtol=2e-5, atol=2e-6)
    res = ol.regression_loss(out, labels, *ALL)
    np.testing.assert_allclose(float(res["loss"].detach()), float(g[f"{name}/loss"]), rtol=1e-5)
    res["loss"].backward()
    for k, p in params.items():
        np.testing.assert_allclose(strided_sample(p.grad).numpy(), g[f"{name}/grad_sample/{k}"], rtol=2e-4, atol=1e-5)


def transformer_shapes(D=23, T=20, E=30, L=3, ff=60):
    d = 3 * D + 9 + E
    shapes = {"temporal_embedding.embedding.weight": (T, E), "fc.weight": (11, d), "fc.bias": (11,),
              "com_attention.query_linear.weight": (d, d), "com_attention.query_linear.bias": (d,),
              "com_attention.key_linear.weight": (d, d), "com_attention.key_linear.bias": (d,)}
    for l in range(L):
        shapes.update(layer_shapes(d, ff, f"transformer_layers.{l}."))
    return shapes


def layer_shapes(d, ff, p=""):
    return {p + "multihead_attention.in_proj_weight": (3 * d, d), p + "multihead_attention.in_proj_bias": (3 * d,),
            p + "multihead_attention.out_proj.weight": (d, d), p + "multihead_attention.out_proj.bias": (d,),
            p + "feedforward.0.weight": (ff, d), p + "feedforward.0.bias": (ff,),
            p + "feedforward.2.weight": (d, ff), p + "feedforward.2.bias": (d,),
            p + "norm1.weight": (d,), p + "norm1.bias": (d,), p + "norm2.weight": (d,), p + "norm2.bias": (d,)}


@pytest.mark.parametrize("name", ["t20", "t200"])
def test_transformer_golden(golden, name):
    g = golden("transformer.npz")
    D, B, T, seed, iseed = (int(v) for v in g[f"{name}/meta"])
    sd = seeded_state_dict(transformer_shapes(D, T), seed, dtype=torch.float64)
    x = {k: seeded_tensor((B, c, T), iseed + 10 * i, dtype=torch.float64)
         for i, (k, c) in enumerate([("pos", D), ("vel", D), ("acc", D), ("comPos", 3), ("comVel", 3), ("comAcc", 3)])}
    out = om.transformer_forward(sd, x, 3, 3)
    for k in ("contact", "comAcc", "contactForces"):
        np.testing.assert_allclose(out[k].numpy(), g[f"{name}/{k}"], rtol=1e-9, atol=1e-10)


@pytest.mark.parametrize("name", ["d128", "d512"])
def test_denoiser_layer_is_reference_layer(golden, name):
    g = golden("denoiser_layers.npz")
    dm, heads, ff, B, T, seed, xseed, gseed = (int(v) for v in g[f"{name}/meta"])
    sd = seeded_state_dict(layer_shapes(dm, ff), seed)
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    x = seeded_tensor((B, T, dm), xseed).requires_grad_(True)
    y = om.transformer_layer(params, "", x, heads)
    np.testing.assert_allclose(y.detach().numpy(), g[f"{name}/y"], rtol=1e-4, atol=2e-5)
    (y * seeded_tensor((B, T, dm), gseed)).sum().backward()
    np.testing.assert_allclose(x.grad.numpy(), g[f"{name}/dx"], rtol=1e-3, atol=1e-4)
