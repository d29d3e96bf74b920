"""shared test helpers (tolerances, synthetic inputs, model/oracle construction)."""
import argparse
import copy

import numpy as np

import torch

from dagr_b200.data import EventBatch, format_data, synth_batch
from dagr_b200.utils.args import default_args

# north_star: node features and boxes within 1e-4 relative (fp32).  "relative" is taken against
# |ref| + mean|ref| of the tensor so that exact zeros (ReLU) do not blow up the ratio.
RTOL = 1e-4


def rel_err(a: torch.Tensor, b: torch.Tensor) -> float:
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    if b.numel() == 0:
        assert a.numel() == 0
        return 0.0
    s = b.abs().mean().clamp(min=1e-12)
    return float(((a - b).abs() / (b.abs() + s)).max())


def plain_rel_err(a: torch.Tensor, b: torch.Tensor) -> float:
    """max |a-b|/|b| over the elements with |b| > 1e-3 * mean|b| (plain relative error, no softening term)."""
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    if b.numel() == 0:
        return 0.0
    m = b.abs() > 1e-3 * b.abs().mean().clamp(min=1e-12)
    if not bool(m.any()):
        return 0.0
    return float(((a - b).abs()[m] / b.abs()[m]).max())


# every assert_close call leaves (softened, plain) max relative errors here; tests/conftest.py dumps the table to
# gpurun_out/parity_errors.json at the end of a GPU session (committed copy: profiles/r02_parity_errors.json)
ERROR_LOG = {}


def assert_close(a, b, tol=RTOL, what=""):
    assert a.shape == b.shape, (what, a.shape, b.shape)
    e = rel_err(a, b)
    pe = plain_rel_err(a, b)
    prev = ERROR_LOG.get(what, (0.0, 0.0, 0))
    ERROR_LOG[what] = (max(prev[0], e), max(prev[1], pe), prev[2] + 1)
    assert e <= tol, f"{what}: relative error {e:.3e} > {tol:.1e} (plain relative, |ref| > 1e-3 mean: {pe:.3e})"


def randomize_bn(model, seed=1):
    """BN running stats / affine randomised so that eval-BN is not the identity (SURVEY 8d)."""
    g = torch.Generator().manual_seed(seed)
    for m in model.modules():
        if isinstance(m, (torch.nn.BatchNorm1d, torch.nn.BatchNorm2d)):
            with torch.no_grad():
                m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=g) * 0.1)
                m.running_var.copy_(0.5 + torch.rand(m.running_var.shape, generator=g))
                m.weight.copy_(0.5 + torch.rand(m.weight.shape, generator=g))
                m.bias.copy_(torch.randn(m.bias.shape, generator=g) * 0.1)
    # *_pred biases are zero-initialised: make them non-trivial too
    for n, p in model.named_parameters():
        if n.endswith("bias") and "pred" in n:
            with torch.no_grad():
                p.copy_(torch.randn(p.shape, generator=g) * 0.1)
    return model


def make_model(size="s", height=480, width=640, seed=0, dataset="dsec", **over):
    from dagr_b200.model.dagr import DAGR
    torch.manual_seed(seed)
    args = default_args(size, dataset=dataset, **over)
    model = DAGR(args, height=height, width=width).eval()
    randomize_bn(model, seed + 1)
    return model, args


def make_inputs(B, n_events, width, height, seed=42, kind="uniform", ragged=False, window_us=50_000):
    raw = synth_batch(B, n_events, width, height, seed=seed, kind=kind, ragged=ragged, window_us=window_us)
    data = format_data(raw.clone())
    return raw, data


def golden_weights(model: torch.nn.Module, seed: int):
    """deterministic, non-trivial values for EVERY floating tensor of a state_dict (keys in sorted order, one CPU
    generator): both the reference model and this repo's model are filled by the same rule, so fixtures only store
    inputs and outputs.  BN statistics / affine are kept away from the identity (SURVEY 8d)."""
    sd = model.state_dict()
    g = torch.Generator().manual_seed(int(seed))
    keys = sorted(sd.keys())
    new = {}
    for k in keys:
        t = sd[k]
        if not t.dtype.is_floating_point:
            new[k] = t.clone()
            continue
        shape = tuple(t.shape)
        prefix = k.rsplit(".", 1)[0]
        is_bn = (prefix + ".running_mean") in sd
        if k.endswith("running_var"):
            v = 0.5 + torch.rand(shape, generator=g)
        elif k.endswith("running_mean"):
            v = 0.1 * torch.randn(shape, generator=g)
        elif is_bn and k.endswith("weight"):
            v = 0.5 + torch.rand(shape, generator=g)
        elif len(shape) <= 1:
            v = 0.1 * torch.randn(shape, generator=g)
        else:
            fan = shape[1] if len(shape) == 2 else 2 * shape[1] if len(shape) == 3 else int(np.prod(shape[1:]))
            v = torch.randn(shape, generator=g) / float(np.sqrt(max(fan, 1)))
            if "_pred" in k:                                      # keep exp(wh) of the decode finite
                v = v * 0.1
        new[k] = v.to(t.dtype)
    model.load_state_dict(new, strict=True)
    return float(sum(v.double().abs().sum() for v in new.values() if v.dtype.is_floating_point))


# ------------------------------------------------------------------------------------------------------------------
# fixtures produced by the REFERENCE's own model code (tests/golden/make_reference_forward_golden.py)
# ------------------------------------------------------------------------------------------------------------------
REFERENCE_FIXTURES = ("events_s_320x215", "events_n_ncaltech_240x180", "image_n_240x180")


def load_reference_fixture(name):
    """-> (model on CPU with the fixture's weights, args, data (EventBatch, formatted), expected dict shaped like
    oracle.ref_model.RefModel.forward's output, meta)."""
    from pathlib import Path
    from dagr_b200.model.dagr import DAGR
    f = np.load(Path(__file__).resolve().parent / "golden" / f"reference_forward_{name}.npz")
    W, H, B, seed, use_image = (int(v) for v in f["meta"])
    args = default_args(str(f["size"]), dataset=str(f["dataset"]), batch_size=B, use_image=bool(use_image), img_net="resnet18")
    torch.manual_seed(0)
    model = DAGR(args, height=H, width=W).eval()
    checksum = golden_weights(model, seed)
    # same key set, same shapes, same deterministic rule as the reference's module tree -> same numbers
    assert abs(checksum - float(f["weight_checksum"])) <= 1e-9 * checksum, "state_dict layout differs from the reference's"
    t = lambda k: torch.from_numpy(f[k])
    data = EventBatch(x=t("x"), pos=t("pos"), batch=t("batch").long(), width=torch.full((B,), W), height=torch.full((B,), H),
                      time_window=torch.full((B,), 1_000_000), num_graphs=B)
    if use_image:
        data.image = t("image_u8").float() / 255.0
    nscale = args.num_scales
    exp = dict(edge_index=t("edge_index").long(), x1a=t("x1a"), x1=t("x1"), out3=t("out3"), out4=t("out4"), decoded=t("decoded"),
               levels=[dict(x=t(f"level{i}_x"), pos=t(f"level{i}_pos"), batch=t(f"level{i}_batch").long(),
                            edge_index=t(f"level{i}_edge_index").long(), ambiguous=t(f"level{i}_ambiguous")) for i in range(4)],
               dense=[{nm: t(f"dense_{nm}{k + 1}") for nm in ("cls", "reg", "obj")} for k in range(nscale)],
               detections=[dict(boxes=t(f"det{b}_boxes"), scores=t(f"det{b}_scores"), labels=t(f"det{b}_labels").long()) for b in range(B)])
    return model, args, data, exp, dict(W=W, H=H, B=B, use_image=bool(use_image), num_scales=nscale)


def sha256(*tensors) -> str:
    """hex SHA-256 of the tensors' bytes (C order, dtype as given): pins inputs and outputs too large to store."""
    import hashlib
    h = hashlib.sha256()
    for t in tensors:
        h.update(np.ascontiguousarray(t.detach().cpu().numpy()).tobytes())
    return h.hexdigest()


# ------------------------------------------------------------------------------------------------------------------
# inputs of the comparisons with the reference's own CUDA extensions (fixtures: tests/golden/make_reference_kernels_golden.py)
# ------------------------------------------------------------------------------------------------------------------
# dagr-n, make_inputs(B, n, W, H, seed, kind); K = max_neighbors, Q = max_queue_size of the reference's graph builder
REF_GRAPH_CASE = dict(W=320, H=215, B=2, n=40000, seed=21, kind="clustered", K=16, Q=128)


def masked_ops_inputs(dev):
    """seeded inputs of the masked linear / batch-norm / is-different kernels of the asynchronous path."""
    g = torch.Generator().manual_seed(0)
    Rn, Cin, Cout, K = 500, 18, 64, 77
    t = dict(idx=torch.randperm(Rn, generator=g)[:K], x=torch.randn(Rn, Cin, generator=g), w=torch.randn(Cout, Cin, generator=g),
             b=torch.randn(Cout, generator=g), base=torch.randn(Rn, Cout, generator=g), mean=torch.randn(Cout, generator=g),
             var=torch.rand(Cout, generator=g) + 0.5, gamma=torch.rand(Cout, generator=g) + 0.5, beta=torch.randn(Cout, generator=g),
             xin=torch.randn(Rn, Cout, generator=g), a=torch.rand(Rn, Cin, generator=g) + 0.5)
    idx, a = t["idx"], t["a"]
    c = a.clone()
    c[idx[::3], 3] += 0.5
    a[idx[1], 0] = -2.0; c[idx[1], 0] = -2.0                         # quirk Q3 row
    t["c"] = c
    return {k: v.to(dev) for k, v in t.items()}


def image_branch_cpu(model, data):
    """the dense image trunk + CNN head on the CPU in fp32 (library code on both sides): the tensors the graph path consumes."""
    with torch.no_grad():
        feats, outs = model.backbone.net(data.image.float())
        sizes = model.backbone.get_output_sizes()[-model.head.num_scales:]
        cnn_in = [torch.nn.functional.interpolate(o, size=tuple(sz)) for o, sz in zip(outs[-model.head.num_scales:], sizes)]
        image_outs = model.head.cnn_head(cnn_in)
    return [f.float().contiguous() for f in feats], {k: [t.float().contiguous() for t in v] for k, v in image_outs.items()}
