"""Writes tests/golden/reference_graph_kernels.npz and tests/golden/reference_masked_ops.npz: outputs of the reference's
own CUDA extensions, compiled unmodified by oracle/build_ref.py into oracle/_ref/, on the seeded inputs the GPU parity
tests build (tests/helpers.py: REF_GRAPH_CASE, masked_ops_inputs).  Needs a CUDA device.

  ev_graph_cuda  insert_in_queue_cuda + fill_edges_cuda, driven as graph/utils.py:6-23 + ev_graph.py:63-103 do.  The
                 whole edge_index (~0.95 M edges, 15 MB) is too large to store: the fixture keeps the edge count, the SHA-256 of
                 the int64 [2, E] edge_index and every edge of a seeded sample of 500 destination events.
  asy_tools      masked_lin, masked_lin_no_bias, masked_inplace_BN (the rows they write), masked_isdiff.

    python tests/golden/make_reference_kernels_golden.py [OUT_DIR]      # default: next to this file
"""
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
import numpy as np
import torch

from oracle import ref_ops as R
from tests.helpers import REF_GRAPH_CASE, make_inputs, make_model, masked_ops_inputs, sha256

OUT = Path(sys.argv[1]) if len(sys.argv) > 1 else Path(__file__).resolve().parent


def ref_ext(name):
    d = ROOT / "oracle" / "_ref" / name
    if not any(d.glob(f"{name}*.so")):
        raise SystemExit(f"{d}: not built (python oracle/build_ref.py)")
    sys.path.insert(0, str(d))
    return __import__(name)


def graph_fixture():
    ext = ref_ext("ev_graph_cuda")
    c = REF_GRAPH_CASE
    W, H, B, K, Q = c["W"], c["H"], c["B"], c["K"], c["Q"]
    _, args = make_model("n", H, W)
    assert args.max_neighbors == K
    raw, data = make_inputs(B, c["n"], W, H, seed=c["seed"], kind=c["kind"])
    batch_h, pos_h = data.batch.int(), R.denormalize_pos(data.pos, W, H, 1_000_000)
    dev = "cuda"
    batch_i, pos_i = batch_h.to(dev), pos_h.to(dev)
    N = len(batch_i)
    queue = torch.full((B, Q, H, W), -1, dtype=torch.int32, device=dev)
    indices = torch.arange(N, dtype=torch.int32, device=dev)
    lin = pos_i[:, 0] + W * pos_i[:, 1] + W * H * batch_i
    s_lin, s_idx = torch.sort(lin, stable=True)
    uniq, cnt = torch.unique_consecutive(s_lin, return_counts=True)
    queue = ext.insert_in_queue_cuda(indices[s_idx].int().contiguous(), uniq.contiguous(), torch.cumsum(cnt, 0).int().contiguous(), queue)
    edges = torch.full((2, K * N), -1, dtype=torch.int64, device=dev)
    r = int(args.radius * W + 1)
    ext.fill_edges_cuda(batch_i, pos_i, pos_i[:, 2].contiguous(), queue, indices, K, float(r), float(int(args.radius * 1e6)), edges, 0)
    torch.cuda.synchronize()
    ref = edges[:, edges[1] >= 0].cpu()
    oracle = R.RefGraph(W, H, B, K, Q, r, int(args.radius * 1000000)).forward(batch_h, pos_h)
    assert torch.equal(oracle, ref), "oracle/graph_oracle.c disagrees with the reference kernels"
    sample_dst = np.sort(np.random.default_rng(0).choice(N, 500, replace=False))
    keep = torch.from_numpy(np.isin(ref[1].numpy(), sample_dst))
    return dict(inputs_sha256=sha256(batch_h, pos_h), num_edges=ref.shape[1], edges_sha256=sha256(ref),
                sample_dst=sample_dst.astype(np.int32), sample_edges=ref[:, keep].int().numpy())


def masked_ops_fixture():
    ext = ref_ext("asy_tools")
    t = masked_ops_inputs("cuda")
    idx, base = t["idx"], t["base"]
    out = dict(inputs_sha256=sha256(*(t[k] for k in sorted(t))))

    def written_rows(o):
        rest = torch.ones(len(base), dtype=torch.bool, device=o.device)
        rest[idx] = False
        assert torch.equal(o[rest], base[rest])                       # the kernels write the indexed rows only
        return o[idx].cpu().numpy()

    for add in (0, 1):
        o = base.clone()
        ext.masked_lin(idx, t["x"], o, t["w"], t["b"], bool(add))
        out[f"masked_lin_add{add}"] = written_rows(o)
        o = base.clone()
        ext.masked_lin_no_bias(idx, t["x"], o, t["w"], bool(add))
        out[f"masked_lin_no_bias_add{add}"] = written_rows(o)
    o = base.clone()
    ext.masked_inplace_BN(idx, t["xin"], o, t["mean"], t["var"], t["gamma"], t["beta"], 1e-5)
    out["masked_inplace_bn"] = written_rows(o)
    out["masked_isdiff"] = ext.masked_isdiff(idx.clone(), t["a"], t["c"], 1e-8, 1e-5).cpu().numpy()
    return out


if __name__ == "__main__":
    OUT.mkdir(parents=True, exist_ok=True)
    for name, fix in (("reference_graph_kernels", graph_fixture()), ("reference_masked_ops", masked_ops_fixture())):
        np.savez_compressed(OUT / f"{name}.npz", **fix)
        print("wrote", OUT / f"{name}.npz", {k: getattr(v, "shape", v) for k, v in fix.items()})
