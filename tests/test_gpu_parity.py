"""GPU parity suite: hand-written sm_100a kernels (through the C-ABI) against the CPU oracle, and against the
outputs of the reference's own CUDA kernels stored under tests/golden.  Integer results bit-exact; fp32 features
within 1e-4 relative (tests/helpers.py).
"""
from pathlib import Path

import numpy as np
import pytest
import torch

from tests.helpers import (REF_GRAPH_CASE, REFERENCE_FIXTURES, RTOL, assert_close, make_inputs, make_model, masked_ops_inputs,
                           rel_err, sha256)

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
GOLD = ROOT / "tests" / "golden"
DUMP = ROOT / "gpurun_out"


def _run_graph(model, data, B):
    dev = "cuda"
    d = data.clone().cuda()
    batch_i, pos_i, feat, W, H = model._prepare_events(d)
    model.engine.keep_node_features = True
    dec = model.engine.forward_events(batch_i, pos_i, feat, B, W, H)
    torch.cuda.synchronize()
    return dec, batch_i, pos_i


def _oracle_graph(args, W, H, B, batch, pos_i):
    from oracle import ref_ops as R
    g = R.RefGraph(W, H, B, args.max_neighbors, 128, int(args.radius * W + 1), int(args.radius * 1000000))
    return g.forward(batch.cpu().int(), pos_i.cpu())


# ---------------------------------------------------------------------------------------------
def test_denormalize_bit_exact():
    from oracle import ref_ops as R
    model, args = make_model("n", 480, 640)
    raw, data = make_inputs(2, 50000, 640, 480, seed=5)
    d = data.clone().cuda()
    _, pos_i, _, _, _ = model._prepare_events(d)
    ref = R.denormalize_pos(data.pos, 640, 480, 1000000)
    assert torch.equal(pos_i.cpu(), ref)


GRAPH_CASES = [
    # (W, H, B, n_events, kind, ragged, window_us, size)
    (240, 180, 1, 20000, "uniform", False, 50000, "n"),
    (240, 180, 3, 15000, "clustered", True, 50000, "n"),
    (320, 215, 2, 30000, "uniform", False, 50000, "n"),
    (640, 480, 1, 60000, "clustered", False, 50000, "n"),
    (640, 480, 2, 40000, "uniform", True, 20000, "n"),       # denser in time: more K-cap saturation
]


@pytest.mark.parametrize("W,H,B,n,kind,ragged,win,size", GRAPH_CASES)
def test_graph_edges_bit_exact_vs_oracle(W, H, B, n, kind, ragged, win, size):
    model, args = make_model(size, H, W)
    model.cuda()
    raw, data = make_inputs(B, n, W, H, seed=11, kind=kind, ragged=ragged, window_us=win)
    _, batch_i, pos_i = _run_graph(model, data, B)
    mine = model.engine.export_edges().cpu()
    ref = _oracle_graph(args, W, H, B, batch_i, pos_i)
    if not torch.equal(mine, ref):
        DUMP.mkdir(exist_ok=True)
        torch.save(dict(mine=mine, ref=ref, pos=pos_i.cpu(), batch=batch_i.cpu()), DUMP / f"graph_mismatch_{W}x{H}_{B}.pt")
    assert mine.shape == ref.shape, (mine.shape, ref.shape)
    assert torch.equal(mine, ref)


def test_graph_hot_pixel_fifo_depth_and_small_k():
    """> Q events on one pixel: only the newest 128 of the call are visible (ev_graph.cu:201-211)."""
    from dagr_b200.data import EventBatch
    W, H = 240, 180
    model, args = make_model("n", H, W, max_neighbors=6)
    model.cuda()
    n = 400
    g = torch.Generator().manual_seed(0)
    x = torch.randint(100, 104, (n,), generator=g); y = torch.randint(50, 53, (n,), generator=g)
    x[::2] = 101; y[::2] = 51                                  # 200 events on one pixel
    t = torch.sort(torch.randint(990000, 999999, (n,), generator=g)).values
    pos_denorm = torch.stack([x, y, t], 1).int()
    data = EventBatch(x=torch.ones(n, 1), pos=torch.zeros(n, 3), batch=torch.zeros(n, dtype=torch.long),
                      width=torch.tensor([W]), height=torch.tensor([H]), time_window=torch.tensor([1000000]),
                      pos_denorm=pos_denorm, num_graphs=1)
    _, batch_i, pos_i = _run_graph(model, data, 1)
    mine = model.engine.export_edges().cpu()
    ref = _oracle_graph(args, W, H, 1, batch_i, pos_i)
    assert torch.equal(mine, ref)
    deg = torch.bincount(mine[1], minlength=n)
    assert int(deg.max()) == 6


def test_dense_voxel_falls_back_to_global_probe_and_split_path_agrees():
    """> BL_CAP staged records around one voxel exercises the global-memory fallback of the fused build
    kernel; the v1 split kernels (graph_search + l1_conv_a) must give the same adjacency and features."""
    from dagr_b200.data import EventBatch
    W, H = 640, 480
    model, args = make_model("n", H, W)
    model.cuda()
    g = torch.Generator().manual_seed(3)
    n_dense, n_bg = 9000, 20000
    x = torch.cat([torch.randint(300, 330, (n_dense,), generator=g), torch.randint(0, W, (n_bg,), generator=g)])
    y = torch.cat([torch.randint(200, 230, (n_dense,), generator=g), torch.randint(0, H, (n_bg,), generator=g)])
    n = n_dense + n_bg
    t = torch.sort(torch.randint(950000, 999999, (n,), generator=g)).values
    perm = torch.randperm(n, generator=g)
    pos_denorm = torch.stack([x[perm], y[perm], t], 1).int()
    p = (torch.randint(0, 2, (n,), generator=g) * 2 - 1).float().view(-1, 1)
    data = EventBatch(x=p, pos=torch.zeros(n, 3), batch=torch.zeros(n, dtype=torch.long), width=torch.tensor([W]),
                      height=torch.tensor([H]), time_window=torch.tensor([1000000]), pos_denorm=pos_denorm, num_graphs=1)
    eng = model.engine
    eng.fused_build = True
    dec_f, batch_i, pos_i = _run_graph(model, data, 1)
    e_f = eng.export_edges().cpu()
    N = eng.last["N"]
    nbr_f = eng.last["ws"]["nbr"][:16 * N].clone(); xa_f = eng.xa_rows().clone(); dec_f = dec_f.clone()
    mask_f = eng.last["grids"][0].mask.clone()
    eng.fused_build = False
    dec_s, _, _ = _run_graph(model, data, 1)
    eng.fused_build = True
    assert torch.equal(e_f, eng.export_edges().cpu())
    assert torch.equal(e_f, _oracle_graph(args, W, H, 1, batch_i, pos_i))
    deg = nbr_f[15 * N:16 * N]
    assert torch.equal(deg, eng.last["ws"]["nbr"][15 * N:16 * N])
    assert torch.equal(mask_f, eng.last["grids"][0].mask)
    assert_close(xa_f.cpu(), eng.xa_rows().cpu(), tol=1e-5, what="fused vs split conv_a")
    assert_close(dec_f.cpu(), dec_s.cpu(), tol=1e-5, what="fused vs split decoded")


def test_events_not_time_sorted_still_bit_exact():
    """the input contract says events are time-sorted per sample; if they are not, the build kernel must
    notice (flag from the sort) and drop its time-bucket pruning instead of returning different edges."""
    from dagr_b200.data import EventBatch
    W, H, n = 240, 180, 12000
    model, args = make_model("n", H, W)
    model.cuda()
    g = torch.Generator().manual_seed(9)
    x = torch.randint(0, W, (n,), generator=g); y = torch.randint(0, H, (n,), generator=g)
    t = torch.randint(950000, 999999, (n,), generator=g)               # NOT sorted
    data = EventBatch(x=torch.ones(n, 1), pos=torch.zeros(n, 3), batch=torch.zeros(n, dtype=torch.long),
                      width=torch.tensor([W]), height=torch.tensor([H]), time_window=torch.tensor([1000000]),
                      pos_denorm=torch.stack([x, y, t], 1).int(), num_graphs=1)
    _, batch_i, pos_i = _run_graph(model, data, 1)
    assert torch.equal(model.engine.export_edges().cpu(), _oracle_graph(args, W, H, 1, batch_i, pos_i))


def test_graph_empty_and_single_event():
    from dagr_b200.data import EventBatch
    W, H = 240, 180
    model, args = make_model("n", H, W, dataset="ncaltech101")
    model.cuda()
    for n in (0, 1):
        data = EventBatch(x=torch.ones(n, 1), pos=torch.rand(n, 3) * 0.99, batch=torch.zeros(n, dtype=torch.long),
                          width=torch.tensor([W]), height=torch.tensor([H]), time_window=torch.tensor([1000000]), num_graphs=1)
        dec, _, _ = _run_graph(model, data, 1)
        e = model.engine.export_edges().cpu()
        assert e.shape == (2, n)
        assert torch.isfinite(dec).all() and dec.shape == (1, 35, 105)
        out = model(data.clone().cuda())
        assert len(out[0]) == 1


def _assert_reference_graph_edges(e, gold, who):
    """edge_index int64[2, E] == the reference kernels' (tests/golden/reference_graph_kernels.npz): every edge of the
    stored sample of destination events, then the edge count and the SHA-256 of the whole edge_index."""
    e = e.cpu().long()
    keep = torch.from_numpy(np.isin(e[1].numpy(), gold["sample_dst"]))
    assert torch.equal(e[:, keep], torch.from_numpy(gold["sample_edges"]).long()), f"{who}: edges of the sampled events"
    assert e.shape[1] == int(gold["num_edges"]), (who, e.shape[1], int(gold["num_edges"]))
    assert sha256(e) == str(gold["edges_sha256"]), f"{who}: edge_index differs from the reference kernels'"


def test_graph_vs_reference_cuda_kernels():
    """our edge_index == the reference's own insert_in_queue_cuda + fill_edges_cuda on the same events (fixture made by
    tests/golden/make_reference_kernels_golden.py)."""
    gold = np.load(GOLD / "reference_graph_kernels.npz")
    c = REF_GRAPH_CASE
    W, H, B = c["W"], c["H"], c["B"]
    model, args = make_model("n", H, W)
    model.cuda()
    raw, data = make_inputs(B, c["n"], W, H, seed=c["seed"], kind=c["kind"])
    _, batch_i, pos_i = _run_graph(model, data, B)
    assert sha256(batch_i.int(), pos_i.int()) == str(gold["inputs_sha256"]), "events differ from the ones the fixture was made from"
    _assert_reference_graph_edges(model.engine.export_edges(), gold, "CUDA path")
    # and the C oracle agrees with the reference kernels too (pins oracle/graph_oracle.c)
    _assert_reference_graph_edges(_oracle_graph(args, W, H, B, batch_i, pos_i), gold, "C oracle")


# ---------------------------------------------------------------------------------------------
FWD_CASES = [
    (1280, 720, 1, 60000, "clustered", "n", "dsec"),          # r = 13 px: cell walk instead of the ring walk (tiles wider than 32 px)
    (240, 180, 1, 6000, "uniform", "n", "ncaltech101"),
    (320, 215, 2, 12000, "clustered", "s", "dsec"),
    (640, 480, 2, 25000, "uniform", "s", "dsec"),
    (320, 215, 1, 8000, "clustered", "l", "dsec"),            # widest variant: C = 128 (Cin 130 at the coarse levels)
    (240, 180, 2, 5000, "uniform", "m", "dsec"),
]


def _pos_hints(L):
    """the product's rounded pooled positions per level (normalised), handed to the oracle for the voxels the oracle
    itself flags as ambiguous (mean within float noise of a pixel boundary; the reference's fp32 atomic mean is not
    run-to-run stable there, SURVEY H3b) so that the comparison continues below such a voxel."""
    from dagr_b200 import export
    geom = L["geom"]
    return [export.grid_nodes(L["grids"][lv], geom.levels[lv], geom)["pos"].cpu() for lv in range(4)]


def _run_product(model, data, B, H, W, image_feats=None, image_outs=None, image=False):
    eng = model.engine
    eng.keep_node_features = True
    d = data.clone().cuda()
    if image:
        dec = model.forward_decoded(d)
    else:
        batch_i, pos_i, feat, _, _ = model._prepare_events(d)
        dec = eng.forward_events(batch_i, pos_i, feat, B, W, H, image_feats=image_feats, image_outs=image_outs)
    torch.cuda.synchronize()
    return dec.clone()


def _compare_with(model, dec, o, hinted=True, dense=True):
    """product state of the last forward vs an expected dict shaped like RefModel.forward's output (the oracle's, or a
    fixture produced by the reference's own code): edges bit-exact, per-event activations, every pooled level (node sets,
    batch, rounded positions, coarse edges bit-exact; features 1e-4), out3/out4, dense head maps, decoded outputs."""
    from dagr_b200 import export
    eng = model.engine
    L = eng.last
    N = L["N"]
    mine = eng.export_edges().cpu()
    assert mine.shape == o["edge_index"].shape, (mine.shape, o["edge_index"].shape)
    assert torch.equal(mine, o["edge_index"])
    perm = L["ws"]["perm"]
    assert_close(export.unsort_rows(eng.xa_rows(), perm, N).cpu(), o["x1a"], what="conv_block1.conv_block1 output")
    assert_close(export.unsort_rows(L["x1"], perm, N).cpu(), o["x1"], what="conv_block1 output")
    geom = L["geom"]
    for lv in range(4):
        gs, level, pl = L["grids"][lv], geom.levels[lv], o["levels"][lv]
        nodes = export.grid_nodes(gs, level, geom)
        assert len(nodes["cell"]) == pl["x"].shape[0], f"level {lv}: node count"
        assert torch.equal(nodes["batch"].cpu(), pl["batch"]), f"level {lv}: batch"
        same = (nodes["pos"].cpu() == pl["pos"][:, :2]).all(1)
        if hinted:
            # ambiguous voxels adopted the product's position in the oracle (pos_hints): everything is bit-exact
            assert bool(same.all()), f"level {lv}: rounded positions"
        else:
            assert bool(same[~pl["ambiguous"]].all()), f"level {lv}: rounded positions"
        assert torch.equal(export.grid_edges(gs, level).cpu(), pl["edge_index"]), f"level {lv}: coarse edge_index"
        assert_close(nodes["x"].cpu(), pl["x"], what=f"level {lv} pooled features")
        if not bool(same.all()):
            # a static fixture cannot adopt the product's position at a voxel whose mean lies within float noise of a
            # pixel boundary (flagged by the oracle when the fixture was made): levels below it are not comparable
            print(f"level {lv}: {int((~same).sum())} oracle-flagged ambiguous voxel(s) rounded differently; stopping the comparison here")
            return False
    assert_close(L["inter"]["o4"][L["grids"][2].cnt[:L["grids"][2].cells] > 0].cpu(), o["out3"], what="out3")
    assert_close(L["inter"]["o5"][L["grids"][3].cnt[:L["grids"][3].cells] > 0].cpu(), o["out4"], what="out4")
    if dense:
        for k, dd in enumerate(L["dense"]):
            for name in ("cls", "reg", "obj"):
                assert_close(dd[name].cpu(), o["dense"][k][name], what=f"dense {name}{k + 1}")
    assert_close(dec.cpu(), o["decoded"], what="decoded outputs")
    return True


def _check_forward(model, args, data, B, H, W, image=False, mirror_t_quirk=True, check_public=True):
    """one forward against the oracle run on the same inputs (see _compare_with) + the detections of the public forward."""
    from oracle.ref_model import RefModel
    dec = _run_product(model, data, B, H, W, image=image)
    L = model.engine.last
    ref = RefModel({k: v.cpu() for k, v in model.state_dict().items()}, args, H, W)
    kw = {}
    if image:
        kw = dict(image_feats=[f.cpu() for f in model.last_image_feats],
                  image_outs={k: [t.cpu() for t in v] for k, v in model.last_image_outs.items()})
    o = ref.forward(data.x, data.pos, data.batch, B, pos_hints=_pos_hints(L), mirror_t_quirk=mirror_t_quirk, **kw)
    assert _compare_with(model, dec, o, hinted=True)
    if not check_public:
        return o
    # detections through the public forward
    dets = model(data.clone().cuda())[0]
    _assert_same_detections(dets, o["detections"], B)
    return o


def _assert_same_detections(dets, ref, B):
    """same detection SET per image (boxes / scores 1e-4, labels equal).  Both sides list detections by descending score;
    candidates whose scores differ by less than fp32 noise may swap places, so rows are matched by nearest box first."""
    assert len(dets) == B
    for b in range(B):
        rb = ref[b]
        n = len(rb["boxes"])
        assert len(dets[b]["boxes"]) == n, f"image {b}: #detections {len(dets[b]['boxes'])} vs {n}"
        if n == 0:
            continue
        mine = torch.cat([dets[b]["boxes"].cpu().float(), dets[b]["scores"].cpu().float().view(-1, 1)], 1)
        want = torch.cat([rb["boxes"].float(), rb["scores"].float().view(-1, 1)], 1)
        scale = want.abs().amax(0, keepdim=True).clamp(min=1e-6)
        cost = ((mine[None] - want[:, None]) / scale).abs().amax(-1)          # [n_ref, n_mine]
        pick = cost.argmin(1)
        assert len(set(pick.tolist())) == n, f"image {b}: detections do not match one to one"
        assert int((pick != torch.arange(n)).sum()) <= n // 4 + 2, f"image {b}: score order differs beyond near-ties"
        assert torch.equal(dets[b]["labels"].cpu()[pick], rb["labels"])
        assert_close(mine[pick, :4], want[:, :4], what="boxes")
        assert_close(mine[pick, 4], want[:, 4], what="scores")


@pytest.mark.parametrize("W,H,B,n,kind,size,dataset", FWD_CASES)
def test_forward_parity_vs_oracle(W, H, B, n, kind, size, dataset):
    model, args = make_model(size, H, W, dataset=dataset)
    model.cuda()
    raw, data = make_inputs(B, n, W, H, seed=31, kind=kind, ragged=True)
    _check_forward(model, args, data, B, H, W)


@pytest.mark.parametrize("name", REFERENCE_FIXTURES)
def test_cuda_path_equals_the_references_own_forward(name):
    """tests/golden/reference_forward_*.npz: outputs of the reference's UNMODIFIED DAGR.forward (its own net.py, dagr.py,
    pooling.py, spline_conv.py LUT path, model/utils.py post-processing with torchvision NMS; third-party packages
    stood in for by tests/golden/ref_shim.py).  No oracle code runs in this test."""
    from tests.helpers import image_branch_cpu, load_reference_fixture
    model, args, data, exp, meta = load_reference_fixture(name)
    W, H, B = meta["W"], meta["H"], meta["B"]
    feats = outs = None
    if meta["use_image"]:
        feats, outs = image_branch_cpu(model, data)                     # dense trunk: fp32 on the CPU, as upstream ran it
        feats = [f.cuda() for f in feats]
        outs = {k: [t.cuda() for t in v] for k, v in outs.items()}
    model.cuda()
    dec = _run_product(model, data, B, H, W, image_feats=feats, image_outs=outs)
    complete = _compare_with(model, dec, exp, hinted=False, dense=not meta["use_image"])
    if complete:
        det, ndet = model.engine.postprocess(dec.clone(), model.conf_threshold, model.nms_threshold, W, H)
        torch.cuda.synchronize()
        dets = [dict(boxes=det[b, :int(ndet[b]), :4], scores=det[b, :int(ndet[b]), 4], labels=det[b, :int(ndet[b]), 5].long()) for b in range(B)]
        _assert_same_detections(dets, exp["detections"], B)


# the BENCHMARKED regime (BASELINE.json configs[1]: dagr-s, 640x480, 300k events per sample in a 50 ms window): mean
# degree ~15.4 with the K cap saturated almost everywhere, > 160 events per pool1 voxel (multi-chunk loops of the
# per-voxel kernels), multi-record pixels; the clustered stream adds voxels beyond the staging capacities
# (BL_CAP / CB2_CAP -> global-memory fallbacks) and low-degree noise events.
FULL_DENSITY_CASES = [
    # B, stream, seed, Engine.dense_worklists
    (1, "uniform", 2042, "auto"),         # one sample of the bench batch (bench.py seed 42 + 1000 * 2)
    (1, "clustered", 2042, False),        # over-capacity voxels: global-memory fallback inside the per-voxel kernels
    (1, "clustered", 2042, True),         # ... queued for the persistent dense kernels
    (2, "uniform", 2052, "auto"),
]


@pytest.mark.parametrize("B,kind,seed,dense", FULL_DENSITY_CASES)
def test_full_density_forward_parity_vs_oracle(B, kind, seed, dense):
    W, H, n = 640, 480, 300000
    model, args = make_model("s", H, W, batch_size=B)
    model.cuda()
    model.engine.dense_worklists = dense
    raw, data = make_inputs(B, n, W, H, seed=seed, kind=kind)
    _check_forward(model, args, data, B, H, W)
    N = model.engine.last["N"]
    deg = model.engine.last["ws"]["nbr"][15 * N:16 * N].float()
    if kind == "uniform":
        assert float(deg.mean()) > 13.0                       # the K cap (15 neighbours + self loop) is hit almost everywhere
    else:
        hdr = model.engine._zs(model.engine.last["ws"], "wl_hdr", torch.int32).cpu()
        assert int(hdr[0]) > 100 and int(hdr[4]) > 100        # this stream really has voxels beyond both staging capacities
    if dense == "auto" and kind == "uniform":
        assert model.engine._dense_policy(model.engine.last["ws"], None, False) == [0, 0, 0]


def test_last_event_at_t_equals_T_quirk_h3a():
    """Quirk Q1 / H3a (dsec_data.py:145, pooling.py:31,56): real DSEC windows end with an event at normalised t == 1.0,
    which torch_cluster.grid_cluster puts into temporal cell 1 of a one-cell axis, so in the reference it aliases into the
    NEXT sample's voxel (or a phantom voxel behind the last sample).  The graph build does not care (edges stay
    bit-exact).  The kernels key voxels by (batch, y, x) only, i.e. they keep the event in its own sample's voxel: the
    forward equals the oracle with the quirk switched off, and the oracle with the quirk on differs (documented gap)."""
    from dagr_b200.data import EventBatch
    from oracle.ref_model import RefModel
    W, H, B, T = 320, 215, 2, 1_000_000
    model, args = make_model("s", H, W, batch_size=B)
    model.cuda()
    raw, data = make_inputs(B, 9000, W, H, seed=77, kind="uniform")
    pos = data.pos.clone()
    for b in range(B):
        last = int(torch.nonzero(data.batch == b).flatten()[-1])
        pos[last, 2] = 1.0                                        # t == T exactly (dsec_data.py:145)
    d = EventBatch(x=data.x, pos=pos, batch=data.batch, width=data.width, height=data.height, time_window=data.time_window, num_graphs=B)
    o = _check_forward(model, args, d, B, H, W, mirror_t_quirk=False)
    ref = RefModel({k: v.cpu() for k, v in model.state_dict().items()}, args, H, W)
    q = ref.forward(d.x, d.pos, d.batch, B, mirror_t_quirk=True)
    assert torch.equal(q["edge_index"], o["edge_index"])
    # with the quirk the last event of the last sample lands in a phantom voxel behind the batch
    assert q["levels"][0]["x"].shape[0] == o["levels"][0]["x"].shape[0] + 1


@pytest.mark.parametrize("W,H,B,n,size,img_net", [(240, 180, 2, 5000, "n", "resnet18"), (320, 215, 1, 9000, "s", "resnet18"),
                                                  (640, 480, 2, 40000, "s", "resnet50")])       # the last one: config 3's shape
def test_image_fusion_parity_vs_oracle(W, H, B, n, size, img_net):
    """use_image: sampled ResNet features enter every Layer input and every pooling, CNN head maps are added to the
    dense outputs.  The dense trunk is torch/cuDNN on both sides (its tensors are handed to the oracle)."""
    from dagr_b200.data import format_data, synth_batch
    model, args = make_model(size, H, W, use_image=True, img_net=img_net, batch_size=B)
    model.cuda()
    raw = synth_batch(B, n, W, H, seed=77, kind="clustered", with_image=True, ragged=True)
    data = format_data(raw.clone())
    _check_forward(model, args, data, B, H, W, image=True, check_public=False)


@pytest.mark.parametrize("W,H,B,n,chunks,kto", [(240, 180, 1, 8000, [7999, 1], False), (640, 480, 2, 30000, [0.5, 0.2, 0.2, 0.1], False),
                                                  (320, 215, 1, 12000, [0.4, 0.3, 0.3], True)])
def test_async_incremental_equals_dense(W, H, B, n, chunks, kto):
    """the reference's own invariant (evaluate_flops.py:90,139-147): init on N-1 events + 1-event update == dense
    forward on N events; generalised to several chunks and to B > 1 (tolerance 1e-5 instead of 1e-3)."""
    from dagr_b200.asynchronous import AsyncDAGR
    from dagr_b200.data import EventBatch
    from dagr_b200 import export
    model, args = make_model("n", H, W, keep_temporal_ordering=kto)
    model.cuda()
    raw, data = make_inputs(B, n, W, H, seed=5, kind="clustered")
    dense, _, _ = _run_graph(model, data, B)
    dense = dense.clone()
    g_dense = [export.grid_nodes(model.engine.last["grids"][lv], model.engine.last["geom"].levels[lv], model.engine.last["geom"]) for lv in range(2)]
    g_dense = [dict(x=g["x"].clone(), pos=g["pos"].clone(), cell=g["cell"].clone()) for g in g_dense]
    e_dense = export.grid_edges(model.engine.last["grids"][0], model.engine.last["geom"].levels[0]).clone()

    # split every sample's (time-sorted) events into the same fractions
    per_sample = [torch.nonzero(data.batch == b).flatten() for b in range(B)]
    bounds = []
    for idx in per_sample:
        if isinstance(chunks[0], float):
            cuts = (torch.tensor([0.0] + list(chunks)).cumsum(0) * len(idx)).long()
            cuts[-1] = len(idx)
        else:
            cuts = torch.tensor([0] + list(chunks)).cumsum(0).clamp(max=len(idx))
            cuts[-1] = len(idx)
        bounds.append(cuts)
    a = AsyncDAGR(model)
    dec = None
    for c in range(len(chunks)):
        sel = torch.cat([per_sample[b][bounds[b][c]:bounds[b][c + 1]] for b in range(B)])
        chunk = EventBatch(x=data.x[sel], pos=data.pos[sel], batch=data.batch[sel], width=data.width, height=data.height,
                           time_window=data.time_window, num_graphs=B)
        dec = a.step_decoded(chunk.cuda(), batch_size=B)
    torch.cuda.synchronize()
    L = model.engine.last
    for lv in range(2):
        g = export.grid_nodes(L["grids"][lv], L["geom"].levels[lv], L["geom"])
        assert torch.equal(g["cell"], g_dense[lv]["cell"]) and torch.equal(g["pos"], g_dense[lv]["pos"])
        assert_close(g["x"], g_dense[lv]["x"], tol=1e-5, what=f"async level {lv} features")
    assert torch.equal(export.grid_edges(L["grids"][0], L["geom"].levels[0]), e_dense)
    assert_close(dec, dense, tol=1e-5, what="async decoded vs dense")
    # sliding window: evict the oldest 20 ms and compare with the dense forward on the live window
    t_cut = 970000
    dec_live = a.evict_older_than(t_cut).clone()
    keep = (model._prepare_events(data.clone().cuda())[1][:, 2] >= t_cut).cpu()
    live = EventBatch(x=data.x[keep], pos=data.pos[keep], batch=data.batch[keep], width=data.width, height=data.height,
                      time_window=data.time_window, num_graphs=B)
    dense_live, _, _ = _run_graph(model, live, B)
    assert a.num_events == int(keep.sum())
    assert_close(dec_live, dense_live, tol=1e-5, what="live window after eviction vs dense")


def test_forward_vs_committed_golden_fixture():
    """the committed oracle fixture (tests/golden/forward_dagr_n_240x180.pt): no oracle code runs here."""
    from dagr_b200 import export
    from dagr_b200.data import EventBatch
    fix = torch.load(ROOT / "tests" / "golden" / "forward_dagr_n_240x180.pt")
    m = fix["meta"]
    model, args = make_model(m["size"], m["H"], m["W"], seed=m["model_seed"])
    model.cuda()
    data = EventBatch(x=fix["x"], pos=fix["pos"], batch=fix["batch"], width=torch.full((m["B"],), m["W"]),
                      height=torch.full((m["B"],), m["H"]), time_window=torch.full((m["B"],), 1000000), num_graphs=m["B"])
    dec, _, _ = _run_graph(model, data, m["B"])
    eng, L = model.engine, model.engine.last
    assert torch.equal(eng.export_edges().cpu().int(), fix["edge_index"])
    N = L["N"]
    assert_close(export.unsort_rows(eng.xa_rows(), L["ws"]["perm"], N).cpu(), fix["x1a"], what="golden x1a")
    assert_close(export.unsort_rows(L["x1"], L["ws"]["perm"], N).cpu(), fix["x1"], what="golden x1")
    for lv in range(4):
        nodes = export.grid_nodes(L["grids"][lv], L["geom"].levels[lv], L["geom"])
        amb = fix["level_ambiguous"][lv]
        same = nodes["pos"].cpu() == fix["level_pos"][lv]
        assert torch.equal(nodes["batch"].cpu().int(), fix["level_batch"][lv]) and bool(same[~amb].all())
        if not bool(same.all()):
            break
        assert torch.equal(export.grid_edges(L["grids"][lv], L["geom"].levels[lv]).cpu().int(), fix["level_edges"][lv])
        if lv < 2:
            assert_close(nodes["x"].cpu(), fix["level_x"][lv], what=f"golden level {lv}")
    else:
        assert_close(dec.cpu(), fix["decoded"], what="golden decoded")
        dets = model(data.clone().cuda())[0]
        assert [len(d["boxes"]) for d in dets] == fix["n_det"]


def test_keep_temporal_ordering_filters_coarse_edges_like_the_reference():
    """--keep_temporal_ordering (pooling.py:69-72): coarse edges survive only if t_max[dst] > t_max[src]."""
    W, H, B = 240, 180, 2
    model, args = make_model("n", H, W, keep_temporal_ordering=True, batch_size=B)
    model.cuda()
    raw, data = make_inputs(B, 4000, W, H, seed=17, kind="clustered")
    _check_forward(model, args, data, B, H, W)


def test_interframe_growing_windows_like_run_test_interframe():
    """scripts/run_test_interframe.py:83-86: synchronous forward on windows num_us = linspace(0, 50000, steps), first one empty."""
    from dagr_b200.data import EventBatch
    W, H, B = 320, 215, 2
    model, args = make_model("s", H, W)
    model.cuda()
    raw, data = make_inputs(B, 20000, W, H, seed=23, kind="uniform")
    t_us = (data.pos[:, 2].double() * 1e6).round()
    counts = []
    for n_us in np.linspace(0, 50000, 5):
        m = t_us < (950000 + n_us)
        d = EventBatch(x=data.x[m], pos=data.pos[m], batch=data.batch[m], width=data.width, height=data.height,
                       time_window=data.time_window, num_graphs=B)
        dets = model(d.cuda())[0]
        assert len(dets) == B and all(torch.isfinite(x["boxes"]).all() for x in dets)
        counts.append(int(m.sum()))
    assert counts[0] == 0 and counts[-1] == len(t_us)


def test_overlapped_steps_equal_serial_steps():
    """Engine.overlap / PipelinedDetector: coarse stack + NMS of step i on a side stream while step i+1's event-level
    kernels run.  Different inputs in flight back to back must give bit-identical results to the serial forward."""
    from dagr_b200.pipeline import PipelinedDetector
    W, H, B = 320, 215, 2
    model, args = make_model("s", H, W)
    model.cuda()
    datas = [make_inputs(B, n, W, H, seed=31 + k, kind="uniform")[1].cuda() for k, n in enumerate([15000, 9000, 20000, 12000, 15000, 7000])]
    serial = []
    for d in datas:
        dec = model.forward_decoded(d)
        det, ndet = model.engine.postprocess(dec, model.conf_threshold, model.nms_threshold, W, H)
        torch.cuda.synchronize()
        serial.append((dec.clone(), det.clone(), ndet.clone()))
    eng = model.engine
    eng.overlap = True
    got = []
    for rep in range(2):                                   # second round replays the captured per-slot graphs
        got = []
        for d in datas:
            dec = model.forward_decoded(d)
            det, ndet = eng.postprocess(dec, model.conf_threshold, model.nms_threshold, W, H)
            with eng.result_stream():                      # consume on the producing stream, as bench.py's all-gather does
                got.append((dec.clone(), det.clone(), ndet.clone()))
        eng.join()
        torch.cuda.synchronize()
        for k, ((d0, t0, n0), (d1, t1, n1)) in enumerate(zip(serial, got)):
            assert torch.equal(d0, d1), f"decoded differs at step {k} (round {rep})"
            assert torch.equal(n0, n1)
            for b in range(B):
                assert torch.equal(t0[b, :int(n0[b])], t1[b, :int(n1[b])])
    eng.overlap = False
    # public pipelined API == drop-in synchronous call
    pd = PipelinedDetector(model)
    want = [model(d)[0] for d in datas]
    handles, res = [], []
    h_prev = None
    for d in datas:
        h = pd.submit(d)
        if h_prev is not None:
            res.append(h_prev.result())
        h_prev = h
    res.append(h_prev.result())
    for w, r in zip(want, res):
        for b in range(B):
            assert torch.equal(w[b]["boxes"].cpu(), r[b]["boxes"]) and torch.equal(w[b]["scores"].cpu(), r[b]["scores"])
            assert torch.equal(w[b]["labels"].cpu(), r[b]["labels"])


def test_batch_independence_and_full_size_properties():
    """config-2 shape (640x480, B=8, 300k events/sample): size-independent properties."""
    W, H, B, n = 640, 480, 8, 300000
    model, args = make_model("s", H, W)
    model.cuda()
    raw, data = make_inputs(B, n, W, H, seed=42, kind="uniform")
    dec, batch_i, pos_i = _run_graph(model, data, B)
    e = model.engine.export_edges()
    N = len(batch_i)
    src, dst = e[0], e[1]
    assert bool((dst[1:] >= dst[:-1]).all()) and bool((src <= dst).all())          # ev_tgn.py:53-55
    deg = torch.bincount(dst, minlength=N)
    assert int(deg.max()) <= args.max_neighbors and int(deg.min()) >= 1
    assert bool((batch_i[src] == batch_i[dst]).all())
    d = pos_i[dst] - pos_i[src]
    r = int(args.radius * W + 1)
    assert int(d[:, :2].abs().max()) <= r and int(d[:, 2].min()) >= 0 and int(d[:, 2].max()) <= int(args.radius * 1e6)
    key = src * N + dst
    assert len(torch.unique(key)) == len(key)
    assert torch.isfinite(dec).all()
    # a sample processed alone gives the same outputs as inside the batch (batch shards cleanly, SURVEY 8e)
    b = 3
    m = data.batch == b
    from dagr_b200.data import EventBatch
    single = EventBatch(x=data.x[m], pos=data.pos[m], batch=torch.zeros(int(m.sum()), dtype=torch.long),
                        width=data.width[:1], height=data.height[:1], time_window=data.time_window[:1], num_graphs=1)
    dec1, _, _ = _run_graph(model, single, 1)
    assert_close(dec1[0].cpu(), dec[b].cpu(), tol=1e-5, what="sample alone vs inside batch")


# ---------------------------------------------------------------------------------------------
def test_masked_ops_vs_oracle_and_reference():
    import ctypes as C
    from dagr_b200 import _lib
    from oracle import ref_ops as R
    lib = _lib.load()
    t = masked_ops_inputs("cuda")
    idx, x, w, b, base = t["idx"], t["x"], t["w"], t["b"], t["base"]
    K, Cin, Cout = len(idx), x.shape[1], w.shape[0]
    # outputs of the reference's own asy_tools kernels on these inputs (tests/golden/make_reference_kernels_golden.py)
    gold = np.load(GOLD / "reference_masked_ops.npz")
    assert sha256(*(t[k] for k in sorted(t))) == str(gold["inputs_sha256"]), "inputs differ from the ones the fixture was made from"

    def reference(name):
        o = base.cpu().clone()
        o[idx.cpu()] = torch.from_numpy(gold[name])                   # the reference kernels write the indexed rows only
        return o

    for add in (0, 1):
        for bias in (b, None):
            out = base.clone()
            _lib.check(lib.dagr_masked_lin(_lib.ptr(idx), K, _lib.ptr(x), _lib.ptr(out), _lib.ptr(w), _lib.ptr(bias), Cin, Cout, add,
                                           _lib.stream_ptr()))
            ref = R.masked_lin(idx.cpu(), x.cpu(), base.cpu().clone(), w.cpu(), None if bias is None else bias.cpu(), bool(add))
            assert_close(out.cpu(), ref, tol=1e-5, what="masked_lin")
            o2 = reference(f"masked_lin_add{add}" if bias is not None else f"masked_lin_no_bias_add{add}")
            assert_close(out.cpu(), o2, tol=1e-6, what="masked_lin vs reference asy_tools")
    mean, var, g, be, xin = t["mean"], t["var"], t["gamma"], t["beta"], t["xin"]
    out = base.clone()
    _lib.check(lib.dagr_masked_inplace_bn(_lib.ptr(idx), K, _lib.ptr(xin), _lib.ptr(out), _lib.ptr(mean), _lib.ptr(var), _lib.ptr(g),
                                          _lib.ptr(be), Cout, 1e-5, _lib.stream_ptr()))
    ref = R.masked_inplace_bn(idx.cpu(), xin.cpu(), base.cpu().clone(), mean.cpu(), var.cpu(), g.cpu(), be.cpu(), 1e-5)
    assert_close(out.cpu(), ref, tol=1e-5, what="masked_inplace_bn")
    assert_close(out.cpu(), reference("masked_inplace_bn"), tol=1e-6, what="masked_inplace_bn vs reference")
    a, c = t["a"], t["c"]                                             # c differs from a in column 3 of idx[::3]; Q3 row idx[1]
    cand = idx.clone()
    _lib.check(lib.dagr_masked_isdiff(_lib.ptr(cand), K, _lib.ptr(a), _lib.ptr(c), Cin, 1e-8, 1e-5, _lib.stream_ptr()))
    mine = cand[cand > -1].cpu()
    ref = R.masked_isdiff(idx.cpu(), a.cpu(), c.cpu(), 1e-8, 1e-5)
    assert torch.equal(mine, ref)
    assert torch.equal(mine, torch.from_numpy(gold["masked_isdiff"]))


def test_ingest_downsampler_vs_reference_golden_and_oracle():
    """csrc/ingest.cu vs (a) the golden vectors made by the reference's own numba down-sampler, chunk by chunk with the
    change map carried over, and (b) the oracle on a larger random stream with hot pixels; bit-exact (mask, coordinates,
    accumulator map)."""
    from dagr_b200 import ingest
    from oracle import ref_ingest as R
    g = np.load(ROOT / "tests" / "golden" / "downsample_golden.npz")
    for case in range(3):
        iw, ih, ow, oh = (int(v) for v in g[f"c{case}_shape"])
        cm = None
        for k in range(3):
            ev = {q: torch.from_numpy(g[f"c{case}_k{k}_in_{q}"].astype({"x": "int16", "y": "int16", "p": "int8", "t": "int64"}[q])).cuda()
                  for q in "xypt"}
            out, cm = ingest.downsample_events(ev, ih, iw, oh, ow, change_map=cm)
            for q in "xypt":
                assert np.array_equal(out[q].cpu().numpy().astype("int64"), g[f"c{case}_k{k}_out_{q}"].astype("int64")), (case, k, q)
            assert np.array_equal(cm.cpu().numpy(), g[f"c{case}_k{k}_map"])
    rng = np.random.default_rng(11)
    n, iw, ih, ow, oh = 300000, 640, 480, 320, 240
    ev = dict(x=rng.integers(0, iw, n).astype("int16"), y=rng.integers(0, ih, n).astype("int16"),
              p=(2 * rng.integers(0, 2, n) - 1).astype("int8"), t=np.sort(rng.integers(0, 50000, n)).astype("int64"))
    ev["x"][:20000] = 101; ev["y"][:20000] = 57; ev["p"][:20000:4] = 1          # one very hot pixel block
    want, wm = R.downsample_events({k: v.astype("uint16") if k in "xy" else v for k, v in ev.items()}, ih, iw, oh, ow)
    got, gm = ingest.downsample_events({k: torch.from_numpy(v).cuda() for k, v in ev.items()}, ih, iw, oh, ow)
    for q in "xypt":
        assert np.array_equal(got[q].cpu().numpy().astype("int64"), want[q].astype("int64")), q
    assert np.array_equal(gm.cpu().numpy(), wm)
    empty, cm0 = ingest.downsample_events({k: torch.from_numpy(v[:0]).cuda() for k, v in ev.items()}, ih, iw, oh, ow)
    assert all(v.numel() == 0 for v in empty.values()) and float(cm0.abs().sum()) == 0.0


def test_ingest_window_vs_oracle_and_forward():
    """raw (x, y, t, p) -> batch/pos_denorm/polarity on the device equals the oracle's restatement of
    preprocess_events + to_data + format_data + denormalize_pos, and the collated batch drives DAGR.forward to the same
    detections as the formatted float batch."""
    from dagr_b200 import ingest
    from dagr_b200.data import EventBatch, format_data
    from oracle import ref_ingest as R
    W, H, T, B = 320, 215, 1_000_000, 2
    rng = np.random.default_rng(5)
    samples, raw = [], []
    for b in range(B):
        n = 9000 + 1000 * b
        ev = dict(x=rng.integers(0, W, n).astype("int16"), y=rng.integers(0, 240, n).astype("int16"),
                  t=np.sort(rng.integers(7_000_000, 7_060_000, n)).astype("int64"), p=rng.integers(0, 2, n).astype("int8"))
        cut = 7_050_000
        den, pol = R.preprocess_window({k: v.astype("uint16") if k in "xy" else v for k, v in ev.items()}, W, H, T, t_cut=cut)
        bt, pos, feat = ingest.ingest_window({k: torch.from_numpy(v).cuda() for k, v in ev.items()}, W, H, T, t_cut=cut, sample=b)
        assert np.array_equal(pos.cpu().numpy(), den) and np.array_equal(feat.cpu().numpy(), pol)
        assert int(bt.min()) == b and int(bt.max()) == b
        samples.append((bt, pos, feat))
        keep = (ev["t"] < cut) & (ev["y"] < H)
        t_rel = T + ev["t"][keep] - ev["t"][keep][-1]                    # dsec_data.py:145, before any float round trip
        raw.append((np.stack([ev["x"][keep], ev["y"][keep], t_rel], axis=1), pol))
    e0 = ingest.ingest_window({k: torch.zeros(0, dtype=torch.int64, device="cuda") for k in "xytp"}, W, H, T)
    assert e0[1].shape == (0, 3)
    model, args = make_model("s", H, W)
    model.cuda()
    d_int = ingest.collate(samples, W, H, T)
    det_int = model(d_int)[0]
    # the same events through the reference's float interface (format_data on int16 pos + int32 t)
    pos16 = torch.from_numpy(np.concatenate([r[0][:, :2] for r in raw]).astype("int16"))
    t32 = torch.from_numpy(np.concatenate([r[0][:, 2] for r in raw]).astype("int32"))
    dflt = EventBatch(x=torch.from_numpy(np.concatenate([r[1] for r in raw])).view(-1, 1), pos=pos16, t=t32,
                      batch=torch.cat([s[0] for s in samples]).long().cpu(), width=torch.full((B,), W), height=torch.full((B,), H),
                      time_window=torch.full((B,), T), num_graphs=B)
    det_f = model(format_data(dflt).cuda())[0]
    for a, b_ in zip(det_int, det_f):
        assert a["boxes"].shape == b_["boxes"].shape
        assert_close(a["boxes"].cpu(), b_["boxes"].cpu(), what="boxes (ingest vs float batch)")


def test_streaming_window_equals_dense_forward_on_live_window():
    """dagr_b200.streaming (config 5): watermark eviction + append in a device ring, the whole step one CUDA graph replay.
    After every chunk the detections must equal the synchronous forward over the live window -- checked before the window
    is full, across >= 3 evictions, and on both the eager (first two) and the replayed steps."""
    import numpy as np
    from dagr_b200.data import EventBatch
    from dagr_b200.streaming import StreamingDetector, synth_stream
    W, H = 320, 215
    model, args = make_model("s", H, W, batch_size=1)
    model.cuda()
    window_us, chunk_us = 20_000, 2_000
    x, y, t, p = synth_stream(400_000, 0.06, W, H, seed=5, kind="clustered")
    det = StreamingDetector(model, window_us=window_us, max_chunk=4096, capacity=1 << 15)
    bounds = np.searchsorted(t, np.arange(0, 60_000 + chunk_us, chunk_us))
    checked = 0
    for k in range(len(bounds) - 1):
        a, b = int(bounds[k]), int(bounds[k + 1])
        t_end = (k + 1) * chunk_us
        out = det.push(x[a:b], y[a:b], t[a:b], p[a:b], t_end)
        if k in (0, 1, 2, 5, 11, 12, 13, 20, 29):
            st = det.window_state
            live = (t >= t_end - window_us) & (t < t_end)
            assert st["live"] == int(live.sum()) and not st["overflow"], (k, st, int(live.sum()))
            if k >= 11:
                assert st["evicted"] > 0
            pos, feat = det.live_window()
            assert np.array_equal(pos[:, 2].cpu().numpy(), t[live])
            n = len(feat)
            d = EventBatch(x=feat.view(-1, 1).clone(), pos=torch.zeros(n, 3, device="cuda"), batch=torch.zeros(n, dtype=torch.long, device="cuda"),
                           width=torch.tensor([W]), height=torch.tensor([H]), time_window=torch.tensor([1_000_000]),
                           pos_denorm=pos.clone(), num_graphs=1, dims=(W, H, 1_000_000))
            want = model(d)[0][0]
            assert len(out[0]["boxes"]) == len(want["boxes"]), (k, len(out[0]["boxes"]), len(want["boxes"]))
            assert torch.equal(out[0]["boxes"], want["boxes"].cpu()) and torch.equal(out[0]["scores"], want["scores"].cpu())
            checked += 1
    assert checked == 9 and det.graph is not None


def test_no_events_returns_the_image_only_head_like_the_reference():
    """--no_events (dagr.py:284): the detector outputs come from the CNN head maps alone (collect_outputs + decode_outputs)."""
    from dagr_b200.data import format_data, synth_batch
    from oracle import ref_ops as R
    W, H, B = 240, 180, 2
    model, args = make_model("n", H, W, use_image=True, img_net="resnet18", no_events=True, batch_size=B)
    model.cuda()
    data = format_data(synth_batch(B, 3000, W, H, seed=3, with_image=True).clone())
    dec = model.forward_decoded(data.clone().cuda())
    torch.cuda.synchronize()
    outs = {k: [t.cpu() for t in v] for k, v in model.last_image_outs.items()}
    maps = [torch.cat([outs["reg_output"][k], torch.sigmoid(outs["obj_output"][k]), torch.sigmoid(outs["cls_output"][k])], 1) for k in range(2)]
    want = R.decode_outputs(torch.cat([m.flatten(start_dim=2) for m in maps], dim=2).permute(0, 2, 1), [m.shape[-2:] for m in maps],
                            model.backbone.strides)
    assert_close(dec.cpu(), want, tol=1e-6, what="no_events decoded")
    dets = model(data.clone().cuda())[0]
    assert len(dets) == B


@pytest.mark.parametrize("use_image", [False, True])
def test_reloading_weights_after_graph_capture_takes_effect(use_image):
    """the coarse stack (and the image branch) are replayed as CUDA graphs that hold pointers to packed weights: after
    load_state_dict the next forward must use the NEW weights (graph cache keyed on a pack generation, image graphs dropped)."""
    from dagr_b200.data import format_data, synth_batch
    W, H, B = 240, 180, 2
    kw = dict(use_image=True, img_net="resnet18") if use_image else {}
    model_a, _ = make_model("n", H, W, seed=0, batch_size=B, **kw)
    model_b, _ = make_model("n", H, W, seed=5, batch_size=B, **kw)
    model_a.cuda(); model_b.cuda()
    data = format_data(synth_batch(B, 4000, W, H, seed=9, with_image=use_image).clone()).cuda()
    for _ in range(4):                                         # eager, warm, capture, replay
        out_a = model_a.forward_decoded(data.clone()).clone()
    want_b = model_b.forward_decoded(data.clone()).clone()
    torch.cuda.synchronize()
    assert not torch.equal(out_a, want_b)
    model_a.load_state_dict(model_b.state_dict())
    for k in range(3):
        got = model_a.forward_decoded(data.clone()).clone()
        torch.cuda.synchronize()
        if use_image:                                          # cuDNN may pick another algorithm for the re-captured branch
            assert_close(got, want_b, tol=1e-4, what="decoded after reload (image)")
        else:
            assert torch.equal(got, want_b), f"forward {k} after load_state_dict still uses old weights"


@pytest.mark.parametrize("variant", ["k8_r4", "mean_pooling", "empty_middle_sample", "one_scale", "k1"])
def test_config_variants_parity_vs_oracle(variant):
    """corners of the config surface (config/*.yaml keys): fewer neighbours / smaller radius, mean pooling, a sample without
    events inside the batch, a single head scale, self loops only."""
    from dagr_b200.data import EventBatch
    W, H, B = 320, 215, 3
    over = dict(k8_r4=dict(max_neighbors=8, radius=0.006), mean_pooling=dict(pooling_aggr="mean"), empty_middle_sample={},
                one_scale=dict(num_scales=1), k1=dict(max_neighbors=1))[variant]
    model, args = make_model("n", H, W, batch_size=B, **over)
    model.cuda()
    raw, data = make_inputs(B, 7000, W, H, seed=13, kind="clustered", ragged=True)
    if variant == "empty_middle_sample":
        keep = data.batch != 1
        data = EventBatch(x=data.x[keep], pos=data.pos[keep], batch=data.batch[keep], width=data.width, height=data.height,
                          time_window=data.time_window, num_graphs=B)
    _check_forward(model, args, data, B, H, W)


def test_mean_pooling_with_image_fusion_parity_vs_oracle():
    """pooling_aggr: mean also averages the sampled image channels appended before pool1 (net.py:128-131, pooling.py:76-77)."""
    from dagr_b200.data import format_data, synth_batch
    W, H, B = 240, 180, 2
    model, args = make_model("n", H, W, use_image=True, img_net="resnet18", batch_size=B, pooling_aggr="mean")
    model.cuda()
    raw = synth_batch(B, 5000, W, H, seed=78, kind="clustered", with_image=True, ragged=True)
    _check_forward(model, args, format_data(raw.clone()), B, H, W, image=True, check_public=False)
