"""GPU suite, multi-GPU part of the native aggregators (needs >= 2 GPUs; skipped where the box has fewer than the
case wants): GraphSAGE-max and GraphSAGE-mean partitioned over 2, 4 and 8 ranks — the winner ids and the mean's
scaled gradients travel through the halo exchange (peer writes, or staged rows + NCCL) — against the fp64 witness
on the whole graph: the stitched logits and the all-reduced dW."""
import os
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, rel_close

pytestmark = [pytest.mark.gpu, pytest.mark.multigpu]

LAYERS = (24, 32, 16, 7)


def _case():
    from roc_b200 import datasets
    re_t, col_t = datasets.rmat_graph(11, 12000, seed=21)
    row_end, col = re_t.numpy().astype(np.uint64), col_t.numpy().astype(np.uint32)
    feats, labels, mask = datasets.node_data(row_end.shape[0], LAYERS[0], LAYERS[-1], seed=5)
    return row_end, col, feats.numpy(), labels.numpy(), mask.numpy()


def _worker(rank, world, port, tmpdir, aggr):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from roc_b200.model import Host, Model, build_sage
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.cuda.set_device(rank)
    row_end, col, feats, labels, mask = _case()
    host = Host(rank, rank, world)
    uid = [Host.nccl_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    host.nccl_init(uid[0])
    host.graph_from_arrays(row_end, col)
    info = host.graph_info()
    rl, rr = info["rowLeft"], info["rowRight"]
    m = Model(host, seed=1)
    h = build_sage(m, list(LAYERS), 0.0, aggr=aggr)
    m.set_tensor(h["input"], feats[rl:rr + 1])
    m.set_labels(h["label"], labels[rl:rr + 1])
    m.set_tensor(h["mask"], mask[rl:rr + 1].astype(np.int32))
    out = {"rl": rl, "rr": rr, "w0": [m.get_parameter(p) for p in range(m.num_parameters())]}
    m.train_mode(); m.zero_gradients(); m.forward()
    out["logits"] = m.get_tensor(h["logits"])
    if aggr in ("max", "min"):
        out["args"] = [m.sg_arg(t) for t in h["sage_outs"]]
    m.backward()
    m.update()
    out["dW_reduced"] = [m.get_parameter(p, "grad") for p in range(m.num_parameters())]
    np.save(os.path.join(tmpdir, "rank%d.npy" % rank), np.array([out], dtype=object), allow_pickle=True)
    host.close()
    dist.destroy_process_group()


@pytest.mark.parametrize("halo", ["p2p", "nccl"])
@pytest.mark.parametrize("aggr", ["max", "mean"])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_multi_gpu_sage_matches_witness(tmp_path, world, aggr, halo, monkeypatch):
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    if halo == "nccl" and world != 2:
        pytest.skip("the NCCL exchange is cross-checked at 2 ranks")
    import torch.multiprocessing as mp
    from test_aggr_cpu import assert_args_differ_only_at_near_ties, sage_witness
    if halo == "nccl":
        monkeypatch.setenv("ROC_B200_HALO", "nccl")
    else:
        monkeypatch.delenv("ROC_B200_HALO", raising=False)
    port = 29400 + (os.getpid() * 7 + world) % 1000
    mp.spawn(_worker, args=(world, port, str(tmp_path), aggr), nprocs=world, join=True)
    r = [np.load(tmp_path / ("rank%d.npy" % k), allow_pickle=True)[0] for k in range(world)]
    case = _case()
    assert r[world - 1]["rr"] == case[0].shape[0] - 1
    args = None
    if aggr != "mean":
        args = [np.concatenate([r[q]["args"][i] for q in range(world)]) for i in range(len(r[0]["args"]))]
        _, _, own, pre = sage_witness(*case, LAYERS, r[0]["w0"], aggr)
        for g, o, p in zip(args, own, pre):
            assert_args_differ_only_at_near_ties(g, o, p)
    wl, wdw, _, _ = sage_witness(*case, LAYERS, r[0]["w0"], aggr, args=args)
    rel_close(np.concatenate([r[q]["logits"] for q in range(world)]), wl, what="stitched logits")
    for p in range(len(wdw)):
        for q in range(1, world):
            assert np.array_equal(r[0]["dW_reduced"][p], r[q]["dW_reduced"][p])
        rel_close(r[0]["dW_reduced"][p], wdw[p], rtol=2e-4, atol_scale=2e-5, what="all-reduced dW[%d]" % p)
