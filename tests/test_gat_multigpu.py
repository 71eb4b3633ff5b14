"""GPU suite, multi-GPU part of graph attention (needs >= 2 GPUs; skipped where the box has fewer than the case
wants): build_gat partitioned over 2, 4 and 8 ranks — h, s_src / s_dst, dOut and lse / c travel through the halo
exchange (peer writes at every size, staged rows + NCCL at 2) — against the fp64 witness on the whole graph: the
stitched logits and the all-reduced dW, bitwise equal on every rank.  The whole-matrix all-gather
(ROC_B200_HALO=0) is refused at init."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, rel_close

pytestmark = [pytest.mark.gpu, pytest.mark.multigpu]

LAYERS, HEADS = (24, 32, 7), 4


def _case():
    from roc_b200 import datasets
    re_t, col_t = datasets.rmat_graph(11, 12000, seed=21)
    row_end, col = re_t.numpy().astype(np.uint64), col_t.numpy().astype(np.uint32)
    feats, labels, mask = datasets.node_data(row_end.shape[0], LAYERS[0], LAYERS[-1], seed=5)
    return row_end, col, feats.numpy(), labels.numpy(), mask.numpy()


def _worker(rank, world, port, tmpdir):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from roc_b200.model import Host, Model, build_gat
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
    h = build_gat(m, list(LAYERS), HEADS, 0.0)
    m.set_tensor(h["input"], feats[rl:rr + 1])
    m.set_labels(h["label"], labels[rl:rr + 1])
    m.set_tensor(h["mask"], mask[rl:rr + 1].astype(np.int32))
    out = {"rl": rl, "rr": rr, "w0": [m.get_parameter(p) for p in range(m.num_parameters())]}
    m.train_mode(); m.zero_gradients(); m.forward()
    out["logits"] = m.get_tensor(h["logits"])
    m.backward()
    m.update()
    out["dW_reduced"] = [m.get_parameter(p, "grad") for p in range(m.num_parameters())]
    np.save(os.path.join(tmpdir, "rank%d.npy" % rank), np.array([out], dtype=object), allow_pickle=True)
    host.close()
    dist.destroy_process_group()


@pytest.mark.parametrize("halo", ["p2p", "nccl"])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_multi_gpu_gat_matches_witness(tmp_path, world, halo, monkeypatch):
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    if halo == "nccl" and world != 2:
        pytest.skip("the NCCL exchange is cross-checked at 2 ranks")
    import torch.multiprocessing as mp
    from test_gat_gpu import gat_witness
    if halo == "nccl":
        monkeypatch.setenv("ROC_B200_HALO", "nccl")
    else:
        monkeypatch.delenv("ROC_B200_HALO", raising=False)
    port = 29400 + (os.getpid() * 7 + world * 3 + 1) % 1000
    mp.spawn(_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    r = [np.load(tmp_path / ("rank%d.npy" % k), allow_pickle=True)[0] for k in range(world)]
    case = _case()
    assert r[world - 1]["rr"] == case[0].shape[0] - 1
    wl, wdw = gat_witness(*case, LAYERS, HEADS, r[0]["w0"])
    rel_close(np.concatenate([r[q]["logits"] for q in range(world)]), wl, what="stitched logits")
    for p in range(len(wdw)):
        for q in range(1, world):
            assert np.array_equal(r[0]["dW_reduced"][p], r[q]["dW_reduced"][p])
        rel_close(r[0]["dW_reduced"][p], wdw[p], rtol=2e-4, atol_scale=2e-5, what="all-reduced dW[%d]" % p)


_REFUSE = r"""
import os, sys
sys.path.insert(0, sys.argv[1])
import torch, torch.distributed as dist
rank, world, port = int(sys.argv[2]), int(sys.argv[3]), sys.argv[4]
os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = port
dist.init_process_group("gloo", rank=rank, world_size=world)
torch.cuda.set_device(rank)
from roc_b200 import datasets
from roc_b200.model import Host, Model, build_gat
re_t, col_t = datasets.rmat_graph(9, 3000, seed=2)
host = Host(rank, rank, world)
uid = [Host.nccl_unique_id() if rank == 0 else None]
dist.broadcast_object_list(uid, src=0)
host.nccl_init(uid[0])
host.graph_from_arrays(re_t.numpy().astype("uint64"), col_t.numpy().astype("uint32"))
build_gat(Model(host, seed=1), [8, 16, 3], 2, 0.0)
print("initialised")
"""


def test_multi_gpu_gat_refuses_whole_matrix_all_gather(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "refuse.py"
    script.write_text(_REFUSE)
    env = dict(os.environ, ROC_B200_HALO="0")
    port = str(29400 + (os.getpid() * 7 + 5) % 1000)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, str(k), "2", port], env=env,
                              stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for k in range(2)]
    outs = [p.communicate(timeout=300) for p in procs]
    for p, (o, e) in zip(procs, outs):
        assert p.returncode != 0 and "initialised" not in o
        assert "graph_attention needs the halo exchange" in e, e[-2000:]
