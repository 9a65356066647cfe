"""Multi-GPU parity (SURVEY §8e), `pytest -m gpu` on a box with >= 2 GPUs (skipped on one): one process per GPU, batch
sharded over the ranks, codebooks replicated.  After every training step

  * every rank's codebook buffers are BIT-identical (the replicas must not drift), and
  * they equal the single-process oracle run over the WHOLE batch (the reference semantics of
    vector_quantize_pytorch.py:603-617: sum of the shards' statistics) to 1e-5,

for VectorQuantize (fused peer-memory EMA in one chain), ResidualVQ (shared codebook) and GroupedResidualVQ
(BASELINE.json configs[4] shape family).  Also run with VQB_NO_PEER=1, i.e. through the NCCL all-reduce fallback.
"""
import os
import socket
import subprocess
import sys
import textwrap

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = textwrap.dedent('''
    import os, sys, json
    import numpy as np
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.environ["VQB_ROOT"]); sys.path.insert(0, os.path.join(os.environ["VQB_ROOT"], "tests"))
    import vector_quantize_pytorch_b200 as vqb
    from oracle import vq_oracle as O

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    kind = os.environ["VQB_CASE"]
    torch.manual_seed(1234)
    D, K, steps, rows = 64, 96, 3, 256          # rows per rank and step
    gen = torch.Generator().manual_seed(99)
    if kind == "vq":
        module = vqb.VectorQuantize(dim=D, codebook_size=K, sync_codebook=True).to(dev)
    elif kind == "rvq":
        module = vqb.ResidualVQ(dim=D, num_quantizers=3, codebook_size=K, shared_codebook=True, sync_codebook=True).to(dev)
    else:
        module = vqb.GroupedResidualVQ(dim=2 * D, groups=2, num_quantizers=3, codebook_size=K, sync_codebook=True).to(dev)
    books = []
    for sub in module.modules():
        if isinstance(sub, vqb.Codebook) and all(sub is not b for b in books):
            books.append(sub)
    states = []
    for cb in books:
        e = torch.randn(K, D, generator=gen)
        with torch.no_grad():
            cb.embed.copy_(e[None]); cb.embed_avg.copy_(e[None])
        states.append(O.CodebookState.from_embed(e.numpy()))
    module.train()
    cfg = O.VQConfig(dim=D, codebook_size=K)
    width = 2 * D if kind == "grvq" else D
    used_peer = None
    for step in range(steps):
        full = torch.randn(world * rows, 1, width, generator=gen)        # the GLOBAL batch, identical on every rank
        mine = full[rank * rows:(rank + 1) * rows].to(dev)
        q, ind, loss = module(mine)[:3]
        torch.cuda.synchronize()
        # oracle over the whole batch in one process
        x = full.numpy()
        if kind == "vq":
            _, io, _, _ = O.vq_forward(x, "fp32", states[0], cfg)
            ref_idx = io[rank * rows:(rank + 1) * rows]
        elif kind == "rvq":
            _, io, _, _ = O.rvq_forward(x, "fp32", [states[0]] * 3, cfg, shared_codebook=True)
            ref_idx = io[rank * rows:(rank + 1) * rows]
        else:
            _, io, _, _ = O.grouped_rvq_forward(x, "fp32", [states[:3], states[3:]], cfg)
            ref_idx = io[:, rank * rows:(rank + 1) * rows]
        assert np.array_equal(ind.cpu().numpy(), ref_idx), f"rank {rank} step {step}: indices differ from the full-batch oracle"
        for cb, st in zip(books, states):
            np.testing.assert_allclose(cb.cluster_size[0].cpu().numpy(), st.cluster_size, rtol=1e-5, atol=1e-5)
            np.testing.assert_allclose(cb.embed_avg[0].cpu().numpy(), st.embed_avg, rtol=1e-5, atol=2e-5)
            np.testing.assert_allclose(cb.embed[0].cpu().numpy(), st.embed, rtol=1e-5, atol=2e-5)
            # replicas bit-identical
            mine_bits = torch.cat([cb.embed.reshape(-1), cb.embed_avg.reshape(-1), cb.cluster_size.reshape(-1)]).view(torch.int32)
            lo, hi = mine_bits.clone(), mine_bits.clone()
            dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
            assert torch.equal(lo, hi), f"step {step}: replicas drifted"
    owner = books[0] if kind == "vq" else (module if kind == "rvq" else module.rvqs[0])
    used_peer = getattr(owner, "_peer", None) is not None
    if rank == 0:
        print("RESULT " + json.dumps({"case": kind, "world": world, "peer_memory": used_peer}))
    dist.destroy_process_group()
''')


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.parametrize("no_peer", [False, True])
@pytest.mark.parametrize("case", ["vq", "rvq", "grvq"])
def test_replicas_identical_and_equal_full_batch_oracle(case, no_peer, tmp_path):
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 2
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, VQB_ROOT=ROOT, VQB_CASE=case)
    if no_peer:
        env["VQB_NO_PEER"] = "1"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), str(script)]
    res = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    out = res.stdout + res.stderr
    assert res.returncode == 0, out[-4000:]
    line = [l for l in out.splitlines() if l.startswith("RESULT ")]
    assert line, out[-2000:]
    print(line[-1])
    if no_peer:
        assert '"peer_memory": false' in line[-1]
