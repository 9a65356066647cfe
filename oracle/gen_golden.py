"""Generate tests/golden/*.npz by running the UNMODIFIED reference  (TEST INFRASTRUCTURE ONLY).

Run in the build container (needs /root/reference):   python oracle/gen_golden.py

Each fixture stores, for a seeded case, everything needed to replay it without the reference:
  x                      input values as float32 (bf16 cases: bf16-representable values)
  s{step}_..._pre/post   codebook buffers (embed, embed_avg, cluster_size) before / after each step
  s{step}_quantize/_indices/_loss   the reference outputs of that forward
The reference runs on CPU with torch's fp32 kernels (Codebook.forward upcasts, vqp.py:692).
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from ref_loader import load_reference  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")


def f32(t):
    return t.detach().float().cpu().numpy().astype(np.float32)


def codebooks_of(module):
    """Distinct Codebook objects in forward order."""
    ref = sys.modules["vector_quantize_pytorch.vector_quantize_pytorch"]
    seen, out = set(), []
    for m in module.modules():
        if isinstance(m, ref.Codebook) and id(m) not in seen:
            seen.add(id(m))
            out.append(m)
    return out


def snap(module, tag, store):
    i = 0
    for cb in codebooks_of(module):
        for j in range(cb.embed.shape[0]):   # num_codebooks > 1: separate_codebook_per_head
            store[f"{tag}_cb{i}_embed"] = f32(cb.embed[j])
            store[f"{tag}_cb{i}_embed_avg"] = f32(cb.embed_avg[j])
            store[f"{tag}_cb{i}_cluster_size"] = f32(cb.cluster_size[j])
            i += 1


def randomize_codebooks(module, gen, scale=1.0, cosine=False):
    """Replace the degenerate kaiming init (|c| ~ 5e-3, SURVEY §7.2) by a seeded randn codebook."""
    for cb in codebooks_of(module):
        e = torch.randn(cb.embed.shape, generator=gen) * scale
        if cosine:
            e = torch.nn.functional.normalize(e, dim=-1)
        cb.embed.data.copy_(e)
        cb.embed_avg.data.copy_(e)


def run_case(name, build, x_shape, dtype, steps, meta, randomize=True, scale=1.0, clustered=False, seed_steps=False):
    ref = load_reference()
    torch.manual_seed(1234)
    gen = torch.Generator().manual_seed(4321)
    module = build(ref)
    cosine = bool(meta.get("use_cosine_sim", False))
    if randomize:
        randomize_codebooks(module, gen, scale, cosine)
    store = {}
    tdtype = torch.bfloat16 if dtype == "bf16" else torch.float32
    for step, mode in enumerate(steps):
        x = torch.randn(*x_shape, generator=gen)
        if clustered:
            cb0 = codebooks_of(module)[0].embed[0]
            pick = torch.randint(0, cb0.shape[0], x_shape[:-1], generator=gen)
            if x_shape[-1] == cb0.shape[-1]:
                x = cb0[pick] + 0.3 * x
        x = x.to(tdtype)
        module.train(mode == "train")
        if seed_steps:  # dead-code expiry draws torch.randperm from the global RNG (vqp:156-163): make it replayable
            torch.manual_seed(5000 + step)
        if step == 0:  # later steps: pre(step) == post(step-1)
            snap(module, "s0_pre", store)
        with torch.no_grad():
            out = module(x)
        store[f"s{step}_x"] = f32(x)
        store[f"s{step}_quantize"] = f32(out[0])
        store[f"s{step}_indices"] = out[1].cpu().numpy().astype(np.int64)
        store[f"s{step}_loss"] = f32(out[2])
        snap(module, f"s{step}_post", store)
    meta = dict(meta, name=name, dtype=dtype, steps=list(steps), x_shape=list(x_shape),
                torch=torch.__version__, n_codebooks=sum(cb.embed.shape[0] for cb in codebooks_of(module)))
    store["meta"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **store)
    print(f"{name}: {os.path.getsize(path) / 1024:.0f} KiB")


def expire_cases():
    """Dead-code expiry (vqp:544-574, rvq:599-601): threshold 2 with 8-cluster data on 64 codes, so that most codes die.
    The sampled replacement rows come from torch's global CPU RNG, re-seeded before every step (replayed by the tests)."""
    T = "train"
    run_case("expire_vq_fp32", lambda r: r.VectorQuantize(dim=32, codebook_size=64, threshold_ema_dead_code=2), (4, 96, 32), "fp32",
             [T, T, T], dict(kind="vq", dim=32, codebook_size=64, threshold_ema_dead_code=2), clustered=True, seed_steps=True)
    run_case("expire_vq_cosine_bf16", lambda r: r.VectorQuantize(dim=32, codebook_size=64, threshold_ema_dead_code=2, use_cosine_sim=True),
             (4, 96, 32), "bf16", [T, T, T], dict(kind="vq", dim=32, codebook_size=64, threshold_ema_dead_code=2, use_cosine_sim=True),
             seed_steps=True)
    run_case("expire_rvq_shared_fp32", lambda r: r.ResidualVQ(dim=32, num_quantizers=3, codebook_size=64, shared_codebook=True,
                                                              threshold_ema_dead_code=2), (3, 64, 32), "fp32", [T, T],
             dict(kind="rvq", dim=32, codebook_size=64, num_quantizers=3, shared_codebook=True, threshold_ema_dead_code=2),
             clustered=True, seed_steps=True)
    run_case("expire_rvq_separate_fp32", lambda r: r.ResidualVQ(dim=32, num_quantizers=3, codebook_size=64, threshold_ema_dead_code=2),
             (3, 64, 32), "fp32", [T, T],
             dict(kind="rvq", dim=32, codebook_size=64, num_quantizers=3, shared_codebook=False, threshold_ema_dead_code=2),
             clustered=True, seed_steps=True)


def kmeans_cases():
    """kmeans_init=True (vqp:238-278, :451-473): the first training batch initialises the codebook with Lloyd iterations;
    `initted` starts False, so `randomize=False` (the zero codebook of vqp:383) and the RNG is re-seeded per step."""
    T = "train"
    run_case("kmeans_vq_fp32", lambda r: r.VectorQuantize(dim=32, codebook_size=24, kmeans_init=True, kmeans_iters=4), (4, 128, 32), "fp32",
             [T, T], dict(kind="vq", dim=32, codebook_size=24, kmeans_init=True, kmeans_iters=4), randomize=False, seed_steps=True)
    run_case("kmeans_vq_cosine_bf16", lambda r: r.VectorQuantize(dim=32, codebook_size=24, kmeans_init=True, kmeans_iters=3, use_cosine_sim=True),
             (4, 128, 32), "bf16", [T, T], dict(kind="vq", dim=32, codebook_size=24, kmeans_init=True, kmeans_iters=3, use_cosine_sim=True),
             randomize=False, seed_steps=True)


def grad_case(name, build, x_shape, dtype, meta, freeze=True):
    """Gradient estimators (vqp:282-318, :1225-1233): the reference's d(sum(quantize * G) + loss)/dx for a seeded x, G.
    `freeze_codebook=True`: the codebook (and so the quantized rows) is the same before and after the call."""
    ref = load_reference()
    torch.manual_seed(1234)
    gen = torch.Generator().manual_seed(2468)
    module = build(ref)
    randomize_codebooks(module, gen, 1.0, bool(meta.get("use_cosine_sim", False)))
    tdtype = torch.bfloat16 if dtype == "bf16" else torch.float32
    x = torch.randn(*x_shape, generator=gen).to(tdtype).requires_grad_(True)
    G = torch.randn(*x_shape, generator=gen).to(tdtype)
    module.train()
    store = {}
    snap(module, "s0_pre", store)
    q, ind, loss = module(x, freeze_codebook=freeze)
    ((q * G).sum() + loss.sum().to(q.dtype)).backward()
    store.update(s0_x=f32(x), s0_G=f32(G), s0_quantize=f32(q), s0_indices=ind.cpu().numpy().astype(np.int64), s0_loss=f32(loss),
                 s0_xgrad=f32(x.grad))
    meta = dict(meta, name=name, dtype=dtype, steps=["train"], x_shape=list(x_shape), torch=torch.__version__,
                n_codebooks=len(codebooks_of(module)))
    store["meta"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **store)
    print(f"{name}: {os.path.getsize(path) / 1024:.0f} KiB")


def grad_cases():
    grad_case("grad_vq_rotation_fp32", lambda r: r.VectorQuantize(dim=32, codebook_size=48), (2, 64, 32), "fp32",
              dict(kind="vq", dim=32, codebook_size=48))
    grad_case("grad_vq_ste_fp32", lambda r: r.VectorQuantize(dim=32, codebook_size=48, rotation_trick=False), (2, 64, 32), "fp32",
              dict(kind="vq", dim=32, codebook_size=48, rotation_trick=False))
    grad_case("grad_vq_rotation_cosine_fp32", lambda r: r.VectorQuantize(dim=32, codebook_size=48, use_cosine_sim=True), (2, 64, 32), "fp32",
              dict(kind="vq", dim=32, codebook_size=48, use_cosine_sim=True))
    grad_case("grad_vq_rotation_bf16", lambda r: r.VectorQuantize(dim=32, codebook_size=48), (2, 64, 32), "bf16",
              dict(kind="vq", dim=32, codebook_size=48))
    grad_case("grad_rvq_rotation_fp32", lambda r: r.ResidualVQ(dim=32, num_quantizers=3, codebook_size=48), (2, 64, 32), "fp32",
              dict(kind="rvq", dim=32, codebook_size=48, num_quantizers=3, shared_codebook=False))


def simvq_cases():
    """SimVQ (sim_vq.py:99-139): seeded x and upstream G; the reference's outputs and the gradients of sum(quantize * G) + loss
    with respect to x and to the weight of the codebook transform."""
    ref = load_reference()
    for name, rotation in (("simvq_rotation_fp32", True), ("simvq_ste_fp32", False)):
        torch.manual_seed(4321)
        gen = torch.Generator().manual_seed(8642)
        m = ref.SimVQ(dim=32, codebook_size=80, rotation_trick=rotation)
        x = torch.randn(2, 96, 32, generator=gen).requires_grad_(True)
        G = torch.randn(2, 96, 32, generator=gen)
        q, ind, loss = m(x)
        ((q * G).sum() + loss).backward()
        store = dict(s0_x=f32(x), s0_G=f32(G), s0_quantize=f32(q), s0_indices=ind.cpu().numpy().astype(np.int64), s0_loss=f32(loss),
                     s0_xgrad=f32(x.grad), s0_wgrad=f32(m.code_transform.weight.grad), frozen=f32(m.frozen_codebook),
                     weight=f32(m.code_transform.weight))
        meta = dict(kind="simvq", name=name, dim=32, codebook_size=80, rotation_trick=rotation, dtype="fp32", steps=["train"],
                    x_shape=[2, 96, 32], torch=torch.__version__)
        store["meta"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
        path = os.path.join(OUT, name + ".npz")
        np.savez_compressed(path, **store)
        print(f"{name}: {os.path.getsize(path) / 1024:.0f} KiB")


def heads_cases():
    """heads > 1 with ONE codebook shared by the heads (vqp:1044-1049, :1266-1270, :1354-1358); codebook_dim = dim / heads, so
    there is no projection."""
    T, E = "train", "eval"
    run_case("vq_heads4_fp32", lambda r: r.VectorQuantize(dim=64, heads=4, codebook_dim=16, codebook_size=64), (2, 80, 64), "fp32",
             [T, T, E], dict(kind="vq", dim=64, heads=4, codebook_dim=16, codebook_size=64))
    run_case("vq_sepheads4_fp32", lambda r: r.VectorQuantize(dim=64, heads=4, codebook_dim=16, codebook_size=48, separate_codebook_per_head=True),
             (2, 80, 64), "fp32", [T, T, E], dict(kind="vq", dim=64, heads=4, codebook_dim=16, codebook_size=48, separate_codebook_per_head=True))
    run_case("vq_sepheads2_cosine_bf16", lambda r: r.VectorQuantize(dim=64, heads=2, codebook_dim=32, codebook_size=48, use_cosine_sim=True,
                                                                    separate_codebook_per_head=True),
             (2, 80, 64), "bf16", [T, T, E], dict(kind="vq", dim=64, heads=2, codebook_dim=32, codebook_size=48, use_cosine_sim=True,
                                                  separate_codebook_per_head=True))
    run_case("vq_heads2_cosine_bf16", lambda r: r.VectorQuantize(dim=64, heads=2, codebook_dim=32, codebook_size=64, use_cosine_sim=True),
             (2, 80, 64), "bf16", [T, T, E], dict(kind="vq", dim=64, heads=2, codebook_dim=32, codebook_size=64, use_cosine_sim=True))


def mask_cases():
    """Variable-length input (vqp:1116-1119 `mask` / `lens`, :599-600 masked statistics, :1317-1325 loss over the unmasked
    elements against the ORIGINAL input, :1378-1396 padding comes back as zeros / the input and index -1)."""
    ref = load_reference()
    T, E = "train", "eval"
    cases = [
        ("mask_vq_fp32", dict(dim=64, codebook_size=96), (3, 70, 64), "fp32", [T, T, E], "mask"),
        ("mask_vq_lens_bf16", dict(dim=64, codebook_size=96), (3, 70, 64), "bf16", [T, T, E], "lens"),
        ("mask_vq_cosine_keep_fp32", dict(dim=32, codebook_size=48, use_cosine_sim=True, return_zeros_for_masked_padding=False,
                                          commitment_weight=0.5), (2, 90, 32), "fp32", [T, E], "mask"),
    ]
    for name, kw, x_shape, dtype, steps, how in cases:
        torch.manual_seed(1234)
        gen = torch.Generator().manual_seed(97531)
        module = ref.VectorQuantize(**kw)
        randomize_codebooks(module, gen, 1.0, bool(kw.get("use_cosine_sim", False)))
        tdtype = torch.bfloat16 if dtype == "bf16" else torch.float32
        store = {}
        for step, mode in enumerate(steps):
            x = torch.randn(*x_shape, generator=gen).to(tdtype)
            if how == "lens":
                lens = torch.randint(1, x_shape[1] + 1, (x_shape[0],), generator=gen)
                lens[0] = x_shape[1]
                mask = torch.arange(x_shape[1])[None, :] < lens[:, None]
                call = dict(lens=lens)
                store[f"s{step}_lens"] = lens.numpy().astype(np.int64)
            else:
                mask = torch.rand(x_shape[:2], generator=gen) < 0.7
                call = dict(mask=mask)
            module.train(mode == "train")
            if step == 0:
                snap(module, "s0_pre", store)
            with torch.no_grad():
                out = module(x, **call)
            store[f"s{step}_x"] = f32(x)
            store[f"s{step}_mask"] = mask.numpy()
            store[f"s{step}_quantize"] = f32(out[0])
            store[f"s{step}_indices"] = out[1].cpu().numpy().astype(np.int64)
            store[f"s{step}_loss"] = f32(out[2])
            snap(module, f"s{step}_post", store)
        meta = dict(kw, kind="vq", name=name, dtype=dtype, steps=list(steps), x_shape=list(x_shape), how=how,
                    torch=torch.__version__, n_codebooks=1)
        store["meta"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
        path = os.path.join(OUT, name + ".npz")
        np.savez_compressed(path, **store)
        print(f"{name}: {os.path.getsize(path) / 1024:.0f} KiB")


def layout_cases():
    """Input layouts (vqp:1121-1125 one token, :1136-1147 image / 3-D feature maps and channel-first, restored at :1265-1277 and
    :1364-1376); codebook_dim * heads == dim everywhere, so there is no projection and the fixtures replay exactly."""
    T, E = "train", "eval"
    run_case("layout_vq_image_fp32", lambda r: r.VectorQuantize(dim=32, codebook_size=48, accept_image_fmap=True), (2, 32, 6, 9), "fp32",
             [T, T, E], dict(kind="vq", layout="image", dim=32, codebook_size=48))
    run_case("layout_vq_3d_bf16", lambda r: r.VectorQuantize(dim=32, codebook_size=48, accept_3d_fmap=True), (2, 32, 3, 4, 5), "bf16",
             [T, T, E], dict(kind="vq", layout="3d", dim=32, codebook_size=48))
    run_case("layout_vq_chfirst_cosine_fp32", lambda r: r.VectorQuantize(dim=32, codebook_size=48, channel_last=False, use_cosine_sim=True),
             (2, 32, 50), "fp32", [T, T, E], dict(kind="vq", layout="channel_first", dim=32, codebook_size=48, use_cosine_sim=True))
    run_case("layout_vq_single_fp32", lambda r: r.VectorQuantize(dim=32, codebook_size=48), (37, 32), "fp32",
             [T, T, E], dict(kind="vq", layout="single", dim=32, codebook_size=48))
    run_case("layout_vq_image_heads2_fp32", lambda r: r.VectorQuantize(dim=32, codebook_size=48, accept_image_fmap=True, heads=2,
                                                                       codebook_dim=16), (2, 32, 5, 7), "fp32",
             [T, T, E], dict(kind="vq", layout="image", dim=32, codebook_size=48, heads=2, codebook_dim=16))


def mask_rvq_cases():
    """ResidualVQ / GroupedResidualVQ with a mask (rvq:493-500: every layer receives it; rvq:698 the groups pass it on):
    padding comes back as zeros / index -1 in every stage, the losses and the EMA statistics see the unmasked rows only."""
    ref = load_reference()
    T, E = "train", "eval"
    cases = [
        ("mask_rvq_shared_bf16", "rvq", dict(dim=32, num_quantizers=3, codebook_size=64, shared_codebook=True), (3, 40, 32), "bf16", [T, T, E]),
        ("mask_rvq_separate_fp32", "rvq", dict(dim=32, num_quantizers=3, codebook_size=64), (3, 40, 32), "fp32", [T, T, E]),
        ("mask_grvq_fp32", "grvq", dict(dim=64, groups=2, num_quantizers=2, codebook_size=48), (2, 44, 64), "fp32", [T, E]),
    ]
    for name, kind, kw, x_shape, dtype, steps in cases:
        torch.manual_seed(1234)
        gen = torch.Generator().manual_seed(86420)
        module = ref.ResidualVQ(**kw) if kind == "rvq" else ref.GroupedResidualVQ(**kw)
        randomize_codebooks(module, gen, 1.0, False)
        tdtype = torch.bfloat16 if dtype == "bf16" else torch.float32
        store = {}
        for step, mode in enumerate(steps):
            x = torch.randn(*x_shape, generator=gen).to(tdtype)
            mask = torch.rand(x_shape[:2], generator=gen) < 0.7
            module.train(mode == "train")
            if step == 0:
                snap(module, "s0_pre", store)
            with torch.no_grad():
                out = module(x, mask=mask)
            store[f"s{step}_x"] = f32(x)
            store[f"s{step}_mask"] = mask.numpy()
            store[f"s{step}_quantize"] = f32(out[0])
            store[f"s{step}_indices"] = out[1].cpu().numpy().astype(np.int64)
            store[f"s{step}_loss"] = f32(out[2])
            snap(module, f"s{step}_post", store)
        meta = dict(kw, kind=kind, name=name, dtype=dtype, steps=list(steps), x_shape=list(x_shape), how="mask",
                    shared_codebook=bool(kw.get("shared_codebook", False)), torch=torch.__version__,
                    n_codebooks=len(codebooks_of(module)))
        store["meta"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
        path = os.path.join(OUT, name + ".npz")
        np.savez_compressed(path, **store)
        print(f"{name}: {os.path.getsize(path) / 1024:.0f} KiB")


def dropout_cases():
    """quantize_dropout (rvq:423-439, :473-476): in training the layers after a randomly drawn index are skipped (index -1,
    loss 0).  The seed is passed explicitly (`rand_quantize_dropout_fixed_seed`), one per step, and stored."""
    ref = load_reference()
    T, E = "train", "eval"
    cases = [
        ("dropout_rvq_separate_fp32", dict(dim=32, num_quantizers=4, codebook_size=64, quantize_dropout=True), (2, 64, 32), "fp32",
         [T, T, T, E], [3, 11, 5, 0]),
        ("dropout_rvq_shared_bf16", dict(dim=32, num_quantizers=6, codebook_size=64, shared_codebook=True, quantize_dropout=True,
                                         quantize_dropout_cutoff_index=1, quantize_dropout_multiple_of=2), (2, 64, 32), "bf16",
         [T, T, T, E], [7, 2, 9, 0]),
    ]
    for name, kw, x_shape, dtype, steps, seeds in cases:
        torch.manual_seed(1234)
        gen = torch.Generator().manual_seed(13579)
        module = ref.ResidualVQ(**kw)
        randomize_codebooks(module, gen, 1.0, False)
        tdtype = torch.bfloat16 if dtype == "bf16" else torch.float32
        store = {}
        for step, mode in enumerate(steps):
            x = torch.randn(*x_shape, generator=gen)
            cb0 = codebooks_of(module)[0].embed[0]
            x = (cb0[torch.randint(0, cb0.shape[0], x_shape[:-1], generator=gen)] + 0.3 * x).to(tdtype)
            module.train(mode == "train")
            if step == 0:
                snap(module, "s0_pre", store)
            with torch.no_grad():
                out = module(x, rand_quantize_dropout_fixed_seed=seeds[step])
            store[f"s{step}_x"] = f32(x)
            store[f"s{step}_quantize"] = f32(out[0])
            store[f"s{step}_indices"] = out[1].cpu().numpy().astype(np.int64)
            store[f"s{step}_loss"] = f32(out[2])
            snap(module, f"s{step}_post", store)
        meta = dict(kw, kind="rvq", name=name, dtype=dtype, steps=list(steps), x_shape=list(x_shape), seeds=seeds,
                    shared_codebook=bool(kw.get("shared_codebook", False)), torch=torch.__version__,
                    n_codebooks=len(codebooks_of(module)))
        store["meta"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
        path = os.path.join(OUT, name + ".npz")
        np.savez_compressed(path, **store)
        print(f"{name}: {os.path.getsize(path) / 1024:.0f} KiB", [int((store[f's{i}_indices'][0, 0] >= 0).sum()) for i in range(len(steps))])


STATE_DICT_CASES = [
    ("VectorQuantize", dict(dim=64, codebook_size=32, use_cosine_sim=True)),
    ("ResidualVQ", dict(dim=32, num_quantizers=3, codebook_size=16)),
    ("VectorQuantize", dict(dim=64, codebook_size=32, heads=4, codebook_dim=16)),
    ("VectorQuantize", dict(dim=48, codebook_size=32, heads=2, separate_codebook_per_head=True)),
    ("SimVQ", dict(dim=32, codebook_size=40)),
    ("GroupedResidualVQ", dict(dim=64, groups=2, num_quantizers=2, codebook_size=16, shared_codebook=True)),
]


def state_dict_cases():
    """The reference's freshly constructed state_dict (torch.manual_seed(0) before construction) for each entry of
    STATE_DICT_CASES: key order in meta, every tensor as stored, so that checkpoint loading is checked without the reference."""
    ref = load_reference()
    store, meta = {}, []
    for i, (cls, kw) in enumerate(STATE_DICT_CASES):
        torch.manual_seed(0)
        sd = getattr(ref, cls)(**kw).state_dict()
        for k, v in sd.items():
            store[f"c{i}/{k}"] = v.detach().cpu().numpy()
        meta.append(dict(cls=cls, kw=kw, keys=list(sd)))
    store["meta"] = np.frombuffer(json.dumps(dict(cases=meta, torch=torch.__version__)).encode(), dtype=np.uint8)
    path = os.path.join(OUT, "state_dict", "reference_init.npz")
    os.makedirs(os.path.dirname(path), exist_ok=True)
    np.savez_compressed(path, **store)
    print(f"{path}: {os.path.getsize(path) / 1024:.0f} KiB")


def main():
    if "--state-dict" in sys.argv:
        return state_dict_cases()
    if "--dropout" in sys.argv:
        return dropout_cases()
    if "--mask-rvq" in sys.argv:
        return mask_rvq_cases()
    if "--layout" in sys.argv:
        return layout_cases()
    if "--mask" in sys.argv:
        return mask_cases()
    if "--heads" in sys.argv:
        return heads_cases()
    if "--simvq" in sys.argv:
        return simvq_cases()
    if "--grad" in sys.argv:
        return grad_cases()
    if "--expire" in sys.argv:
        return expire_cases()
    if "--kmeans" in sys.argv:
        return kmeans_cases()
    T, E = "train", "eval"
    # --- VectorQuantize (vqp.py:802) ---
    run_case("vq_euclid_fp32", lambda r: r.VectorQuantize(dim=64, codebook_size=96), (2, 80, 64), "fp32",
             [T, T, E], dict(kind="vq", dim=64, codebook_size=96))
    run_case("vq_euclid_bf16", lambda r: r.VectorQuantize(dim=64, codebook_size=96), (2, 80, 64), "bf16",
             [T, T, E], dict(kind="vq", dim=64, codebook_size=96))
    run_case("vq_cosine_fp32", lambda r: r.VectorQuantize(dim=64, codebook_size=96, use_cosine_sim=True),
             (2, 80, 64), "fp32", [T, T, E], dict(kind="vq", dim=64, codebook_size=96, use_cosine_sim=True))
    run_case("vq_cosine_bf16", lambda r: r.VectorQuantize(dim=64, codebook_size=96, use_cosine_sim=True),
             (2, 80, 64), "bf16", [T, T, E], dict(kind="vq", dim=64, codebook_size=96, use_cosine_sim=True))
    # default (kaiming) init: the tie-heavy regime of SURVEY §7.2
    run_case("vq_euclid_fp32_coldinit", lambda r: r.VectorQuantize(dim=64, codebook_size=96), (1, 128, 64), "fp32",
             [T, T], dict(kind="vq", dim=64, codebook_size=96), randomize=False)
    # README example shape, BASELINE config 1 (README.md:17-29) with a smaller batch
    run_case("vq_readme_fp32", lambda r: r.VectorQuantize(dim=256, codebook_size=512, decay=0.8, commitment_weight=1.),
             (1, 128, 256), "fp32", [T], dict(kind="vq", dim=256, codebook_size=512))
    run_case("vq_decay_cw_fp32", lambda r: r.VectorQuantize(dim=32, codebook_size=40, decay=0.95, commitment_weight=0.25, eps=1e-3),
             (3, 50, 32), "fp32", [T, T], dict(kind="vq", dim=32, codebook_size=40, decay=0.95, commitment_weight=0.25, eps=1e-3))
    # --- ResidualVQ (rvq.py:166) ---
    for dtype in ("fp32", "bf16"):
        run_case(f"rvq_shared_{dtype}", lambda r: r.ResidualVQ(dim=32, num_quantizers=4, codebook_size=64, shared_codebook=True),
                 (2, 64, 32), dtype, [T, T, E], dict(kind="rvq", dim=32, codebook_size=64, num_quantizers=4, shared_codebook=True),
                 clustered=True)
        run_case(f"rvq_separate_{dtype}", lambda r: r.ResidualVQ(dim=32, num_quantizers=4, codebook_size=64),
                 (2, 64, 32), dtype, [T, T, E], dict(kind="rvq", dim=32, codebook_size=64, num_quantizers=4, shared_codebook=False),
                 clustered=True)
    run_case("rvq_cosine_fp32", lambda r: r.ResidualVQ(dim=32, num_quantizers=3, codebook_size=64, use_cosine_sim=True),
             (2, 64, 32), "fp32", [T, E], dict(kind="rvq", dim=32, codebook_size=64, num_quantizers=3, shared_codebook=False,
                                                use_cosine_sim=True))
    # --- GroupedResidualVQ (rvq.py:634) ---
    run_case("grvq_fp32", lambda r: r.GroupedResidualVQ(dim=64, groups=2, num_quantizers=3, codebook_size=48),
             (2, 48, 64), "fp32", [T, T, E], dict(kind="grvq", dim=64, groups=2, codebook_size=48, num_quantizers=3,
                                                  shared_codebook=False))
    run_case("grvq_shared_bf16", lambda r: r.GroupedResidualVQ(dim=64, groups=2, num_quantizers=3, codebook_size=48, shared_codebook=True),
             (2, 48, 64), "bf16", [T, T], dict(kind="grvq", dim=64, groups=2, codebook_size=48, num_quantizers=3,
                                               shared_codebook=True))


if __name__ == "__main__":
    main()
