"""CPU-side checks of the drop-in boundary: the C-ABI library builds/loads without a GPU and exports
every symbol include/vqb200.h declares; argument errors are reported through return codes; the Python
host layer fails loudly instead of falling back to a CPU path."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_functions():
    text = open(os.path.join(ROOT, "include", "vqb200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(vqb_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from vector_quantize_pytorch_b200 import _C
    names = declared_functions()
    assert len(names) >= 14
    lib = ctypes.CDLL(_C.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/vqb200.h but not exported"
        assert n in _C.SIGNATURES, f"{n} has no ctypes signature in _C.py"
    assert _C.lib.vqb_version() == 100


def test_host_only_entry_points():
    from vector_quantize_pytorch_b200 import _C
    lib = _C.lib
    assert lib.vqb_padded_codes(1024) == 1024
    assert lib.vqb_padded_codes(1000) == 1024
    assert lib.vqb_padded_codes(5) == 16
    assert lib.vqb_padded_codes(96) == 96
    assert lib.vqb_stats_offset(5) == 8 and lib.vqb_stats_floats(5, 8) == 48
    assert lib.vqb_ema_stats_workspace(1000, 64) > 1000 * 4
    assert b"ok" in lib.vqb_strerror(0)
    assert b"aligned" in lib.vqb_strerror(-3)


def test_argument_errors_are_return_codes_not_crashes():
    from vector_quantize_pytorch_b200 import _C
    lib = _C.lib
    assert lib.vqb_codebook_prepare(None, 10, 8, 0, None, None, None, None, None, None) == -1
    assert lib.vqb_assign(None, 1, 10, 8, None, None, None, 4, 0.0, 0, None, None, None, None, None, None) == -1
    assert lib.vqb_gather(None, 0, 1, 8, None, None, None, None, 1, None, None, None, None, None) == -1
    assert lib.vqb_ema_stats(None, 0, 1, 8, None, 4, None, None, 0, None) == -1
    assert lib.vqb_decode(None, 0, 1, 1, 8, None, 1, None, 0, None) == -1


def test_no_cpu_fallback():
    import vector_quantize_pytorch_b200 as m
    vq = m.VectorQuantize(dim=64, codebook_size=32)
    with pytest.raises(RuntimeError, match="no CPU path"):
        vq(torch.randn(1, 8, 64))
    rvq = m.ResidualVQ(dim=32, num_quantizers=2, codebook_size=16)
    with pytest.raises(RuntimeError, match="no CPU path"):
        rvq(torch.randn(1, 8, 32))
    from vector_quantize_pytorch_b200 import ops
    with pytest.raises(RuntimeError, match="no CPU path"):
        ops.prepare_codebook(torch.randn(16, 8), False)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "vector_quantize_pytorch_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert "oracle" not in src.replace("the oracle", ""), fn


def test_state_dict_layout_matches_reference():
    """SURVEY 5: buffer names/shapes/dtypes must match so reference checkpoints load."""
    import vector_quantize_pytorch_b200 as m
    sd = m.VectorQuantize(dim=64, codebook_size=32).state_dict()
    assert list(sd) == ["_codebook.initted", "_codebook.cluster_size", "_codebook.embed_avg", "_codebook.embed"]
    assert sd["_codebook.cluster_size"].shape == (1, 32) and sd["_codebook.embed"].shape == (1, 32, 64)
    assert sd["_codebook.initted"].dtype == torch.bool and bool(sd["_codebook.initted"])
    assert torch.equal(sd["_codebook.cluster_size"], torch.ones(1, 32))
    assert torch.equal(sd["_codebook.embed"], sd["_codebook.embed_avg"])
    rvq = m.ResidualVQ(dim=32, num_quantizers=3, codebook_size=16, shared_codebook=True)
    keys = list(rvq.state_dict())
    assert "layers.0._codebook.embed" in keys and "layers.2._codebook.embed" in keys
    assert rvq.layers[0]._codebook is rvq.layers[2]._codebook
    g = m.GroupedResidualVQ(dim=64, groups=2, num_quantizers=2, codebook_size=16)
    assert "rvqs.1.layers.1._codebook.cluster_size" in g.state_dict()


def test_reference_state_dict_loads():
    """The reference's state_dict must load into ours key-for-key.  tests/golden/state_dict/reference_init.npz holds the
    reference's freshly constructed state_dicts under torch.manual_seed(0) (oracle/gen_golden.py --state-dict)."""
    import json
    import numpy as np
    import vector_quantize_pytorch_b200 as m
    z = np.load(os.path.join(ROOT, "tests", "golden", "state_dict", "reference_init.npz"))
    cases = json.loads(bytes(z["meta"]).decode())["cases"]
    assert len(cases) == 6
    for i, case in enumerate(cases):
        sa = {k: torch.from_numpy(z[f"c{i}/{k}"]) for k in case["keys"]}
        torch.manual_seed(0)
        b = getattr(m, case["cls"])(**case["kw"])
        sb = b.state_dict()
        assert list(sa) == list(sb), case
        for k in sa:  # same RNG consumption at construction -> identical initial codebooks
            assert torch.equal(sa[k], sb[k]), (case, k)
        b.load_state_dict(sa)


def test_unsupported_options_raise():
    import vector_quantize_pytorch_b200 as m
    for kw in (dict(learnable_codebook=True), dict(stochastic_sample_codes=True),
               dict(orthogonal_reg_weight=1.0), dict(affine_param=True)):
        with pytest.raises(NotImplementedError):
            m.VectorQuantize(dim=64, codebook_size=32, **kw)
    vq = m.VectorQuantize(dim=64, codebook_size=32, kmeans_init=True, kmeans_iters=3)   # supported since round 2
    assert not bool(vq._codebook.initted) and float(vq._codebook.embed.abs().sum()) == 0.0   # vqp:383, :415
    rvq = m.ResidualVQ(dim=32, num_quantizers=2, codebook_size=16, quantize_dropout=True)   # supported since round 2
    assert rvq.quantize_dropout and not m.ResidualVQ(dim=32, num_quantizers=1, codebook_size=16, quantize_dropout=True).quantize_dropout  # rvq:253
    with pytest.raises(NotImplementedError):
        m.ResidualVQ(dim=32, num_quantizers=2, codebook_size=16, beam_size=4)
