"""CPU: host-side logic -- the C-ABI library loads and exports every declared symbol, module
state_dict layout, neuralop shim, loud failure without CUDA."""
import ctypes
import os
import re

import pytest
import torch

import dlwp_benchmark_b200 as pkg
from dlwp_benchmark_b200 import _lib
from oracle import spectral_oracle as so

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "spectral_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(sb200_[a-z0-9_]+)\s*\(", hdr)))


def test_library_exports_every_declared_symbol():
    lib = ctypes.CDLL(_lib.LIB_PATH)
    syms = _declared_symbols()
    assert len(syms) >= 14
    for s in syms:
        assert hasattr(lib, s), s
    assert set(syms) == set(_lib.SIGNATURES), set(syms) ^ set(_lib.SIGNATURES)
    assert _lib.load().sb200_version() >= 100


def test_no_cpu_path():
    m = pkg.FNO(n_modes=(6, 6), hidden_channels=8, in_channels=1, out_channels=1, lifting_channels=16,
                projection_channels=16, n_layers=2)
    with pytest.raises(_lib.SpectralB200Error):
        m(torch.randn(1, 1, 16, 16))
    a = pkg.AFNO2D(16, num_blocks=4)
    with pytest.raises(_lib.SpectralB200Error):
        a(torch.randn(1, 8, 8, 16))
    with pytest.raises(_lib.SpectralB200Error):
        pkg.SpectralConv(4, 4, (6, 6), fft_norm="forward")(torch.randn(1, 4, 16, 16))


def test_state_dict_layout_dense():
    m = pkg.FNO(n_modes=(12, 12), hidden_channels=32, in_channels=10, out_channels=1, lifting_channels=256,
                projection_channels=256, n_layers=4)
    sd = m.state_dict()
    assert tuple(sd["fno_blocks.convs.weight.0.tensor"].shape) == (32, 32, 12, 7, 2)
    assert tuple(sd["fno_blocks.convs.bias"].shape) == (4, 32, 1, 1)
    assert tuple(sd["fno_blocks.fno_skips.3.weight"].shape) == (32, 32, 1, 1)
    assert tuple(sd["lifting.fcs.0.weight"].shape) == (256, 10, 1, 1)
    assert tuple(sd["lifting.fcs.1.weight"].shape) == (32, 256, 1, 1)
    assert tuple(sd["projection.fcs.1.weight"].shape) == (1, 256, 1, 1)
    n = sum(p.numel() for p in m.parameters())
    assert n == so.fno_param_count((12, 12), 10, 32, 256, 256, 1, 4)
    # every key is consumed by the oracle's forward: same layout on both sides
    want = {"lifting.fcs.0.weight", "lifting.fcs.0.bias", "lifting.fcs.1.weight", "lifting.fcs.1.bias",
            "projection.fcs.0.weight", "projection.fcs.0.bias", "projection.fcs.1.weight", "projection.fcs.1.bias",
            "fno_blocks.convs.bias"}
    want |= {f"fno_blocks.convs.weight.{l}.tensor" for l in range(4)}
    want |= {f"fno_blocks.fno_skips.{l}.weight" for l in range(4)}
    assert set(sd) == want


@pytest.mark.parametrize("hc,label", [(38, 0.999), (54, 2.002), (217, 31.948)])
def test_reference_size_labels_on_module(hc, label):
    m = pkg.FNO(n_modes=(12, 12), hidden_channels=hc, in_channels=10, out_channels=1, n_layers=4)
    assert abs(sum(p.numel() for p in m.parameters()) / 1e6 - label) < 6e-4


def test_state_dict_layout_tucker():
    m = pkg.TFNO(n_modes=(16, 16), hidden_channels=64, in_channels=1, out_channels=1, n_layers=2, rank=0.8)
    sd = m.state_dict()
    assert tuple(sd["fno_blocks.convs.weight.0.core"].shape) == (60, 60, 15, 8, 2)
    assert tuple(sd["fno_blocks.convs.weight.1.factors.factor_0"].shape) == (64, 60, 2)
    assert tuple(sd["fno_blocks.convs.weight.1.factors.factor_3"].shape) == (9, 8, 2)
    # reconstruction agrees with the oracle's einsum
    tw = m.fno_blocks.convs.weight[0]
    ref = so.tucker_to_dense(torch.view_as_complex(tw.core.detach()),
                             [torch.view_as_complex(f.detach()) for f in tw.factors])
    assert torch.allclose(tw.to_dense_complex(), ref, atol=1e-5, rtol=1e-4)


def test_fno_with_rank_kwarg_is_dense():
    # src/nsbench/models/fno/fno.py:205 builds FNO(..., rank=rank): factorization None => dense
    m = pkg.FNO(n_modes=(12, 12), hidden_channels=8, in_channels=10, out_channels=1, n_layers=1, rank=0.5)
    assert "fno_blocks.convs.weight.0.tensor" in m.state_dict()


def test_unknown_kwargs_are_swallowed():
    pkg.FNO(n_modes=(6, 6), hidden_channels=4, type="FNOModule", name="x")


def test_afno_state_dict_matches_reference_layout():
    a = pkg.AFNO2D(64, num_blocks=8, hidden_size_factor=2)
    shapes = {k: tuple(v.shape) for k, v in a.state_dict().items()}
    assert shapes == {"w1": (2, 8, 8, 16), "b1": (2, 8, 16), "w2": (2, 8, 16, 8), "b2": (2, 8, 8)}


def test_mode_block_matches_oracle():
    from dlwp_benchmark_b200.plan import fno_mode_block
    for H, n in ((64, 12), (64, 16), (256, 32), (16, 6), (16, 16), (8, 12)):
        lo, My = so.retained_rows(H, n)
        assert fno_mode_block(H, 64, (n, 7)) == (lo - H // 2, My, 7)


# root of a checkout of amazon-science/dlwp-benchmark, the project whose wrappers the shim serves (not vendored here)
REFERENCE = os.environ.get("DLWP_BENCHMARK_REFERENCE", "")


@pytest.mark.skipif(not REFERENCE or not os.path.isdir(os.path.join(REFERENCE, "src")),
                    reason="set DLWP_BENCHMARK_REFERENCE to a checkout of amazon-science/dlwp-benchmark")
def test_reference_wrappers_import_on_the_shim():
    """The UNMODIFIED reference wrapper modules import and construct on top of the shim."""
    import importlib.util
    pkg.install_neuralop_shim(force=True)
    path = os.path.join(REFERENCE, "src", "nsbench", "models", "fno", "fno.py")
    spec = importlib.util.spec_from_file_location("_ref_ns_fno", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    w = mod.FNOModule(n_modes=[12, 12], in_channels=1, hidden_channels=32, lifting_channels=256,
                      projection_channels=256, out_channels=1, n_layers=4, type="FNOModule", name="t")
    assert isinstance(w.fno, pkg.FNO)
    assert "fno.fno_blocks.convs.weight.0.tensor" in w.state_dict()
    t = mod.TFNO2DModule(n_modes=[12, 12], in_channels=1, hidden_channels=8, lifting_channels=16,
                         projection_channels=16, out_channels=1, n_layers=1, rank=0.5, context_size=2)
    assert "fno.fno_blocks.convs.weight.0.tensor" in t.state_dict()     # dense: the reference's own quirk


def test_neuralop_imports_resolve_to_the_shim():
    """The reference wrappers do `from neuralop.models import FNO, TFNO` (src/nsbench/models/fno/fno.py:7): with the
    shim installed those names, and neuralop's SpectralConv, are this package's classes; the shim refuses to shadow a
    real neuralop unless forced."""
    import sys
    import types
    saved = {k: v for k, v in sys.modules.items() if k.split(".")[0] == "neuralop"}
    try:
        for k in saved:
            del sys.modules[k]
        pkg.install_neuralop_shim()
        from neuralop.models import FNO, TFNO
        from neuralop.layers.spectral_convolution import SpectralConv
        assert (FNO, TFNO, SpectralConv) == (pkg.FNO, pkg.TFNO, pkg.SpectralConv)
        w = FNO(n_modes=[12, 12], in_channels=1, hidden_channels=8, lifting_channels=16, projection_channels=16,
                out_channels=1, n_layers=1, rank=0.5)
        assert "fno_blocks.convs.weight.0.tensor" in w.state_dict()        # FNO(..., rank=rank) stays dense
        pkg.install_neuralop_shim()                                         # installing over the shim is fine
        sys.modules["neuralop"] = types.ModuleType("neuralop")               # a real neuralop imported first
        with pytest.raises(RuntimeError):
            pkg.install_neuralop_shim()
        assert pkg.install_neuralop_shim(force=True).models.FNO is pkg.FNO
    finally:
        for k in [k for k in sys.modules if k.split(".")[0] == "neuralop"]:
            del sys.modules[k]
        sys.modules.update(saved)


def test_sequence_forward_is_the_reference_loop():
    """sequence_forward == FNOModule.forward (src/nsbench/models/fno/fno.py:29-43): teacher forcing for the first
    `teacher_forcing_steps` frames, closed loop afterwards, frames stacked on dim 1 (any callable model)."""
    step = lambda x: 0.5 * x + 1.0
    x = torch.randn(2, 7, 1, 4, 4)
    for tf in (0, 1, 3, 7, 50):
        outs, x_t = [], None
        for t in range(x.shape[1]):                     # literal transcription of the reference loop
            x_t = x[:, t] if t < tf else x_t
            if x_t is None:                             # tf == 0: the reference would fail here too (x_t undefined)
                break
            x_t = step(x_t)
            outs.append(x_t)
        if tf == 0:
            continue
        want = torch.stack(outs, dim=1)
        assert torch.equal(pkg.sequence_forward(step, x, teacher_forcing_steps=tf), want)


def test_rollout_engine_has_no_cpu_path():
    m = pkg.FNO(n_modes=(6, 6), hidden_channels=8, in_channels=1, out_channels=1, lifting_channels=16,
                projection_channels=16, n_layers=2)
    with pytest.raises(_lib.SpectralB200Error):
        pkg.Rollout(m)(torch.randn(1, 1, 16, 16), 3)


def test_bench_reads_traffic_from_the_committed_capture():
    """bench.py fills roofline.traffic from profiles/: the file it names must exist and hold the kernels it looks up."""
    import bench
    for name, approx in (("analysis_fused", None), ("modes_gemm2", None), ("coldft_inv2", None),
                         ("tc_pointwise_kernel<3, 1, 0", None), ("tc_pointwise_kernel<3, 3, 0", None),
                         ("tc_wgrad_kernel<3, 0>", 8 * 64 * 64 * 64 * 64)):
        t = bench._ncu_traffic(name, approx)
        assert isinstance(t, int) and t > 0, name
    # the skip-conv weight gradient reads g and x once each (2 x 67 MB), not the 336 MB of the projection-head launch
    assert bench._ncu_traffic("tc_wgrad_kernel<3, 0>", 8 * 64 * 64 * 64 * 64) < 200e6
    assert bench._cpu_sample(bench.WORKLOADS["cfg2"]) == 64 and bench._cpu_sample(bench.WORKLOADS["cfg3"]) == 2


def test_bench_dump_outputs_stays_within_its_limit(tmp_path):
    """bench.py --dump-outputs: one .npy per array, float32 (float64 kept), whole while the arrays fit the limit;
    beyond it the largest array becomes a flat sample at distinct indices, the same ones on every call."""
    import numpy as np
    import bench
    g = torch.Generator().manual_seed(0)
    arrays = {"loss": torch.tensor(0.25), "w": torch.randn(3, 4, dtype=torch.float64, generator=g),
              "h": torch.randn(64, dtype=torch.float16, generator=g), "none": None,
              "big": torch.randn(50_000, generator=g)}
    bench.dump_outputs(str(tmp_path / "whole"), arrays)
    got = {f[:-4]: np.load(tmp_path / "whole" / f) for f in os.listdir(tmp_path / "whole")}
    assert set(got) == {"loss", "w", "h", "big"}
    assert got["loss"].dtype == np.float32 and got["loss"].shape == () and got["loss"] == 0.25
    assert got["w"].dtype == np.float64 and np.array_equal(got["w"], arrays["w"].numpy())
    assert got["h"].dtype == np.float32 and np.array_equal(got["h"], arrays["h"].float().numpy())
    assert np.array_equal(got["big"], arrays["big"].numpy())
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays, limit=40_000)
        assert sum(os.path.getsize(tmp_path / run / f) for f in os.listdir(tmp_path / run)) <= 40_000
    a, b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert 5_000 < a.size < 10_000 and np.array_equal(a, b) and np.isin(a, got["big"]).all()
    assert np.unique(a).size == a.size                     # distinct indices (the values are distinct normals)
    assert np.array_equal(np.load(tmp_path / "a" / "w.npy"), got["w"])
