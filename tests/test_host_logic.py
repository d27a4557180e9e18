"""Host-side logic that needs no GPU: tensor-core eligibility, checkpoint ingestion, constructor guards."""
import os

import pytest
import torch


class HParams:  # stands in for the omegaconf object Lightning pickles next to the tensors (not a tensor-only pickle)
    tile = 0


def test_tc_supported_limits(pkg):
    """ADVICE r1: 'auto' must only pick the tensor-core path for architectures its kernels accept: the LayerNorm
    epilogue of gemm_tc.cu holds a whole 128 x C fp32 row tile, C <= 188."""
    from grl_image_restoration_b200 import tc

    assert tc.supported(180, 3, 3) and tc.supported(64, 2, 2) and tc.supported(128, 2, 2)
    assert not tc.supported(192, 3, 3)   # C > LN_MAX_C
    assert not tc.supported(256, 4, 4)
    assert not tc.supported(288, 6, 6)
    assert not tc.supported(180, 2, 2)   # head_dim 45 > 32
    assert not tc.supported(182, 7, 7)   # C % 4 != 0
    assert tc.LN_MAX_C == 188


def test_auto_precision_falls_back_for_wide_models(pkg):
    cfg = pkg.configs.micro_config(embed_dim=192, heads=3, window=8, stripe=(8, 16), df=2, img_size=32)
    m = pkg.GRL(**cfg)
    assert m.set_precision("auto") == "fp32"
    with pytest.raises(RuntimeError, match="tensor-core path"):
        m.set_precision("fp16")
    cfg = pkg.configs.micro_config(embed_dim=36, heads=2)
    assert pkg.GRL(**cfg).set_precision("auto") == "fp16"


def test_pretrained_sizes_rejected(pkg):
    cfg = pkg.configs.micro_config()
    with pytest.raises(NotImplementedError):
        pkg.GRL(**cfg, pretrained_window_size=[8, 8])
    with pytest.raises(NotImplementedError):
        pkg.GRL(**cfg, pretrained_stripe_size=[0, 16])


def test_checkpoint_ingestion_variants(pkg, tmp_path):
    """tools/trainer.py:93-115: Lightning 'state_dict' with engine buffers and model.* prefix, extra engine keys, a
    'params' wrapper, a bare state dict; files are read with weights_only=False (hyper_parameters are pickled)."""
    from grl_image_restoration_b200 import checkpoint

    cfg = pkg.configs.micro_config()
    src = pkg.GRL(**cfg)
    with torch.no_grad():
        for p in src.parameters():
            p.add_(0.01)
    sd = src.state_dict()

    def fresh():
        return pkg.GRL(**cfg)

    def same(m):
        return all(torch.equal(v, sd[k]) for k, v in m.state_dict().items())

    # 1. Lightning checkpoint: model.* keys + engine buffers + other engine state + reference-style buffers
    pl = {"model." + k: v.clone() for k, v in sd.items()}
    pl.update(current_val_metric=torch.zeros(1), best_val_metric=torch.zeros(1), best_iter=torch.zeros(1))
    pl["loss.weight"] = torch.ones(3)
    pl["model.index_w"] = torch.zeros(4, dtype=torch.int64)
    pl["model.mask_sh_a2w"] = torch.zeros(4)

    path = str(tmp_path / "last.ckpt")
    torch.save({"state_dict": pl, "hyper_parameters": HParams(), "epoch": 3}, path)
    m = fresh()
    checkpoint.load_reference_checkpoint(m, path)
    assert same(m)
    # 2. 'params' wrapper
    m = fresh()
    checkpoint.load_reference_checkpoint(m, {"params": {k: v.clone() for k, v in sd.items()}})
    assert same(m)
    # 3. bare state dict
    m = fresh()
    checkpoint.load_reference_checkpoint(m, {k: v.clone() for k, v in sd.items()})
    assert same(m)


def test_build_stamp_tracks_nvcc_defines(pkg, monkeypatch):
    """An A/B build (GRL_NVCC_DEFINES) must never be mistaken for the production library: the build records the defines it
    was compiled with and a mismatch makes the library stale."""
    from grl_image_restoration_b200 import build as b

    if not os.path.exists(b.LIB):
        pytest.skip("library not built")
    monkeypatch.delenv("GRL_NVCC_DEFINES", raising=False)
    monkeypatch.setattr(b, "_stamp", lambda: "")
    assert not b._stale()
    monkeypatch.setenv("GRL_NVCC_DEFINES", "-DGRL_A2_DIAG_NOEXP")
    assert b._stale()  # production stamp, A/B build requested
    monkeypatch.setattr(b, "_stamp", lambda: "-DGRL_A2_DIAG_NOEXP")
    assert not b._stale()
    monkeypatch.delenv("GRL_NVCC_DEFINES")
    assert b._stale()  # A/B library left behind, production requested


def _run_bench(args, env_extra=None):
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, **(env_extra or {}))
    p = subprocess.run([sys.executable, os.path.join(root, "bench.py")] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                       text=True, env=env, timeout=600, cwd=root)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.split("\n") if l.strip()]
    return [json.loads(l) for l in lines]


def test_bench_reference_arm_contract():
    """bench.py --impl reference: ONE JSON line on stdout (CPU only, the reference's own forward), same metric / unit / config
    keys as our arm, a cpu_baseline that says what was sampled, an e2e block with zero copies; ranks > 0 print nothing."""
    out = _run_bench(["--impl", "reference", "--workload", "cfg1", "--steps", "1", "--warmup", "0"])
    assert len(out) == 1
    d = out[0]
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "Mpix/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["value"] > 0 and d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and "64x64" in d["cpu_baseline"]["sample"]
    assert "64x64" in d["config"]["workload"]  # the line names the bounded sample it measured
    assert d["e2e"] == {"value": d["value"], "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert _run_bench(["--impl", "reference", "--gpus", "2", "--workload", "cfg1", "--steps", "1", "--warmup", "0"],
                      {"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}) == []


def test_bench_dump_outputs(tmp_path):
    """--dump-outputs writes the last timed step's output as float32 .npy; an output over the size budget becomes the same
    seeded, sorted sample of its elements on every call."""
    import subprocess
    import sys

    import numpy as np

    out = _run_bench(["--impl", "reference", "--workload", "cfg1", "--steps", "1", "--warmup", "0",
                      "--dump-outputs", str(tmp_path / "ref")])
    assert len(out) == 1
    y = np.load(tmp_path / "ref" / "output.npy")
    assert y.dtype == np.float32 and y.shape == (1, 3, 128, 128) and np.isfinite(y).all()

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import sys, torch, bench\n"
            "t = torch.arange(10**6, dtype=torch.float64).reshape(10, 100, 1000)\n"
            "bench.dump_outputs(sys.argv[1], {'a': t, 'b': t}, max_bytes=2 * (4096 + 4 * 1000))\n"
            "bench.dump_outputs(sys.argv[2], {'a': t, 'b': t[0, :2, :400]}, max_bytes=2 * (4096 + 4 * 1000))\n")
    subprocess.run([sys.executable, "-c", code, str(tmp_path / "s1"), str(tmp_path / "s2")], check=True, cwd=root)
    a = np.load(tmp_path / "s1" / "a.npy")
    assert a.dtype == np.float32 and a.shape == (1000,)
    assert (np.diff(a) >= 0).all() and a.min() >= 0 and a.max() < 10**6 and len(np.unique(a)) > 900
    assert np.array_equal(a, np.load(tmp_path / "s1" / "b.npy")) and np.array_equal(a, np.load(tmp_path / "s2" / "a.npy"))
    b = np.load(tmp_path / "s2" / "b.npy")  # within its share: written whole, shape kept
    assert b.shape == (2, 400) and np.array_equal(b, np.arange(2000, dtype=np.float32).reshape(2, 1000)[:, :400])


@pytest.mark.parametrize("kw,size", [(dict(), 32), (dict(embed_dim=60, heads=3, window=8, stripe=(8, 16), df=2), 48),
                                     (dict(window=4, stripe=(16, 8), df=4, depth=2), 32)])
def test_attention_counts_match_the_materialised_attention(pkg, oracle, monkeypatch, kw, size):
    """flops.attention_counts (the numerator of bench.py's roofline) == the number of score elements the oracle actually
    puts through softmax in one forward (it materialises every (N1 x N2) attention map), and f_attn = 4 head_dim per element."""
    from grl_image_restoration_b200 import flops

    cfg = pkg.configs.micro_config(img_size=size, **kw)
    sd = oracle.synth_state_dict(cfg, seed=0, style="init")
    seen = []
    real = torch.softmax

    def counting(t, dim=-1, **k):
        seen.append(tuple(t.shape))
        return real(t, dim=dim, **k)

    monkeypatch.setattr(torch, "softmax", counting)
    with torch.no_grad():
        oracle.grl_forward(sd, cfg, oracle.synth_input((1, 3, size, size), seed=1))
    monkeypatch.undo()
    total = sum(int(torch.tensor(s).prod()) for s in seen)
    counts = flops.attention_counts(cfg, (size, size))
    assert counts["score_elems"] == total
    d = cfg["embed_dim"] // 2 // cfg["num_heads_window"][0]
    assert counts["f_attn"] == 4 * d * total and counts["f_qk"] * 2 == counts["f_attn"]


def test_attention_counts_of_the_baseline_configs(pkg):
    """The per-image figures DESIGN.md section 5 and the bench line quote (GFLOP of QK^T + PV, G score elements)."""
    from grl_image_restoration_b200 import flops

    want = {"cfg4": (("base", "sr", 4, 256), 2899.1029248, 24.15919104), "cfg2": (("small", "sr", 4, 256), 412.316860416, 3.221225472),
            "cfg3": (("base", "dn", 1, 256), 4831.838208, 40.2653184), "cfg5": (("base", "deblur", 1, 480), 2388.7872, 19.90656)}
    for name, ((v, t, s, sz), gf, ge) in want.items():
        c = flops.attention_counts(pkg.configs.grl_config(v, t, s, sz), (sz, sz))
        assert abs(c["f_attn"] / 1e9 - gf) < 1e-6 and abs(c["score_elems"] / 1e9 - ge) < 1e-6, name
