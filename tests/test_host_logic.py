"""CPU tests: host-side logic of the product package and the structural invariants that pin the scheduler oracle
(SURVEY.md Appendix A.5; no diffusers golden vectors exist -> 'parity unpinned' for the scheduler arithmetic).
No compute call of the CUDA library is made here."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from brepgen_b200 import _ffi
from brepgen_b200.models import NETS, reference_sincos_table
from brepgen_b200.sampler import shard_batch
from brepgen_b200.schedulers import DDPMScheduler, PNDMScheduler
from brepgen_b200.spec import denoiser_spec
from oracle import denoisers as O
from oracle.schedulers import DDPMOracle, PNDMOracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "brepgen_b200.h")).read()
    declared = set(re.findall(r"\b(bg_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(_ffi.SIGNATURES), declared ^ set(_ffi.SIGNATURES)
    lib = ctypes.CDLL(_ffi.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert _ffi.lib().bg_version() >= 100


def test_state_dict_keys_and_load():
    for kind, cls in NETS.items():
        for cf in (False, True):
            m = cls(cf)
            assert list(m.state_dict().keys()) == [k for k, _ in denoiser_spec(kind, cf)]
            sd = {k: torch.zeros(s) for k, s in denoiser_spec(kind, cf)}
            m.load_state_dict(sd)      # strict
    with pytest.raises(RuntimeError):
        NETS["surfpos"](False)(torch.zeros(1, 3, 6), torch.tensor([1]), None)   # no CPU path


def test_forward_rejects_wrong_shapes_before_touching_the_device():
    """the C ABI takes raw pointers, so the Python boundary validates every shape (no GPU needed to see the errors)"""
    z = torch.zeros
    cases = [
        (NETS["surfpos"](False), (z(2, 5, 7), torch.tensor([1]), None)),                                  # last dim 6
        (NETS["surfz"](False), (z(2, 5, 48), torch.tensor([1]), z(2, 4, 6), z(2, 5, dtype=torch.bool), None)),   # surfPos S
        (NETS["surfz"](False), (z(2, 5, 48), torch.tensor([1]), z(2, 5, 6), z(2, 6, dtype=torch.bool), None)),   # mask S
        (NETS["edgepos"](False), (z(2, 5, 3, 6), torch.tensor([1]), z(2, 5, 6), z(2, 5, 47), z(2, 5, dtype=torch.bool), None)),
        (NETS["edgepos"](False), (z(2, 5, 6), torch.tensor([1]), z(2, 5, 6), z(2, 5, 48), z(2, 5, dtype=torch.bool), None)),
        (NETS["edgez"](False), (z(2, 5, 3, 18), torch.tensor([1]), z(2, 5, 3, 6), z(2, 5, 6), z(2, 5, 48),
                                z(2, 5, dtype=torch.bool), None)),                                          # per-edge mask
        (NETS["edgez"](False), (z(0, 5, 3, 18), torch.tensor([1]), z(0, 5, 3, 6), z(0, 5, 6), z(0, 5, 48), None, None)),
    ]
    for m, args in cases:
        with pytest.raises(RuntimeError, match="expected|must have shape|empty|required"):
            m(*args)
    with pytest.raises(RuntimeError, match="inference-only"):
        NETS["surfpos"](False)(z(1, 3, 6), torch.tensor([1]), None, is_train=True)
    from brepgen_b200.vae import AutoencoderKL1DFastDecode, AutoencoderKLFastDecode
    for vae, bad in ((AutoencoderKLFastDecode(), z(2, 4, 4, 4)), (AutoencoderKLFastDecode(), z(2, 3, 4)),
                     (AutoencoderKL1DFastDecode(), z(2, 3, 4, 4)), (AutoencoderKL1DFastDecode(), z(0, 3, 4))):
        with pytest.raises(RuntimeError, match="expected a non-empty"):
            vae(bad)
    with pytest.raises(RuntimeError, match="no CPU path"):
        AutoencoderKLFastDecode()(z(2, 3, 4, 4))


def test_scheduler_steps_reject_mismatched_tensors():
    x = torch.zeros(2, 5, 6)
    d, p = DDPMScheduler(clip_sample=True, clip_sample_range=3), PNDMScheduler()
    with pytest.raises(RuntimeError, match="model_output has shape"):
        d.step(torch.zeros(2, 5, 7), 10, x)
    with pytest.raises(RuntimeError, match="noise has shape"):
        d.step(torch.zeros(2, 5, 6), 10, x, noise=torch.zeros(2, 5))
    with pytest.raises(RuntimeError, match="model_output_uncond has shape"):
        d.step(torch.zeros(2, 5, 6), 10, x, model_output_uncond=torch.zeros(1, 5, 6), guidance_w=0.6)
    with pytest.raises(RuntimeError, match="`out` must be"):
        d.step(torch.zeros(2, 5, 6), 10, x, out=torch.zeros(2, 5, 6, dtype=torch.float16))
    with pytest.raises(RuntimeError, match="model_output has shape"):
        p.step(torch.zeros(2, 5, 7), 995, x)
    with pytest.raises(RuntimeError):           # well-formed CPU tensors: there is no CPU path
        d.step(torch.zeros(2, 5, 6), 10, x)


def test_sincos_table_matches_oracle():
    tab = reference_sincos_table()
    ref = O.sincos_embedding(torch.arange(1000))
    assert torch.equal(tab, ref)


def test_scheduler_tables_and_coefficients_match_oracle():
    d, do = DDPMScheduler(clip_sample=True, clip_sample_range=3), DDPMOracle()
    for n in (1000, 200, 8):
        d.set_timesteps(n), do.set_timesteps(n)
        assert torch.equal(d.timesteps, do.timesteps)
        for t in d.timesteps.tolist()[:: max(1, n // 17)] + [0]:
            c, co = d.step_coefficients(t), do.coeffs(t)
            assert np.allclose(c, [float(v) for v in co], rtol=0, atol=0), (t, c, co)
    p, po = PNDMScheduler(), PNDMOracle()
    p.set_timesteps(200), po.set_timesteps(200)
    assert torch.equal(p.timesteps, po.timesteps)
    # the cross-check the reference itself encodes (sample.py:128-129,144-145): 209 entries, [:158] ends at the 255->250
    # update so that DDPM(1000)[-250:] resumes at t = 249
    ts = p.timesteps.tolist()
    assert len(ts) == 209 and ts[:12] == [995, 992, 992, 990, 990, 987, 987, 985, 985, 982, 982, 980]
    assert ts[157] == 255 and ts[158] == 250 and ts[-1] == 0
    d.set_timesteps(1000)
    assert d.timesteps[-250:].tolist()[0] == 249


def test_ddpm_oracle_invariants():
    o = DDPMOracle()
    g = torch.Generator().manual_seed(0)
    x0 = torch.rand(64, generator=g) * 2 - 1
    eps = torch.randn(64, generator=g)
    for t in (999, 500, 249, 10, 1):
        xt = o.add_noise(x0, eps, torch.tensor(t))
        sb, sa, c0, cx, sig = o.coeffs(t)
        assert torch.allclose((xt - sb * eps) / sa, x0, atol=2e-4)            # x0 recovery
        a_prev = o.acp[t - 1]
        # posterior-mean identity c_x0 + c_x sqrt(abar_t) = sqrt(abar_prev); fp32 tables lose digits in 1 - abar at small t
        assert abs(float(c0 + cx * sa) - float(a_prev ** 0.5)) < (1e-6 if t >= 249 else 2e-4)
    assert float(o.acp[0]) == pytest.approx(0.9999, abs=1e-6) and float(o.acp[999]) == pytest.approx(4.036e-5, rel=1e-3)
    assert o.coeffs(0)[4] == 0


def test_pndm_transfer_is_ddim():
    o = PNDMOracle()
    g = torch.Generator().manual_seed(1)
    x0, eps = torch.randn(32, generator=g), torch.randn(32, generator=g)
    for t, p in ((995, 990), (500, 495), (5, 0)):
        a_t, a_p = o.acp[t], o.acp[p]
        xt = a_t ** 0.5 * x0 + (1 - a_t) ** 0.5 * eps
        ref = a_p ** 0.5 * x0 + (1 - a_p) ** 0.5 * eps
        assert torch.allclose(o._prev_sample(xt, t, p, eps), ref, atol=5e-4)
        cs, ce = PNDMScheduler().transfer_coefficients(t, p)
        assert torch.allclose(cs * xt - ce * eps, ref, atol=5e-4)


def test_initial_noise_matches_reference_randn_tensor():
    """the four initial-noise draws of brepgen_b200/sampler.py (CPU generator seeded with cfg.seed, order surfPos, surfZ,
    edgePos, edgeZV) vs the reference's own randn_tensor (utils.py:60-97, exec()ed by tests/golden/make_golden_randn.py)
    under torch.manual_seed(seed): bit-identical"""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import make_golden_randn as G
    gold = np.load(os.path.join(ROOT, "tests", "golden", "randn_golden.npz"))
    gen = torch.Generator().manual_seed(G.SEED)
    for name, shape in G.SHAPES.items():
        assert np.array_equal(torch.randn(shape, generator=gen).numpy(), gold[name]), name
    # and the sampler draws them exactly like this, in this order
    src = open(os.path.join(ROOT, "brepgen_b200", "sampler.py")).read()
    assert "cpu_gen = torch.Generator().manual_seed(cfg.seed)" in src and "torch.randn(shape, generator=cpu_gen)" in src
    order = [src.index(f'noise("{n}"') for n in G.SHAPES]
    assert order == sorted(order)


def test_shard_batch_partitions():
    for gb in (1, 7, 256, 2048):
        for ws in (1, 2, 3, 8):
            spans = [shard_batch(gb, r, ws) for r in range(ws)]
            assert spans[0][0] == 0 and spans[-1][1] == gb
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1


def test_reference_arm_prints_contract_json():
    """`bench.py --impl reference` (the reference's own classes on the host cores when baseline/_ref or /root/reference
    holds network.py, else the oracle port) must print ONE JSON line with the contract keys."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--surfaces", "3", "--edges", "2"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    from oracle.reference_loader import reference_dir
    want = "reference" if reference_dir() else "port"
    assert d["impl"] == "reference" and d["value"] > 0 and d["cpu_baseline"]["kind"] == want
    if want == "reference":          # the pinned restatement is timed beside the reference's own classes
        assert d["cpu_baseline"]["port"]["kind"] == "port" and d["cpu_baseline"]["port"]["value"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_step_noise_key_depends_on_seed_rank_and_stage():
    """the Philox key of the in-kernel DDPM step noise is a 64-bit mix of (cfg.seed, rank, stage): reproducible from the
    seed, distinct across ranks and stages (SURVEY.md 8(e): per-rank independent RNG streams)"""
    from brepgen_b200.schedulers import DDPMScheduler, mix_seed
    keys = {mix_seed(s, r, st) for s in (0, 1, 1000) for r in range(8) for st in range(4)}
    assert len(keys) == 3 * 8 * 4 and all(0 <= k < 2 ** 64 for k in keys)
    assert mix_seed(7, 1, 2) == mix_seed(7, 1, 2) and mix_seed(7, 1, 2) != mix_seed(7, 2, 1)
    a, b = DDPMScheduler(), DDPMScheduler()
    a.set_noise_seed(5, 0, 3)
    b.set_noise_seed(5, 1, 3)
    assert a._philox_seed != b._philox_seed and a._philox_offset == b._philox_offset == 0
    b.set_noise_seed(5, 0, 3)
    assert a._philox_seed == b._philox_seed


def test_valid_token_flops_reduce_to_dense_when_nothing_is_masked():
    """bench.py's valid-token FLOP count (SURVEY.md 8d: the dense formulas with L -> L_valid) equals the dense-algorithmic
    count for all-valid masks and shrinks quadratically in the attention term"""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    S0, S, E, B = 50, 100, 40, 3
    dense = bench.cascade_flops_per_brep(S0, S, E)
    sm = torch.zeros(B, S, dtype=torch.bool)
    em = torch.zeros(B, S, E, dtype=torch.bool)
    assert abs(bench.cascade_flops_valid_tokens(S0, S, E, sm, em) / dense - 1) < 1e-12
    sm[:, S // 2:] = True
    em[:, S // 2:] = True
    half = bench.cascade_flops_valid_tokens(S0, S, E, sm, em)
    assert 0.25 < half / dense < 0.5           # linear terms halve, the L^2 attention term quarters
    assert abs(dense / 1e12 - 1980.1) < 0.1    # SURVEY.md 8d table: 1980.1 TF per B-rep


def test_reference_loader_runs_the_reference_classes_when_available():
    """the reference's own SurfPosNet, imported by the loader, stored by tests/golden/make_golden_loader.py: the oracle
    restatement reproduces it everywhere, and the loader does wherever the reference's network.py is present"""
    import make_golden_loader as G
    from oracle.reference_loader import load_reference_network, reference_dir
    ref = np.load(os.path.join(ROOT, "tests", "golden", "loader_golden.npz"))["surfpos"]
    assert ref.shape == (1, 4, 6)
    sd, x, t = G.case()
    with torch.no_grad():
        y = O.surfpos_forward(sd, x, t).numpy()
    assert np.abs(y - ref).max() < 1e-5 * np.abs(ref).max()
    if reference_dir() is not None:
        m = load_reference_network().SurfPosNet(False)
        m.load_state_dict(sd)
        m.eval()
        with torch.no_grad():
            y = m(x, t, None).numpy()
        assert np.abs(y - ref).max() < 1e-5 * np.abs(ref).max()


def test_load_cascade_and_config_from_eval_args():
    """sample.py:39-99: eval_config.yaml entry -> CascadeConfig, and the six checkpoints -> drop-in modules (CPU: the modules
    only hold parameters until their first CUDA forward).  The VAE checkpoints are full autoencoders: extra keys are ignored."""
    from brepgen_b200.sampler import TEXT2INT, config_from_eval_args, load_cascade
    from brepgen_b200.spec import denoiser_spec, edge_decoder_spec, surf_decoder_spec
    from brepgen_b200.synth import synth_state_dict
    args = {"save_folder": "x", "batch_size": 16, "z_threshold": 0.2, "bbox_threshold": 0.08, "num_surfaces": 60,
            "num_edges": 40, "use_cf": True, "class_label": "chair"}
    sds, store = {}, {}                  # `store` stands in for torch.load(path): no gigabytes written in a unit test
    for i, kind in enumerate(("surfpos", "surfz", "edgepos", "edgez")):
        sds[kind] = synth_state_dict(denoiser_spec(kind, True), seed=40 + i)
        args[f"{kind}_weight"] = f"{kind}.pt"
        store[args[f"{kind}_weight"]] = sds[kind]
    for name, spec, seed in (("surfvae", surf_decoder_spec(), 50), ("edgevae", edge_decoder_spec(), 51)):
        sds[name] = synth_state_dict(spec, seed=seed)
        full = {**sds[name], "encoder.conv_in.weight": torch.zeros(4, 3, 3), "quant_conv.weight": torch.zeros(6, 6, 1)}
        args[f"{name}_weight"] = f"{name}.pt"
        store[args[f"{name}_weight"]] = full

    cfg = config_from_eval_args(args, schedule="ddpm", ddpm_steps=4)
    assert (cfg.batch_size, cfg.num_surfaces, cfg.num_edges, cfg.use_cf, cfg.class_label) == (16, 60, 40, True, TEXT2INT["chair"])
    assert cfg.bbox_threshold == 0.08 and cfg.schedule == "ddpm" and cfg.ddpm_steps == 4
    with pytest.raises(KeyError):
        config_from_eval_args({**args, "class_label": "spaceship"})
    with pytest.raises(TypeError):
        config_from_eval_args(args, no_such_field=1)
    assert config_from_eval_args({**args, "use_cf": False, "class_label": []}).class_label == 0

    casc = load_cascade(args, device="cpu", load=store.__getitem__)
    for kind in ("surfpos", "surfz", "edgepos", "edgez"):
        got = casc.m[kind].state_dict()
        assert set(got) == set(sds[kind]) and all(torch.equal(got[k], sds[kind][k]) for k in got)
        assert not casc.m[kind].training
    for mod, name in ((casc.surf_vae, "surfvae"), (casc.edge_vae, "edgevae")):
        got = mod.state_dict()
        assert all(torch.equal(got[k], sds[name][k]) for k in sds[name] if k in got) and "encoder.conv_in.weight" not in got
    # a denoiser checkpoint with a missing key is an error (strict load, like the reference)
    bad = dict(sds["surfpos"])
    bad.pop(next(iter(bad)))
    store[args["surfpos_weight"]] = bad
    with pytest.raises(RuntimeError):
        load_cascade(args, device="cpu", load=store.__getitem__)
