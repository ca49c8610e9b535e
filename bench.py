#!/usr/bin/env python
"""bench.py -- B-reps/sec of the 1000-step-per-stage ABC cascade (BASELINE.json), one process per GPU.

    python bench.py --gpus 1 --steps 3 --warmup 3
    python bench.py --gpus 1 --steps 3 --warmup 3 --dump-outputs DIR   # + the last timed step's outputs as DIR/*.npy
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
    python bench.py --impl reference ...        # the reference's own classes on the host cores (baseline/_ref), same metric

Workload (BASELINE.json configs[2]; SURVEY.md 8d item 3): full ABC cascade, batch 256 per GPU, S0 = 50 -> S = 100 faces,
E = 40 edges/face (edge-stage sequences of 4000 tokens), dense masks, random-init weights, Gaussian inputs.
One bench "step" = one pass of the whole cascade (SurfPos -> SurfZ -> EdgePos -> EdgeZ, every stage a DDPM loop of
T = --steps-per-stage network evaluations + fused scheduler updates, then both VAE decodes when available) over one batch.
Every DDPM step of a stage costs the same work whatever its t, so the metric (defined at T = 1000) is reported as
    value = n_gpus * B / (seconds_per_step * 1000 / T)
with T stated in `config`; `--steps-per-stage 1000` runs the literal thing (minutes per step at B = 256).
Weak scaling: every rank runs its own batch of B; no collective on the hot path.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "B-reps/sec (1000-step ABC cascade)"
UNIT = "B-reps/s"
KINDS = ("surfpos", "surfz", "edgepos", "edgez")
DUMP_BYTES = 64 * 10**6


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="B-reps per GPU")
    ap.add_argument("--surfaces", type=int, default=50)
    ap.add_argument("--edges", type=int, default=40)
    ap.add_argument("--steps-per-stage", type=int, default=4)
    ap.add_argument("--cf", action="store_true", help="classifier-free guidance (furniture config: 2x forward batch, no late increase)")
    ap.add_argument("--schedule", default="ddpm", choices=["ddpm", "reference"],
                    help="ddpm = N DDPM steps per stage (the metric's definition); reference = the shipped PNDM/DDPM hybrid")
    ap.add_argument("--masks", default="dense", choices=["dense", "flow", "ragged"],
                    help="dense = every slot valid, the metric's dense-FLOP mode; flow = run both dedups (sample.py:159-183,242-261) "
                         "and mask what they remove; ragged = synthetic masks shaped like a trained model's output (1/8..1/2 of "
                         "the faces, 3..E/3 edges per face valid; random-init weights never produce duplicates for flow to remove)")
    ap.add_argument("--compact", type=int, default=1, choices=[0, 1],
                    help="mask-aware token compaction in the denoisers (1, default) or the dense layout with masking only (0)")
    ap.add_argument("--workload", default="cascade", choices=["cascade", "surfpos"],
                    help="cascade = the metric's workload (BASELINE configs[2]); surfpos = BASELINE configs[1]: SurfPosNet, "
                         "1000-step DDPM, 30 face tokens, batch 64 (first stage only), eager loop vs CUDA-graph replay")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the cascade outputs of the last one as DIR/<name>.npy (float32; rank 0; "
                         f"when they exceed {DUMP_BYTES // 10**6} MB together, the same seeded sample of batch rows of each)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "cascade"):
        ap.error("--dump-outputs applies to the cascade workload of --impl b200")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 1590.0, 1400.0, "fallback"


# ------------------------------------------------------------------------------------------------ algorithmic FLOPs
def encoder_flops(L):   # SURVEY.md 8(d): per sample, per forward, dense, mul-add = 2
    return 12 * (L * 7_864_320 + 3072 * L * L)


def mlp_flops(d_in, d_out):
    return 2 * d_in * 768 + 2 * 768 * d_out


def cascade_flops_valid_tokens(S0, S, E, surf_mask, edge_mask, steps=1000):
    """SURVEY.md 8(d): the same formulas with L -> L_valid per sample (mean over the batch).  SurfPos has no mask; SurfZ attends
    over the valid faces; EdgePos over (valid faces) x E (face mask repeated, network.py:1268); EdgeZ over the valid edges."""
    sv = (~surf_mask).sum(1).double()
    ev = (~edge_mask).sum((1, 2)).double()
    enc = lambda L: 12 * (L * 7_864_320 + 3072 * L * L)
    sp = lambda s: encoder_flops(s) + s * (mlp_flops(6, 768) + mlp_flops(768, 6))
    sz = enc(sv) + sv * (mlp_flops(48, 768) + mlp_flops(6, 768) + mlp_flops(768, 48))
    ep = enc(sv * E) + sv * (mlp_flops(6, 768) + mlp_flops(48, 768)) + sv * E * (mlp_flops(6, 768) + mlp_flops(768, 6))
    ez = enc(ev) + sv * (mlp_flops(6, 768) + mlp_flops(48, 768)) + ev * (2 * mlp_flops(6, 768) + mlp_flops(12, 768) + mlp_flops(768, 18))
    return float(steps * (0.75 * sp(S0) + 0.25 * sp(S) + (sz + ep + ez).mean()))


def cascade_flops_per_brep(S0, S, E, steps=1000):
    sp = lambda s: encoder_flops(s) + s * (mlp_flops(6, 768) + mlp_flops(768, 6))
    sz = encoder_flops(S) + S * (mlp_flops(48, 768) + mlp_flops(6, 768) + mlp_flops(768, 48))
    ep = encoder_flops(S * E) + S * (mlp_flops(6, 768) + mlp_flops(48, 768)) + S * E * (mlp_flops(6, 768) + mlp_flops(768, 6))
    ez = encoder_flops(S * E) + S * (mlp_flops(6, 768) + mlp_flops(48, 768)) + S * E * (2 * mlp_flops(6, 768) + mlp_flops(12, 768) + mlp_flops(768, 18))
    return steps * (0.75 * sp(S0) + 0.25 * sp(S) + sz + ep + ez)


# ------------------------------------------------------------------------------------------------ CPU baseline
def cpu_reference_sample(S0, S, E, reps, threads=None, inner_warm=True, kind="auto"):
    """Times the reference's algorithm for this path on the host cores: per stage, one network forward + DDPM scheduler
    step at batch 1, `reps` timed repetitions after one warm-up; extrapolated to the 4 x 1000-step cascade.

    kind = "reference": the reference's OWN classes (SurfPosNet ... EdgeZNet of network.py:1066-1393, stock code path:
    nn.TransformerEncoder etc., eval(), no_grad), imported unmodified from baseline/_ref/network.py (or /root/reference)
    through oracle/reference_loader.py; "port": oracle/denoisers.py (the pinned restatement); "auto": the reference when
    its file is present, else the port.  The scheduler step is oracle/schedulers.py in both cases (diffusers is absent
    offline; the step is < 0.1 % of the time).  Returns (B-reps/s, cores, description, kind_used)."""
    from brepgen_b200.spec import denoiser_spec
    from brepgen_b200.synth import synth_state_dict
    from oracle import denoisers as O
    from oracle.reference_loader import load_reference_network
    from oracle.schedulers import DDPMOracle

    cores = threads or (os.cpu_count() or 1)
    torch.set_num_threads(cores)
    net = load_reference_network(required=False) if kind in ("auto", "reference") else None
    if kind == "reference" and net is None:
        raise RuntimeError("reference classes requested but neither baseline/_ref/network.py nor /root/reference exists")
    used = "reference" if net is not None else "port"
    ref_cls = None if net is None else {"surfpos": net.SurfPosNet, "surfz": net.SurfZNet, "edgepos": net.EdgePosNet,
                                        "edgez": net.EdgeZNet}
    orc = DDPMOracle()
    g = torch.Generator().manual_seed(0)
    r = lambda *s: torch.randn(*s, generator=g)
    t = torch.tensor([500])
    per = {}
    with torch.no_grad():
        for name, knd, shape in (("surfpos@S0", "surfpos", (1, S0, 6)), ("surfpos@S", "surfpos", (1, S, 6)),
                                 ("surfz", "surfz", (1, S, 48)), ("edgepos", "edgepos", (1, S, E, 6)),
                                 ("edgez", "edgez", (1, S, E, 18))):
            sd = synth_state_dict(denoiser_spec(knd, False), seed=1)
            x = r(*shape)
            sP, sZ, eP = r(1, shape[1], 6), r(1, shape[1], 48), r(1, shape[1], E, 6)
            fm = torch.zeros(1, shape[1], dtype=torch.bool)
            em = torch.zeros(1, shape[1], E, dtype=torch.bool)
            if ref_cls is not None:
                m = ref_cls[knd](False)
                m.load_state_dict(sd)
                m.eval()
                fwd = {"surfpos": lambda: m(x, t, None), "surfz": lambda: m(x, t, sP, fm, None),
                       "edgepos": lambda: m(x, t, sP, sZ, fm, None), "edgez": lambda: m(x, t, eP, sP, sZ, em, None)}[knd]
            else:
                fwd = {"surfpos": lambda: O.surfpos_forward(sd, x, t), "surfz": lambda: O.surfz_forward(sd, x, t, sP, fm),
                       "edgepos": lambda: O.edgepos_forward(sd, x, t, sP, sZ, fm),
                       "edgez": lambda: O.edgez_forward(sd, x, t, eP, sP, sZ, em)}[knd]
            if inner_warm:
                orc.step(fwd(), 500, x, r(*shape))
            t0 = time.perf_counter()
            for _ in range(reps):
                orc.step(fwd(), 500, x, r(*shape))
            per[name] = (time.perf_counter() - t0) / reps
            del sd
    sec_per_brep = 750 * per["surfpos@S0"] + 250 * per["surfpos@S"] + 1000 * (per["surfz"] + per["edgepos"] + per["edgez"])
    what = ("the reference's own classes (network.py:1066-1393, stock nn.TransformerEncoder path)" if used == "reference"
            else "oracle port (oracle/denoisers.py)")
    desc = (f"{what}, fp32 torch CPU, {cores} threads, batch 1, {reps} timed (forward + DDPM step) per stage after warm-up; "
            "s/step: " + ", ".join(f"{k}={v:.3f}" for k, v in per.items()) + "; extrapolated to 750/250 + 3x1000 steps")
    return 1.0 / sec_per_brep, cores, desc, used


def best_cpu_threads():
    """torch's intra-op pool does not scale to every hardware thread of a many-core host on these small matrices: probe
    a few thread counts on one encoder-sized matmul chain and keep the fastest (all of them are 'threads it can use')."""
    n = os.cpu_count() or 1
    a, w = torch.randn(4000, 768), torch.randn(2304, 768)
    best, best_t = n, None
    for k in sorted({n, max(1, n // 2), max(1, n // 4), min(n, 32), min(n, 16), min(n, 8)}):
        torch.set_num_threads(k)
        (a @ w.t()).sum()
        t0 = time.perf_counter()
        for _ in range(3):
            q = a @ w.t()
            torch.softmax(q[:, :768] @ q[:, 768:1536].t(), -1).sum()
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = k, dt
    return best


def dump_outputs(out, d):
    """every output of Cascade.run has the batch first: keep the same seeded rows of each so that the sample stays one
    set of whole B-reps, as many as fit DUMP_BYTES (npy headers included)"""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    B = next(iter(out.values())).shape[0]
    row_bytes = sum(v[0].numel() * 4 for v in out.values())
    n = min(B, (DUMP_BYTES - 4096 * len(out)) // row_bytes)
    rows = torch.randperm(B, generator=torch.Generator().manual_seed(0))[:n].sort().values
    for k, v in out.items():
        np.save(os.path.join(d, f"{k}.npy"), v[rows.to(v.device)].float().cpu().numpy())


# ------------------------------------------------------------------------------------------------ clocks sampler
class Clocks(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._halt = index, [], threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._halt.wait(0.2)

    def finish(self):
        self._halt.set()
        self.join(timeout=3)
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        mx = max((int(r[1]) for r in self.rows if r[1].isdigit()), default=None)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ main arms
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    S0, E = args.surfaces, args.edges
    S = 2 * S0
    vals = []
    nthr = best_cpu_threads()
    for _ in range(max(args.warmup, 0)):
        cpu_reference_sample(S0, S, E, 1, nthr, inner_warm=False)
    if args.warmup == 0:
        cpu_reference_sample(S0, S, E, 1, nthr, inner_warm=False)      # never time a cold first pass
    t0 = time.perf_counter()
    for _ in range(args.steps):
        v, cores, desc, used = cpu_reference_sample(S0, S, E, 1, nthr, inner_warm=False)
        vals.append(v)
    port = None
    if used == "reference":     # the pinned restatement beside it (one pass), so both CPU numbers are on record
        pv, _, pdesc, _ = cpu_reference_sample(S0, S, E, 1, nthr, inner_warm=True, kind="port")
        port = {"value": pv, "unit": UNIT, "kind": "port", "sample": pdesc}
    ms = (time.perf_counter() - t0) / max(args.steps, 1) * 1e3
    v = sum(vals) / len(vals)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"abc_cascade S0={S0}->S={S} E={E} L_edge={S * E}, dense masks, 4x1000 DDPM steps",
                       "note": "the reference's CPU PyTorch path on the host cores: batch 1, one forward + scheduler step per "
                               "stage per bench step, extrapolated (one ABC B-rep is ~1 h of CPU); its own sample.py needs "
                               "diffusers/OCC/CUDA, absent offline"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": used, "sample": desc, "port": port},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def run_surfpos(args):
    """BASELINE configs[1]: SurfPosNet 1000-step DDPM, 30 face-bbox tokens, batch 64, one GPU.  1 920 tokens per forward: the
    GPU needs ~0.3 ms per step, ~105 launches from Python need more -- the loop is captured in a CUDA graph
    (sampler.Cascade._loop_graph) and replayed.  Prints one JSON line (not the headline metric: first stage only)."""
    from brepgen_b200 import _ffi
    from brepgen_b200.models import NETS
    from brepgen_b200.sampler import Cascade, CascadeConfig
    from brepgen_b200.spec import denoiser_spec
    from brepgen_b200.synth import synth_state_dict
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B, S, T = (args.batch if args.batch != 256 else 64), 30, 1000
    m = NETS["surfpos"](False)
    m.load_state_dict(synth_state_dict(denoiser_spec("surfpos", False), seed=1))
    casc = Cascade({"surfpos": m.to(dev).eval()}, device=dev)
    x = torch.randn(B, S, 6, generator=torch.Generator().manual_seed(0)).to(dev)
    fwd = lambda xi, t: casc.m["surfpos"](xi, t, None)
    casc.ddpm.set_timesteps(T)
    res = {}
    for mode in ("off", "on"):
        cfg = CascadeConfig(batch_size=B, schedule="ddpm", graph=mode)
        with torch.no_grad():
            casc._loop(cfg, casc.ddpm, casc.ddpm.timesteps[:50], x.clone(), fwd, None, None)      # warm-up
            torch.cuda.synchronize()
            l0 = _ffi.lib().bg_launch_count()
            r0 = _ffi.replayed_launches
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            casc._loop(cfg, casc.ddpm, casc.ddpm.timesteps, x.clone(), fwd, None, None)
            e1.record()
            torch.cuda.synchronize()
        res[mode] = {"ms_per_1000_steps": e0.elapsed_time(e1), "value": B / (e0.elapsed_time(e1) / 1e3),
                     "host_launch_calls": int(_ffi.lib().bg_launch_count() - l0),
                     "kernels_in_graph_replays": int(_ffi.replayed_launches - r0)}
    print(json.dumps({"metric": "B-reps/sec (SurfPosNet 1000-step DDPM stage, BASELINE configs[1])", "value": res["on"]["value"],
                      "unit": UNIT, "n_gpus": 1, "higher_is_better": True, "data": "synthetic",
                      "config": {"workload": f"surfpos B={B} S={S} T={T}", "graph": res["on"], "eager": res["off"],
                                 "graph_over_eager": res["on"]["value"] / res["off"]["value"],
                                 "note": "graph time includes warm-up step, capture and 1000 replays"}}))


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "surfpos":
        return run_surfpos(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"          # keep stdout to the single JSON line
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    from brepgen_b200 import _ffi
    from brepgen_b200.models import NETS
    from brepgen_b200.sampler import Cascade, CascadeConfig
    from brepgen_b200.spec import denoiser_spec
    from brepgen_b200.synth import synth_state_dict
    _ffi.check(_ffi.lib().bg_check_device(), "bg_check_device")

    B, S0, E, T = args.batch, args.surfaces, args.edges, args.steps_per_stage
    S = S0 if args.cf else 2 * S0
    models = {}
    for kind in KINDS:
        m = NETS[kind](args.cf)
        m.load_state_dict(synth_state_dict(denoiser_spec(kind, args.cf), seed=1))
        models[kind] = m.to(dev).eval()
    surf_vae = edge_vae = None
    try:
        from brepgen_b200.vae import build_synthetic_decoders
        surf_vae, edge_vae = build_synthetic_decoders(dev)
    except ImportError:
        pass
    for m in models.values():
        m.compact = args.compact
    casc = Cascade(models, surf_vae, edge_vae, device=dev)
    cfg = CascadeConfig(batch_size=B, num_surfaces=S0, num_edges=E, use_cf=args.cf, class_label=6, schedule=args.schedule,
                        ddpm_steps=T, dense_masks=args.masks == "dense", ragged_masks=args.masks == "ragged", seed=1000 + rank,
                        decode=surf_vae is not None)
    g = torch.Generator().manual_seed(1000 + rank)
    shapes = {"surfPos": (B, S0, 6), "surfZ": (B, S, 48), "edgePos": (B, S, E, 6), "edgeZV": (B, S, E, 18)}
    host_in = {k: torch.randn(s, generator=g).pin_memory() for k, s in shapes.items()}
    dev_in = {k: v.to(dev) for k, v in host_in.items()}

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / k
        if dist is not None:
            tms = torch.tensor([ms], device=dev)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            ms = float(tms)
        barrier()
        return ms

    last = {}

    def step_resident():
        last["out"] = casc.run(cfg, init_noise=dev_in)
    for _ in range(args.warmup):
        step_resident()
    clocks = Clocks(local)
    clocks.start()
    l0 = _ffi.lib().bg_launch_count() + _ffi.replayed_launches
    ms = timed(step_resident, args.steps)
    launches = _ffi.lib().bg_launch_count() + _ffi.replayed_launches - l0      # host launches + kernels inside graph replays
    clk = clocks.finish()
    if args.dump_outputs and rank == 0:
        dump_outputs(last["out"], args.dump_outputs)
    scale = 1000.0 / T if args.schedule == "ddpm" else 1.0     # the shipped hybrid is run literally
    # the two VAE decodes run once per cascade whatever T is: time them alone and keep them out of the 1000/T scaling
    ms_dec = 0.0
    if surf_vae is not None:
        zs = torch.randn(B * S, 3, 4, 4, device=dev)
        ze = torch.randn(B * S * E, 3, 4, device=dev)
        dec = lambda: (surf_vae(zs), edge_vae(ze))
        dec()
        ms_dec = timed(dec, max(1, args.steps))
        del zs, ze
    norm_ms = lambda m: (m - ms_dec) * scale + ms_dec          # ms per batch at 1000 steps per stage
    value = world * B / (norm_ms(ms) / 1e3)

    # end to end through the public API: pinned host noise in, every output back to pinned host memory, per step
    e2e = None
    if not args.no_e2e:
        host_out = {}
        gather_ms = []
        from brepgen_b200.sampler import gather_outputs

        def step_e2e():
            din = {k: v.to(dev, non_blocking=True) for k, v in host_in.items()}
            out = casc.run(cfg, init_noise=din)
            if dist is not None:
                # BASELINE configs[3]: the final all_gather of every output over NCCL (NVLink / NVSwitch), inside the timed
                # region; its own duration is recorded with CUDA events on the same stream
                g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g0.record()
                gathered = gather_outputs(out)
                g1.record()
                gather_ms.append((g0, g1))
                del gathered
            for k, v in out.items():
                if k not in host_out:
                    host_out[k] = torch.empty(v.shape, dtype=v.dtype).pin_memory()
                host_out[k].copy_(v, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        step_e2e()
        gather_ms.clear()
        ms_e = timed(step_e2e, args.steps)
        ms_g = sum(a.elapsed_time(b) for a, b in gather_ms) / max(len(gather_ms), 1) if gather_ms else 0.0
        h2d = sum(v.numel() * v.element_size() for v in host_in.values())
        d2h = sum(v.numel() * v.element_size() for v in host_out.values())
        # the gather, like the decodes, happens once per cascade whatever T is: kept out of the 1000 / T scaling
        norm_e = (ms_e - ms_dec - ms_g) * scale + ms_dec + ms_g
        e2e = {"value": world * B / (norm_e / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": ms_e,
               "final_all_gather_ms": ms_g if dist is not None else None,
               "all_gather_bytes_per_rank": d2h * world if dist is not None else 0}

    # roofline of the dominant kernel (edge-stage flash attention, L = S*E), timed alone with CUDA events
    burst, sustained, src = peaks()
    L = S * E
    qkv = (torch.randn(B * L, 2304, device=dev, dtype=torch.float16))
    ao = torch.empty(B * L, 768, device=dev, dtype=torch.float16)
    # same call form as inside the cascade: an (all-valid) key-padding mask plus the per-forward block list / bit words
    amask = torch.zeros(B, L, dtype=torch.bool, device=dev)
    ascr = torch.zeros(B * (5 * ((L + 127) // 128) + 1), dtype=torch.int32, device=dev)
    attn = lambda: _ffi.check(_ffi.lib().bg_op_attention(qkv.data_ptr(), ao.data_ptr(), B, L, amask.data_ptr(), 1,
                                                          ascr.data_ptr(), _ffi.current_stream()))
    for _ in range(2):
        attn()
    ms_attn = timed(attn, 5)
    fl_attn = B * 3072.0 * L * L
    ach = fl_attn / (ms_attn / 1e3) / 1e12
    del qkv, ao
    traffic = None   # dram__bytes_read.sum + dram__bytes_write.sum of this kernel at this shape (ncu --set full capture)
    tp = os.path.join(ROOT, "profiles", "attn_traffic.json")
    if os.path.exists(tp):
        tj = json.load(open(tp))
        if tj.get("B") == B and tj.get("L") == L:
            traffic = tj["dram_bytes_per_launch"]
    roofline = {"bound": "tensor", "kernel": "attn_kernel<2> (tcgen05 flash attention, B=%d L=%d)" % (B, L),
                "achieved": ach, "peak": burst, "unit": "TFLOP/s", "frac": ach / burst, "peak_source": f"bf16_tflops burst, {src}",
                "traffic": traffic, "ms_per_launch": ms_attn, "flop_per_launch": fl_attn}
    # CFG doubles every forward; the shipped hybrid runs 158 PNDM + 250 DDPM forwards per stage (sample.py:128-155)
    flops_brep = cascade_flops_per_brep(S0, S, E, steps=1000 if args.schedule == "ddpm" else 408) * (2 if args.cf else 1)
    whole = {"algorithmic_tflop_per_brep": flops_brep / 1e12, "achieved_tflops_per_gpu": value / world * flops_brep / 1e12,
             "frac_of_sustained_peak": value / world * flops_brep / 1e12 / sustained,
             "flops": "dense-algorithmic (SURVEY.md 8d): every face / edge slot counted, masks or not"}
    if args.masks != "dense" and "out" in last:
        o = last["out"]
        fv = cascade_flops_valid_tokens(S0, S, E, o["surfMask"].cpu(), o["edgeM"].cpu(),
                                        steps=1000 if args.schedule == "ddpm" else 408) * (2 if args.cf else 1)
        whole["valid_token_tflop_per_brep"] = fv / 1e12
        whole["valid_token_achieved_tflops_per_gpu"] = value / world * fv / 1e12
        whole["valid_token_frac_of_sustained_peak"] = value / world * fv / 1e12 / sustained
        whole["valid_fraction_of_edge_tokens"] = float((~o["edgeM"]).float().mean())

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, cores, desc, used = cpu_reference_sample(S0, S, E, 3, best_cpu_threads())      # ~10-20 s of CPU work
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": used, "sample": desc}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f16 x f16 -> f32 (tcgen05 kind::f16; split hi+lo weights on in/out-proj; fp32 residual/LN/softmax)",
                "data": "synthetic",
                "config": {"workload": f"{'furniture_cfg' if args.cf else 'abc'}_cascade B={B}/GPU S0={S0}->S={S} E={E} L_edge={L}, "
                                       f"{args.masks} masks, schedule={args.schedule}",
                           "ddpm_steps_per_stage_timed": T, "value_normalised_to_steps_per_stage": 1000,
                           "vae_decode_in_step": surf_vae is not None, "vae_decode_ms_per_step": ms_dec,
                           "l2": "activations of one step (GBs) exceed the 126 MB L2; no explicit flush",
                           "precision": models["surfpos"].precision, "token_compaction": bool(args.compact), "parallelism": f"batch-sharded x{world}, no collective"},
                "roofline": roofline, "whole_cascade": whole, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches),
                "clocks": clk}
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
