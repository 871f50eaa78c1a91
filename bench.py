#!/usr/bin/env python
"""Headline benchmark: grid-points/s, forward+backward, Darcy 141^2 Galerkin-transformer (BASELINE C3).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload ("darcy141_galerkin10_sc2d_b8"): FourierTransformer2D with the reference's ex2_darcy
configuration (config.yml:41-80) at the reference's own profiling protocol
(examples/ex2_memory_profile.py:58-71): fine grid 141x141, attention on the 43x43 coarse grid,
d_model 128, 4 heads, 10 Galerkin encoder layers, 2 SpectralConv2d (32 ch, 12 modes), batch 8
per GPU, fp32, synthetic N(0,1) inputs, loss ((preds-target)^2).mean(), model in training mode
with the config's dropouts and the reference's always-on attention dropout ('reference' mode).
A step = one forward + backward over one batch (+ one flat-bucket gradient all-reduce when N>1).

Lines printed (rank 0): one JSON object, see the keys in `main`.
  value  : device-timed (CUDA events per step, L2 flushed between steps), inputs resident in HBM
  e2e    : same metric through the public module API with pinned HOST inputs; H2D copies of the
           step's inputs and the D2H read of the loss are inside the timed region
  roofline / kernels : per-launch CUDA-event attribution pass run right after the timed region
  parts  : the 10-layer encoder stack and the spectral decoder timed alone, same protocol (SURVEY.md 8d)
  cpu_baseline : the oracle (CPU restatement of the reference) timed on this box's host cores
--impl reference : the oracle on CPU only, same metric/config (the reference is pure PyTorch and
  cannot travel to the GPU box; the oracle is pinned to it by tests/golden).
--dump-outputs DIR : after the timed steps, what the last timed step handed its caller -- the loss and the gradient of
  every parameter -- as DIR/loss.npy and DIR/grad.<parameter name>.npy (float32, rank 0).  Inputs, weights and dropout
  streams are seeded, so two builds run with the same arguments can be compared array for array.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

if "--impl" in sys.argv and "reference" in sys.argv:
    # torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm is meant to use the host cores it calibrates to
    os.environ.pop("OMP_NUM_THREADS", None)
    os.environ.pop("MKL_NUM_THREADS", None)

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_FINE, N_COARSE, BATCH = 141, 43, 8
POINTS_PER_SAMPLE = N_FINE * N_FINE
WORKLOAD = "darcy141_galerkin10_sc2d_b8"
METRIC = "grid-points/sec fwd+bwd, Darcy 141^2 Galerkin encoder"


_T0 = time.time()


def log(msg):
    """progress on stderr (stdout carries exactly one JSON line)"""
    print(f"[bench +{time.time() - _T0:6.1f}s] {msg}", file=sys.stderr, flush=True)


def c3_config(dropout_free=False):
    """ex2_darcy section of the reference's config.yml with the BASELINE overrides
    (10 encoder layers; scaler sizes from get_scaler_sizes(141, 43); ex2_darcy.py:67-82)."""
    from galerkin_transformer_b200.utils import scaler_sizes
    down, up = scaler_sizes(N_FINE, N_COARSE)
    cfg = dict(node_feats=1, pos_dim=2, n_targets=1, n_hidden=128, num_feat_layers=0,
               num_encoder_layers=10, n_head=4, dim_feedforward=256, feat_extract_type=None,
               attention_type="galerkin", xavier_init=0.01, diagonal_weight=0.01, symmetric_init=False,
               layer_norm=False, attn_norm=True, norm_eps=1e-7, batch_norm=False,
               return_attn_weight=False, return_latent=False, decoder_type="ifft2", spacial_dim=2,
               spacial_fc=True, upsample_mode="interp", downsample_mode="interp", freq_dim=32,
               boundary_condition="dirichlet", num_regressor_layers=2, fourier_modes=12,
               regressor_activation="silu", downscaler_activation="relu", upscaler_activation="silu",
               last_activation=True, dropout=0.0, downscaler_dropout=0.05, upscaler_dropout=0.0,
               ffn_dropout=0.05, encoder_dropout=0.05, decoder_dropout=0.0, debug=False,
               downscaler_size=down, upscaler_size=up)
    if dropout_free:
        for k in ("dropout", "downscaler_dropout", "upscaler_dropout", "ffn_dropout", "encoder_dropout",
                  "decoder_dropout"):
            cfg[k] = 0.0
    return cfg


def c3_inputs(bsz, device, seed=1127802, pin=False):
    """node, pos, grid, target as the reference's datasets shape them (ft.py:643-651)."""
    g = torch.Generator().manual_seed(seed)
    node = torch.randn(bsz, N_FINE, N_FINE, 1, generator=g)
    target = torch.randn(bsz, N_FINE, N_FINE, 1, generator=g)
    gc = torch.linspace(0, 1, N_COARSE)
    pos = torch.stack(torch.meshgrid(gc, gc, indexing="ij"), -1).reshape(1, -1, 2).repeat(bsz, 1, 1)
    gf = torch.linspace(0, 1, N_FINE)
    grid = torch.stack(torch.meshgrid(gf, gf, indexing="ij"), -1)[None].repeat(bsz, 1, 1, 1)
    out = [node, pos.contiguous(), grid.contiguous(), target]
    if pin:
        return [t.pin_memory() for t in out]
    return [t.to(device) for t in out]


# ----------------------------------------------------------------------------------------------
# BASELINE.json configs 2-5 as bench workloads (C1 is the reference's own CPU case; it is a parity test)
# ----------------------------------------------------------------------------------------------
def _mesh2(n, bsz):
    g = torch.linspace(0, 1, n)
    return torch.stack(torch.meshgrid(g, g, indexing="ij"), -1)[None].repeat(bsz, 1, 1, 1)


class Workload:
    """name, model class name, config, per-GPU batch, grid points per sample, inputs(bsz, seed) -> list of CPU tensors
    (last one = target), forward(model, *inputs[:-1]) -> prediction, oracle(sd, cfg, *inputs[:-1]) -> prediction"""

    def __init__(self, key):
        self.key = key
        getattr(self, "_" + key)()

    # C3: Darcy 141^2, 43^2 attention grid, 10 Galerkin layers + 2 SpectralConv2d  (the headline)
    def _c3(self):
        self.name, self.model_cls, self.cfg, self.batch, self.points = WORKLOAD, "FourierTransformer2D", c3_config(), BATCH, POINTS_PER_SAMPLE
        self.desc = dict(grid="141x141 fine / 43x43 attention", encoder_layers=10, d_model=128, heads=4,
                         decoder="2x SpectralConv2d(32, modes 12)")
        self.inputs = lambda bsz, seed=1127802: c3_inputs(bsz, "cpu", seed=seed)
        self.forward = lambda m, node, pos, grid: m(node, None, pos, grid)["preds"]
        self.oracle = lambda O, sd, cfg, node, pos, grid, **kw: O.fourier_transformer_2d(sd, cfg, node, pos, grid, **kw)

    # C2: 1-D Burgers n = 8192, Galerkin encoder 6 layers d_model 96 (config.yml ex1_burgers: 1 head, d_ff 192), batch 8
    def _c2(self):
        cfg = dict(node_feats=1, edge_feats=None, pos_dim=1, n_targets=1, n_hidden=96, num_feat_layers=0, num_encoder_layers=6,
                   n_head=1, pred_len=0, n_freq_targets=0, dim_feedforward=192, feat_extract_type=None,
                   attention_type="galerkin", xavier_init=0.001, diagonal_weight=0.01, symmetric_init=False, layer_norm=False,
                   attn_norm=True, batch_norm=False, spacial_residual=False, return_attn_weight=False, return_latent=False,
                   residual_type="plus", seq_len=None, bulk_regression=False, decoder_type="ifft", freq_dim=48,
                   num_regressor_layers=2, fourier_modes=16, spacial_dim=1, spacial_fc=False, dropout=0.0, encoder_dropout=0.0,
                   ffn_dropout=0.0, decoder_dropout=0.0, debug=False)
        self.name, self.model_cls, self.cfg, self.batch, self.points = "burgers8192_galerkin6_sc1d_b8", "SimpleTransformer", cfg, 8, 8192
        self.desc = dict(grid="n = 8192 (1-D)", encoder_layers=6, d_model=96, heads=1, decoder="2x SpectralConv1d(48, modes 16)")

        def inputs(bsz, seed=1127802):
            g = torch.Generator().manual_seed(seed)
            node = torch.randn(bsz, 8192, 1, generator=g)
            target = torch.randn(bsz, 8192, 1, generator=g)
            pos = torch.linspace(0, 1, 8192)[None, :, None].repeat(bsz, 1, 1)
            return [node, pos.contiguous(), target]
        self.inputs = inputs
        self.forward = lambda m, node, pos: m(node, None, pos)["preds"]
        self.oracle = lambda O, sd, cfg, node, pos, **kw: O.simple_transformer(sd, cfg, node, pos, **kw)

    # C4: Darcy inverse 211^2 with 10 % noise, Fourier-type (Q K^T) V attention on the 71^2 grid, pointwise decoder
    def _c4(self):
        from galerkin_transformer_b200.utils import scaler_sizes
        down, _ = scaler_sizes(211, 71)
        cfg = dict(node_feats=1, pos_dim=2, n_targets=1, n_hidden=192, num_feat_layers=0, num_encoder_layers=6, n_head=4,
                   dim_feedforward=384, feat_extract_type=None, attention_type="fourier", xavier_init=0.01, diagonal_weight=0.01,
                   symmetric_init=False, layer_norm=False, attn_norm=True, norm_eps=1e-7, batch_norm=False,
                   return_attn_weight=False, return_latent=False, decoder_type="pointwise", regressor_activation="silu",
                   spacial_dim=2, spacial_fc=True, upsample_mode="interp", downsample_mode="interp", boundary_condition="free",
                   num_regressor_layers=1, dropout=0.05, downscaler_dropout=0.05, upscaler_dropout=0.05, ffn_dropout=0.05,
                   encoder_dropout=0.05, decoder_dropout=0.05, debug=False, downscaler_size=down,
                   upscaler_size=((71, 71), (71, 71)))
        self.name, self.model_cls, self.cfg, self.batch, self.points = "darcyinv211_fourier6_pointwise_b4", "FourierTransformer2D", cfg, 4, 211 * 211
        self.desc = dict(grid="211x211 fine (10% noise) / 71x71 attention and target", encoder_layers=6, d_model=192, heads=4,
                         decoder="PointwiseRegressor")

        def inputs(bsz, seed=1127802):
            g = torch.Generator().manual_seed(seed)
            node = torch.randn(bsz, 211, 211, 1, generator=g)
            node = node + 0.1 * torch.randn(bsz, 211, 211, 1, generator=g)
            target = torch.randn(bsz, 71, 71, 1, generator=g)
            pos = _mesh2(71, bsz).reshape(bsz, -1, 2)
            return [node, pos.contiguous(), _mesh2(71, bsz).contiguous(), target]
        self.inputs = inputs
        self.forward = lambda m, node, pos, grid: m(node, None, pos, grid)["preds"]
        self.oracle = lambda O, sd, cfg, node, pos, grid, **kw: O.fourier_transformer_2d(sd, cfg, node, pos, grid, **kw)

    # C5: Navier-Stokes 64x64, 10-step autoregressive rollout (libs/ns_lite.py:205-238), Galerkin + SpectralConv2d
    def _c5(self):
        cfg = dict(node_feats=10 + 2, pos_dim=2, n_targets=1, n_hidden=48, num_feat_layers=0, num_encoder_layers=4, n_head=1,
                   dim_feedforward=96, attention_type="galerkin", feat_extract_type=None, xavier_init=0.01, diagonal_weight=0.01,
                   layer_norm=True, attn_norm=False, return_attn_weight=False, return_latent=False, decoder_type="ifft",
                   freq_dim=20, num_regressor_layers=2, fourier_modes=12, spacial_dim=2, spacial_fc=False, dropout=0.0,
                   encoder_dropout=0.0, decoder_dropout=0.0, ffn_dropout=0.05, debug=False)
        self.name, self.model_cls, self.cfg, self.batch, self.points = "ns64x64x10_galerkin4_sc2d_b8", "FourierTransformer2DLite", cfg, 8, 64 * 64 * 10
        self.desc = dict(grid="64x64, 10-step rollout", encoder_layers=4, d_model=48, heads=1, decoder="2x SpectralConv2d(20, modes 12)")

        def inputs(bsz, seed=1127802):
            g = torch.Generator().manual_seed(seed)
            node = torch.randn(bsz, 64, 64, 10, generator=g)
            target = torch.randn(bsz, 64, 64, 10, generator=g)
            grid = _mesh2(64, bsz)
            return [node, grid.reshape(bsz, -1, 2).contiguous(), grid.contiguous(), target]
        self.inputs = inputs

        def rollout(step_fn, node, pos, grid):
            x, preds = node, []
            for _ in range(10):
                u = step_fn(x, pos, grid)
                x = torch.cat((x[..., 1:], u), dim=-1)
                preds.append(u)
            return torch.cat(preds, dim=-1)
        self.forward = lambda m, node, pos, grid: rollout(lambda x, p_, g_: m(x, None, p_, g_)["preds"], node, pos, grid)
        self.oracle = lambda O, sd, cfg, node, pos, grid, **kw: rollout(
            lambda x, p_, g_: O.fourier_transformer_2d_lite(sd, cfg, x, p_, g_, **kw), node, pos, grid)

    def build(self, device):
        import galerkin_transformer_b200 as G
        return getattr(G, self.model_cls)(**self.cfg).to(device)

    def loss(self, model, *inputs):
        return ((self.forward(model, *inputs[:-1]) - inputs[-1]) ** 2).mean()


# ----------------------------------------------------------------------------------------------
def _cpu_steps(wl, sd, data, n, attn_dropout=True):
    from oracle import galerkin_oracle as O
    times = []
    for _ in range(n):
        t0 = time.perf_counter()
        pred = wl.oracle(O, sd, wl.cfg, *data[:-1], attn_dropout=attn_dropout)
        loss = ((pred - data[-1]) ** 2).mean()
        grads = torch.autograd.grad(loss, [v for v in sd.values() if v.requires_grad], allow_unused=True)
        loss.item()
        del grads
        times.append(time.perf_counter() - t0)
    return times


def cpu_reference_run(wl, steps, warmup, bsz):
    """fwd+bwd of the oracle's restatement of the workload's model on the host cores, faithful attention dropout;
    returns (grid-points/s, seconds per step, threads).

    Thread count: eager PyTorch on a many-core host gets SLOWER past a point on these small
    operators, so the count is calibrated (one small-batch step at 8/16/32/64/all threads, best
    wins) and reported as `cores` -- "all the host threads it can use" productively."""
    ncpu = os.cpu_count() or 1
    torch.manual_seed(1127802)
    model = wl.build("cpu")                        # parameter container only (never run on CPU)
    sd = {k: v.detach().clone().requires_grad_(v.is_floating_point()) for k, v in model.state_dict().items()}
    small = wl.inputs(min(2, bsz))
    best, threads = None, ncpu
    for cand in sorted({min(c, ncpu) for c in (8, 16, 32, 64, ncpu)}):
        torch.set_num_threads(cand)
        _cpu_steps(wl, sd, small, 1)
        t = _cpu_steps(wl, sd, small, 1)[0]
        log(f"cpu calibration: {cand} threads -> {t:.3f} s per batch-{min(2, bsz)} step")
        if best is None or t < best:
            best, threads = t, cand
        elif t > 1.3 * best:          # past the knee: more threads only get slower (128 -> 100 s/step)
            break
    torch.set_num_threads(threads)
    data = wl.inputs(bsz)
    _cpu_steps(wl, sd, data, warmup)
    times = _cpu_steps(wl, sd, data, steps)
    sec = sum(times) / len(times)
    return bsz * wl.points / sec, sec, threads


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            pass

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out = ""
        sm, smax, reasons = [], [], set()
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                 f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=max(smax) if smax else None,
                    samples=len(sm), reasons=sorted(reasons))


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], bf16_tflops=p["bf16_tflops"],
                    bf16_tflops_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


def merge_gemm_layouts(summary):
    """The tcgen05 GEMM is ONE kernel template; fold its operand-layout variants (nt / nn / tn) into one row."""
    out = {}
    for fam, a in summary.items():
        key = "gemm_tc_kernel" if fam.startswith("gemm_tc_") else ("gemm_simt_kernel" if fam.startswith("gemm_simt_") else fam)
        o = out.setdefault(key, dict(launches=0, ms=0.0, flops=0.0, bytes=0.0))
        for k in o:
            o[k] += a[k]
    return out


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture of the CURRENT
    build (profiles/ncu_traffic.json is rewritten by tools/ncu_summary.py from every tools/final_profile.sh run)."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(path):
        with open(path) as f:
            table = json.load(f)
        for key, v in table.items():
            if key.split("::")[-1].replace("_kernel", "").replace("void ", "").split("<")[0] in (kernel, kernel + "_kernel"):
                return v
        stem = kernel.replace("_kernel", "")
        for key, v in table.items():
            if stem in key:
                return v
    return None


DUMP_LIMIT_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, loss, model):
    """Write the loss and every parameter gradient of the last timed step as float32 .npy files; returns the file count."""
    import numpy as np
    arrays = {"loss": loss}
    arrays.update((f"grad.{n}", p.grad) for n, p in model.named_parameters() if p.grad is not None)
    total = sum(t.numel() * 4 for t in arrays.values())
    assert total <= DUMP_LIMIT_BYTES, f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit"
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())
    return len(arrays)


def kernel_table(summary, steps, peaks):
    """Per kernel family: launches/step, ms/step, achieved GB/s and TFLOP/s on ALGORITHMIC work."""
    rows = []
    tf32_peak = peaks["bf16_tflops_sustained"] / 2.0        # dense TF32 = 1/2 dense bf16 on tcgen05
    ridge = tf32_peak * 1e12 / (peaks["hbm_gbs"] * 1e9)
    for fam, a in summary.items():
        ms = a["ms"] / steps
        if ms <= 0:
            continue
        gbs = a["bytes"] / steps / (ms * 1e-3) / 1e9
        tfs = a["flops"] / steps / (ms * 1e-3) / 1e12
        ai = a["flops"] / max(a["bytes"], 1.0)
        bound = "tensor" if ai > ridge else "hbm"
        frac = tfs / tf32_peak if bound == "tensor" else gbs / peaks["hbm_gbs"]
        rows.append(dict(kernel=fam, launches_per_step=a["launches"] / steps, ms_per_step=round(ms, 4),
                         alg_gbs=round(gbs, 1), alg_tflops=round(tfs, 3), bound=bound, frac=round(frac, 4),
                         ms_per_launch=round(a["ms"] / a["launches"], 5),
                         alg_bytes_per_launch=a["bytes"] / a["launches"],
                         alg_flops_per_launch=a["flops"] / a["launches"]))
    rows.sort(key=lambda r: -r["ms_per_step"])
    return rows, tf32_peak


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c3", choices=["c2", "c3", "c4", "c5"],
                    help="BASELINE.json config: c3 (default, the headline metric), c2 Burgers, c4 Darcy inverse / Fourier, c5 NS rollout")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: the config's batch per GPU; strong: the config's batch is the GLOBAL batch, split over the GPUs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--attn-dropout", default="reference", choices=["reference", "off"])
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of CUDA-graph replay")
    ap.add_argument("--no-parts", action="store_true", help="skip the encoder-only / decoder-only timings")
    ap.add_argument("--batch-streams", type=int, default=int(os.environ.get("GB200_BATCH_STREAMS", "1")),
                    help="split the per-GPU batch into this many concurrent micro-batch chains inside the graph")
    ap.add_argument("--precision", default="x3", choices=["x3", "tf32", "fp32"],
                    help="x3 (default): bf16x3 fused encoder / conv kernels + TF32 weight gradients + exact fp32 elsewhere; "
                         "tf32: every GEMM single-pass TF32; fp32: exact SIMT")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's loss and parameter gradients to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the b200 implementation only")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    wl = Workload(args.config)
    if args.scaling == "strong":
        assert wl.batch % world == 0, f"strong scaling: global batch {wl.batch} must divide over {world} GPUs"
        bsz = wl.batch // world
    else:
        bsz = wl.batch
    metric = METRIC if args.config == "c3" else f"grid-points/sec fwd+bwd, {wl.name}"
    config = dict(workload=wl.name, baseline_config=args.config.upper(), **wl.desc, batch_per_gpu=bsz, global_batch=bsz * world,
                  parallelism=f"dp{world}",
                  dropout="the reference config's dropouts; attention p=0.5 " + args.attn_dropout,
                  l2="256 MiB buffer written between timed steps (L2 flush)",
                  launch="eager" if args.no_graph else "whole fwd+bwd step replayed from one CUDA graph",
                  gemm_precision=args.precision, micro_batch_chains=args.batch_streams,
                  backward_streams="dW / db launches on side streams (parallel graph branches)"
                  if os.environ.get("GB200_BWD_STREAMS", "1") != "0" else "off")

    if args.impl == "reference":
        if rank != 0:
            return
        cbsz = wl.batch      # always the stated config (the driver runs 20 + 5 steps: ~12 s of CPU work at C3 batch 8)
        val, sec, threads = cpu_reference_run(wl, args.steps, args.warmup, cbsz)
        config["batch_per_gpu"], config["global_batch"], config["parallelism"] = cbsz, cbsz, "cpu"
        sample = f"{args.steps} fwd+bwd steps of {wl.name} on a batch of {cbsz} (CPU oracle, fp32, faithful attention dropout)"
        print(json.dumps(dict(
            impl="reference", metric=metric, value=val, unit="grid-points/s", n_gpus=args.gpus, steps=args.steps,
            warmup=args.warmup, ms_per_step=sec * 1e3, higher_is_better=True, scaling=args.scaling, vs_baseline=None,
            dtype="f32", data="synthetic", config=config,
            cpu_baseline=dict(value=val, unit="grid-points/s", cores=threads, kind="port", sample=sample),
            e2e=dict(value=val, unit="grid-points/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))))
        return

    import torch.distributed as dist
    import galerkin_transformer_b200 as G
    from galerkin_transformer_b200 import _lib, functional as GF
    from galerkin_transformer_b200.parallel import FlatGradBucket

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"        # keep NCCL's version banner off stdout (one JSON line only)
        dist.init_process_group("nccl", device_id=dev)
    G.set_precision(args.precision)
    torch.manual_seed(1127802)                      # identical replicas
    model = wl.build(dev)
    model.train()
    G.set_attn_dropout(model, args.attn_dropout)
    torch.manual_seed(1127802 + rank)               # per-rank dropout streams / data
    bucket = FlatGradBucket(model)
    data = [t.to(dev) for t in wl.inputs(bsz, seed=1127802 + rank)]
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)

    from galerkin_transformer_b200.graphs import GraphedStep

    def loss_fn(*inp):
        return wl.loss(model, *inp)

    graphed, launches_per_step = None, None
    if not args.no_graph:
        c0 = _lib.launch_count()
        # the flat gradient bucket is filled INSIDE the captured graph (one multi-tensor copy as the graph's last node)
        graphed = GraphedStep(loss_fn, data, model.parameters(), warmup=3, batch_streams=args.batch_streams,
                              post_backward=(lambda grads: bucket.pack(grads)) if world > 1 else None)
        # 3 eager warm-ups + 1 capture pass, all with identical launch sequences
        launches_per_step = (_lib.launch_count() - c0) // 4
        log(f"captured CUDA graph: {launches_per_step} libgalerkin_b200 kernels per step")

    def step(*inp):
        if graphed is not None:
            graphed.load_inputs(*inp)
            loss = graphed.replay()
            bucket.all_reduce_packed()          # enqueued right behind the replay: only the collective itself is exposed
            return loss
        bucket.zero()
        GF.advance_rng()
        loss = loss_fn(*inp)
        loss.backward()
        bucket.all_reduce()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # device-resident inputs: the graph's own static buffers (no staging copy inside the timed step)
    resident = graphed.static_inputs if graphed is not None else data
    log("model built; warm-up")
    for _ in range(max(args.warmup, 3)):
        step(*resident)
    barrier()
    log("timed region")

    # ---- timed region: K steps, device-timed per step, L2 flushed in between -----------------
    sampler = ClockSampler(local_rank) if rank == 0 else None
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    launches0 = _lib.launch_count()
    barrier()
    wall0 = time.perf_counter()
    for i in range(args.steps):
        flush.fill_(float(i))
        starts[i].record()
        last_loss = step(*resident)
        ends[i].record()
    barrier()
    wall = time.perf_counter() - wall0
    gpu_launches = _lib.launch_count() - launches0
    if graphed is not None:          # replays issue no host-side launches: kernels per graph x replays
        gpu_launches = launches_per_step * args.steps
    clocks = sampler.stop() if sampler else None
    dev_ms = sum(s.elapsed_time(e) for s, e in zip(starts, ends))
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = t.item()
    ms_per_step = total_ms / args.steps
    value = bsz * world * wl.points / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:       # before the passes below overwrite the gradients
        n = dump_outputs(args.dump_outputs, last_loss, model)
        log(f"wrote {n} arrays of the last timed step to {args.dump_outputs}")

    log(f"device-timed: {ms_per_step:.3f} ms/step; end-to-end pass")
    # ---- end to end: pinned host inputs -> H2D -> fwd+bwd -> D2H loss, every step ------------
    host = [t_.pin_memory() for t_ in wl.inputs(bsz, seed=1127802 + rank)]
    h2d = sum(t_.numel() * t_.element_size() for t_ in host)
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()
    e2e_steps = args.steps

    def to_device(hs):
        # graph path: pinned host -> the graph's static device buffers directly (inside step());
        # eager path: pinned host -> fresh device tensors
        return hs if graphed is not None else [h.to(dev, non_blocking=True) for h in hs]

    for _ in range(2):
        loss_host.copy_(step(*to_device(host)).detach(), non_blocking=True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(e2e_steps):
        loss_host.copy_(step(*to_device(host)).detach(), non_blocking=True)
        torch.cuda.current_stream().synchronize()        # the user reads the loss every step (utils_ft.py:687)
        float(loss_host)
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = bsz * world * wl.points / (t.item() / e2e_steps * 1e-3)

    # ---- exposed communication: the same replay loop with the collective switched off (N > 1 only) ----
    comm_ms = None
    if world > 1 and graphed is not None:
        barrier()
        c0_, c1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0_.record()
        for i in range(args.steps):
            flush.fill_(float(i))
            graphed.replay()
        c1_.record()
        barrier()
        c2_, c3_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c2_.record()
        for i in range(args.steps):
            flush.fill_(float(i))
            graphed.replay()
            bucket.all_reduce_packed()
        c3_.record()
        barrier()
        tt = torch.tensor([c0_.elapsed_time(c1_), c2_.elapsed_time(c3_)], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        comm_ms = (tt[1].item() - tt[0].item()) / args.steps

    # ---- attribution pass: per-launch CUDA events on the launching stream --------------------
    kernels, roofline = [], None
    log("attribution pass")
    if rank == 0:
        peaks = measured_peaks()
        prof_steps = min(args.steps, 5)
        GF.Profiler.reset()
        streams_on = GF._BWD_STREAMS
        GF.set_backward_streams(False)      # serial launches: each event pair then brackets exactly one kernel
        for _ in range(prof_steps):
            # Eager launches, but queued behind a ~30 ms spin kernel so the GPU never waits for the host:
            # the per-launch events then bracket kernel execution, not Python launch latency.
            torch.cuda._sleep(int(30e-3 * 1.9e9))
            GF.Profiler.enabled = True
            for p_ in model.parameters():
                p_.grad = None
            GF.advance_rng()
            loss_fn(*data).backward()
            GF.Profiler.enabled = False
            torch.cuda.synchronize()
        GF.set_backward_streams(streams_on)
        if graphed is not None:
            for p_, g_ in zip(graphed.params, graphed.static_grads):
                p_.grad = g_
        kernels, tf32_peak = kernel_table(merge_gemm_layouts(GF.Profiler.summary()), prof_steps, peaks)
        native_ms = sum(k["ms_per_step"] for k in kernels)
        top = kernels[0]
        traffic = ncu_traffic(top["kernel"])
        roofline = dict(kernel=top["kernel"], bound=top["bound"],
                        achieved=top["alg_tflops"] if top["bound"] == "tensor" else top["alg_gbs"],
                        peak=tf32_peak if top["bound"] == "tensor" else peaks["hbm_gbs"],
                        unit="TFLOP/s" if top["bound"] == "tensor" else "GB/s", frac=top["frac"],
                        traffic=(traffic or {}).get("dram_bytes_per_launch"), traffic_note=(traffic or {}).get("note"),
                        alg_bytes_per_launch=top["alg_bytes_per_launch"], alg_flops_per_launch=top["alg_flops_per_launch"],
                        alg_tflops=top["alg_tflops"], tensor_frac_of_dense_tf32=round(top["alg_tflops"] / tf32_peak, 4),
                        share_of_step=round(top["ms_per_step"] / ms_per_step, 4),
                        share_note="serial per-launch time / timed step; in the timed step the weight-gradient launches "
                                   "run on side streams concurrently, so shares can sum past 1",
                        peak_source=f"MEASURED_PEAKS.json ({peaks['source']}); tensor peak = sustained bf16 / 2 "
                                    "(dense TF32; the bf16x3 kernels issue 3 bf16 products per logical product, so their "
                                    "tensor-pipe time is 1.5x this scale)",
                        timing=f"CUDA events around every launch on the launching stream, {prof_steps}-step eager "
                               "attribution pass after the timed region, launches pre-queued behind a spin kernel "
                               "so events bracket execution, not host launch latency",
                        native_ms_per_step=round(native_ms, 3))
    # ---- SURVEY 8(d): the encoder stack and the decoder timed on their own (same protocol: graph replay, L2 flush) ----
    parts = None
    if rank == 0 and graphed is not None and not args.no_parts and args.config == "c3":
        log("parts: encoder stack / decoder alone")
        node, pos, grid, target = data

        def time_part(fn, inputs, params):
            g = GraphedStep(fn, inputs, params, warmup=3)
            for _ in range(3):
                g.replay()
            ss = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
            ee = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
            for i in range(args.steps):
                flush.fill_(float(i))
                ss[i].record()
                g.replay()
                ee[i].record()
            torch.cuda.synchronize()
            return sum(s.elapsed_time(e) for s, e in zip(ss, ee)) / args.steps

        def enc_fn(x_, p_):
            from galerkin_transformer_b200.model import prepack_encoder_layers
            side = prepack_encoder_layers(model.encoder_layers, x_, p_)
            if side is not None:
                torch.cuda.current_stream().wait_stream(side)
            for layer in model.encoder_layers:
                x_ = layer(x_, p_)
            return x_.square().mean()

        def dec_fn(x_, g_):
            y_ = model.regressor(x_, grid=g_)
            return (y_[0] if isinstance(y_, tuple) else y_).square().mean()

        gen = torch.Generator(device=dev).manual_seed(7)
        xe = torch.randn(bsz, pos.shape[1], 128, device=dev, generator=gen)
        xd = torch.randn(bsz, grid.shape[1], grid.shape[2], 128, device=dev, generator=gen)
        enc_ms = time_part(enc_fn, [xe, pos], list(model.encoder_layers.parameters()))
        dec_ms = time_part(dec_fn, [xd, grid], list(model.regressor.parameters()))
        T = bsz * pos.shape[1]
        parts = dict(encoder_stack=dict(ms_per_step=round(enc_ms, 4), input=f"x ({bsz},{pos.shape[1]},128), 10 layers, "
                                        "fwd+bwd w.r.t. parameters (encoder_memory_profile.py protocol)",
                                        tokens_per_s=round(T / (enc_ms * 1e-3)),
                                        alg_gflop=125.0 * bsz / 8, alg_tflops=round(125.0 * bsz / 8 / enc_ms, 2)),
                     decoder=dict(ms_per_step=round(dec_ms, 4), input=f"x ({bsz},{grid.shape[1]},{grid.shape[2]},128): "
                                  "fc(cat[x,grid]) -> 2x SpectralConv2d(32, 12 modes) -> 32-128-1 head, fwd+bwd w.r.t. "
                                  "parameters", grid_points_per_s=round(bsz * POINTS_PER_SAMPLE / (dec_ms * 1e-3))),
                     note="full model = downscaler + encoder stack + upscaler + decoder (+ loss); SURVEY.md 8(d)")
    if world > 1:
        dist.barrier()

    if rank == 0:
        out = dict(metric=metric, value=value, unit="grid-points/s", n_gpus=world, steps=args.steps,
                   warmup=max(args.warmup, 3), ms_per_step=ms_per_step, higher_is_better=True, scaling=args.scaling,
                   vs_baseline=None, dtype="f32", data="synthetic", config=config, clocks=clocks,
                   e2e=dict(value=e2e_value, unit="grid-points/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=4),
                   gpu_launches=int(gpu_launches), wall_s_timed_region=round(wall, 3),
                   grad_bucket_bytes=bucket.nbytes, roofline=roofline, kernels=kernels[:14])
        if comm_ms is not None:
            out["exposed_comm_ms_per_step"] = round(comm_ms, 4)
        if parts is not None:
            out["parts"] = parts
        if world == 1 and not args.no_cpu_baseline:
            log("cpu baseline (oracle on host cores)")
            cval, csec, threads = cpu_reference_run(wl, 3, 1, wl.batch)
            out["cpu_baseline"] = dict(value=cval, unit="grid-points/s", cores=threads, kind="port",
                                       sample=f"3 fwd+bwd steps (after 1 warm-up) of {wl.name} at batch {wl.batch}, "
                                              "CPU oracle, fp32, faithful attention dropout",
                                       ms_per_step=csec * 1e3)
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
