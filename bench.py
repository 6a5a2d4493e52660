#!/usr/bin/env python
"""Benchmark of the per-knee hot path (BASELINE.json metric: knee volumes/s for seg + ICON reg + warps; conv TFLOP/s;
warp HBM GB/s).

    python bench.py --gpus 1 --steps 5 --warmup 3                       # BASELINE configs[2], this repo's CUDA path
    python bench.py --config seg|reg|warp-sweep|batch64 ...             # BASELINE configs[0], [1], [4], [3]
    python bench.py --impl reference --gpus 1 --steps 2 --warmup 1      # the reference's CPU path (oracle port)
    torchrun ... bench.py --gpus N ...                                  # N ranks, knees sharded by volume, no collective
    python bench.py --steps 5 --warmup 3 --dump-outputs DIR             # --config full only: also write the last
                                                                        # timed step's outputs to DIR/<name>.npy

--config full (default): one "step" = one synthetic 160x384x384 knee through 3-D UNet segmentation (160 overlapping
32x128x128 tiles), GradICON registration to the atlas (both directions), warp of the FC/TC probability maps onto the
atlas grid and warp of 85 370 thickness-mesh vertices into atlas space.  Every config prints ONE JSON line carrying
`roofline` (dominant kernel, measured live with CUDA events) and, at N = 1, `cpu_baseline`.

Baselines beside the number (never the thing shipped): `cpu_baseline` times oracle/ (the CPU restatement of the
reference path) on the host cores; `library_bar` times the reference's own torch-CUDA path -- the same torch ops the
reference issues (cuDNN convolutions with TF32 as torch defaults, F.grid_sample) -- on this GPU.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PATCH, OVERLAP = [128, 128, 32], (16, 16, 8)
SEG_FLOP_PER_VOLUME = 156.31e12      # SURVEY §8(d): 160 tiles x 976.94 GFLOP (every MAC the reference executes)
REG_BYTES_PER_PAIR = 2.6e9           # SURVEY §8(d) config 2: ideal fp32 traffic of 8 UNet forwards + compositions + warps
METRIC = "knee volumes/sec (seg+ICON reg+warp)"
WORKLOADS = {
    "full": "BASELINE configs[2]: full per-knee path on one B200 (3-D UNet segmentation of a 160x384x384 knee in 160 "
            "tiles of 32x128x128 + GradICON registration 80x192x192 both directions + FC/TC warp to the atlas grid + "
            "85370-vertex warp); one knee per step per GPU, knees sharded by volume",
    "seg": "BASELINE configs[0]: single synthetic 160x384x384 DESS knee, 3-D UNet cartilage segmentation, random-init "
           "weights; one knee per step per GPU",
    "reg": "BASELINE configs[1]: ICON/GradICON knee-to-atlas registration of one 80x192x192 pair (both directions) incl. "
           "field composition and image warp; one pair per step per GPU",
    "batch64": "BASELINE configs[3]: batch of 64 synthetic knees sharded by volume across the ranks (strong scaling); "
               "one step = the whole batch through the streamed host API",
    "warp-sweep": "BASELINE configs[4]: trilinear warp / composition micro-benchmark sweep 64^3-384^3, 1-8 channels; "
                  "one step = one pass over all cases",
}


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(tflops=float(p["bf16_tflops_sustained"]), tflops_burst=float(p["bf16_tflops"]),
                    hbm=float(p["hbm_gbs"]), source="measured (MEASURED_PEAKS.json)")
    except Exception:  # noqa: BLE001
        return dict(tflops=1400.0, tflops_burst=1650.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.path = tempfile.mktemp(suffix=".clocks.csv")
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=open(self.path, "w"),
                                         stderr=subprocess.DEVNULL)
        except Exception:  # noqa: BLE001
            self.proc = None

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, reasons = [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                c = [v.strip() for v in line.split(",")]
                if len(c) < 8:
                    continue
                sm.append(float(c[1]))
                out["sm_max_mhz"] = float(c[2])
                for n, v in zip(names, c[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            os.unlink(self.path)
        except Exception:  # noqa: BLE001
            pass
        if sm:
            busy = [v for v in sm if v > 0.5 * max(sm)]
            out["sm_mhz"] = float(np.median(busy))
            out["samples"] = len(sm)
        out["reasons"] = sorted(reasons)
        return out


# ----------------------------------------------------------------------------------------------- building blocks
def write_seg_config_file(tmp):
    cfg_json = os.path.join(tmp, "segmentation_train_config.pth.tar")
    with open(cfg_json, "w") as f:
        json.dump({"patch_size": PATCH, "model": "UNet",
                   "model_setting": {"in_channels": 1, "n_classes": 2, "bias": True, "BN": True}}, f)
    return cfg_json


def build_segmenter(device, tiles_per_batch=None):
    import torch

    from oai_analysis_2_b200.segmentation.segmenter import Segmenter3DInPatchClassWise
    tmp = tempfile.mkdtemp(prefix="oai_bench_")
    # ckpoint_path=None -> the reference's own random init (segmentation/utils.py:42-44 -> UNet.weights_init)
    seg_cfg = dict(ckpoint_path=None, training_config_file=write_seg_config_file(tmp), device=str(device), batch_size=4,
                   overlap_size=OVERLAP, output_prob=True, output_itk=True, tiles_per_batch=tiles_per_batch)
    torch.manual_seed(1234)
    seg = Segmenter3DInPatchClassWise(mode="pred", config=seg_cfg)
    seg.pred_setup()
    return seg


def build_reg_model():
    import torch

    from oai_analysis_2_b200.icon_registration import pretrained_models
    torch.manual_seed(4321)
    reg = pretrained_models.OAI_knees_gradICON_model(pretrained=False)
    for net in reg.nets.values():  # icon zero-initialises lastConv (zero displacement); give the warps real work
        net._sd["lastConv.weight"].normal_(0, 0.02)
        net._sd["lastConv.bias"].normal_(0, 0.05)
        net._packed = None
    return reg


def build_pipeline(device, tiles_per_batch=None):
    from oai_analysis_2_b200 import synthetic
    from oai_analysis_2_b200.pipeline import KneePipeline
    from oai_analysis_2_b200.transforms import Geometry
    seg = build_segmenter(device, tiles_per_batch)
    reg = build_reg_model()
    geom = Geometry(synthetic.OAI_SHAPE[::-1], synthetic.OAI_SPACING)
    atlas = synthetic.synthetic_knee(synthetic.OAI_SHAPE, seed=1)
    pipe = KneePipeline(seg, reg, atlas, geom, device)
    return pipe, geom


def make_inputs(rank, n_distinct=2):
    from oai_analysis_2_b200 import synthetic
    base = synthetic.synthetic_knee(synthetic.OAI_SHAPE, seed=100 + rank)
    vols = [base]
    for i in range(1, n_distinct):  # cheap distinct variants: mirrored / rolled copies of the blob field
        vols.append(np.ascontiguousarray(np.roll(base[:, ::-1, :], 17 * i, axis=2)))
    verts = np.concatenate([synthetic.synthetic_vertices(synthetic.N_VERTS_FC, seed=rank),
                            synthetic.synthetic_vertices(synthetic.N_VERTS_TC, seed=1000 + rank)])
    return vols, verts


DUMP_BYTES_PER_ARRAY = 8 << 20   # the five outputs of --config full stay under 64 MB in all


def dump_outputs(out_dir, arrays):
    """Write each output as <out_dir>/<name>.npy in its own dtype (float32 / float64).  An array larger than
    DUMP_BYTES_PER_ARRAY is written as a sample of its flattened elements at sorted indices drawn with a fixed seed, so
    two builds run with the same arguments can be compared value for value."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        k = DUMP_BYTES_PER_ARRAY // a.itemsize
        if a.size > k:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, k, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def conv_profile_end(lib, check):
    ms, n, fl, xfl = ctypes.c_double(), ctypes.c_longlong(), ctypes.c_double(), ctypes.c_double()
    check(lib.oai_profile_end(ctypes.byref(ms), ctypes.byref(n), ctypes.byref(fl), ctypes.byref(xfl)), "profile")
    return ms.value, n.value, fl.value, xfl.value


def conv_roofline(conv_ms, conv_n, conv_fl, conv_xfl, prof_steps, ms_per_step, peaks):
    """`frac` is the tensor-pipe utilisation: MACs actually ISSUED (dead-halo rows skipped, split-precision terms
    counted) per second over the measured sustained cuBLAS bf16 rate.  The algorithmic figure (every MAC the reference
    executes on its tile grid / kernel time) is kept beside it; it can exceed 1 because 39 % of those MACs are skipped."""
    traffic, traffic_src = None, None
    for name in ("r02_conv_dram_traffic.json", "r01_conv_dram_traffic.json"):
        try:   # per-launch DRAM bytes of the conv kernel from the committed ncu capture of this same command
            with open(os.path.join(ROOT, "profiles", name)) as f:
                t = json.load(f)
            traffic, traffic_src = float(t["dram_bytes_per_launch"]), "profiles/" + name
            break
        except Exception:  # noqa: BLE001
            pass
    alg = conv_fl / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0
    issued = conv_xfl / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0
    return dict(bound="tensor", kernel="conv_igemm_kernel (tcgen05 implicit-GEMM conv3d)", achieved=issued,
                peak=peaks["tflops"], unit="TFLOP/s", frac=issued / peaks["tflops"],
                peak_source=peaks["source"] + ": sustained cuBLAS bf16 (fp16 runs at the same tcgen05 kind::f16 rate); "
                            f"burst {peaks['tflops_burst']}",
                frac_of_burst=issued / peaks["tflops_burst"], traffic=traffic, traffic_source=traffic_src,
                launches_per_step=conv_n / prof_steps, kernel_ms_per_step=conv_ms / prof_steps,
                share_of_step=(conv_ms / prof_steps) / ms_per_step if ms_per_step else None,
                issued_flops_per_step=conv_xfl / prof_steps, algorithmic_flops_per_step=conv_fl / prof_steps,
                algorithmic_achieved=alg, algorithmic_frac=alg / peaks["tflops"],
                note="achieved / frac = MACs issued to the tensor pipe; algorithmic_* counts every MAC the reference "
                     "executes on its tile grid (SURVEY §8d), of which the dead-halo elimination skips 39 % while the "
                     "split-precision layers issue some twice")


def base_line(args, world, config, value, unit, ms_per_step, dtype, **extra):
    line = dict(metric=METRIC if config in ("full", "batch64") else
                {"seg": "knee volumes/sec (segmentation stage)", "reg": "registration pairs/sec (GradICON, both directions)",
                 "warp-sweep": "warp/composition HBM GB/s (algorithmic bytes)"}[config],
                value=value, unit=unit, n_gpus=world, steps=args.steps, warmup=args.warmup, ms_per_step=ms_per_step,
                higher_is_better=True, scaling="strong" if config == "batch64" else "weak", vs_baseline=None,
                dtype=dtype, data="synthetic",
                config=dict(workload=WORKLOADS[config],
                            weights="random init (reference UNet.weights_init / icon default init)",
                            l2="per-step working set (tens of GB of activations / > 126 MB per warp case) exceeds L2; "
                               "inputs rotate over distinct volumes; the warp sweep rewrites a 256 MB buffer between "
                               "cases"))
    line.update(extra)
    return line


SEG_DTYPE = {"mixed": "fp16 operands / fp32 accumulate (tcgen05 kind::f16), the full-resolution decoder layers read fp16 "
                      "hi+lo activations (dc2: skip input only; dc1)",
             "fp16": "fp16 operands / fp32 accumulate (tcgen05 kind::f16)", "bf16": "bf16 operands / fp32 accumulate",
             "fp16x2": "fp16 hi+lo activations x fp16 weights / fp32 accumulate",
             "fp16x3": "fp16 hi+lo activations x fp16 hi+lo weights / fp32 accumulate (fp32-faithful)"}


# ----------------------------------------------------------------------------------------------- config: full
def run_full(args):
    import torch

    from oai_analysis_2_b200 import _lib, sharding

    rank, world, local = sharding.init_process_group()
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    pipe, geom = build_pipeline(device, args.tiles_per_batch)
    precision = pipe.segmenter.model.precision
    vols_h, verts_h = make_inputs(rank)
    vols_d = [torch.from_numpy(v).to(device) for v in vols_h]
    verts_d = torch.from_numpy(verts_h).to(device)
    vols_pin = [torch.from_numpy(v).pin_memory() for v in vols_h]
    verts_pin = torch.from_numpy(verts_h).pin_memory()

    # the drop-in entry points first, eagerly, while the allocator is still empty (the CUDA graph captured below keeps
    # its activation workspace in a private pool for as long as the graph lives)
    e2e_dropin = None
    if rank == 0 and world == 1 and not args.no_dropin:
        e2e_dropin = dropin_e2e(pipe, vols_h, geom)
        torch.cuda.synchronize()
        torch.cuda.empty_cache()

    launches_per_step = None
    if not args.no_graph:
        # the whole per-knee path is one CUDA graph; the conv profiling events are recorded inside it
        mark = {}

        def on_record():
            if not os.environ.get("OAI_BENCH_NO_CONV_EVENTS"):   # A/B: what the 32 event-record nodes in the graph cost
                _lib.lib.oai_profile_begin()
            mark["n0"] = _lib.launch_count()

        pipe.capture(vols_d[0].shape, geom, verts_d.shape[0], on_record, overlap_registration=args.overlap_registration)
        launches_per_step = _lib.launch_count() - mark["n0"]   # kernels recorded into the graph = launches per replay

    def step_device(i):
        if args.no_graph:
            return pipe.run_device(vols_d[i % len(vols_d)], geom, verts_d)
        return pipe.run_device_graph(vols_d[i % len(vols_d)], geom, verts_d)

    for i in range(args.warmup):
        step_device(i)
    torch.cuda.synchronize()

    sampler = ClockSampler(local)
    sharding.barrier(world)
    if rank == 0:
        sampler.start()
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    if args.no_graph:
        _lib.lib.oai_profile_begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        last = step_device(i)
    e1.record()
    torch.cuda.synchronize()
    conv_ms, conv_n, conv_fl, conv_xfl = conv_profile_end(_lib.lib, _lib.check)
    if args.no_graph:
        launches = _lib.launch_count() - n0
        prof_steps = args.steps
    else:  # the events inside the graph hold the timings of the last replay: one step's worth of conv launches
        launches = launches_per_step * args.steps
        prof_steps = 1
    sharding.barrier(world)
    clocks = sampler.stop() if rank == 0 else None
    ms = sharding.max_over_ranks(e0.elapsed_time(e1), world)
    ms_per_step = ms / args.steps
    value = world * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        # before the e2e arm below replays the graph, which overwrites the static outputs `last` aliases
        dump_outputs(args.dump_outputs, dict(prob=last["prob"], warped=last["warped"], phi_AB=last["phi_AB"].disp,
                                             phi_BA=last["phi_BA"].disp, vertices=last["vertices"]))

    # end to end through the public host API: pinned host volume in, atlas-space maps / fields / vertices out
    pipe.run(vols_pin[0], geom, verts_pin)  # allocates the pinned result buffers
    if not args.no_graph:
        for _ in pipe.run_stream((vols_pin[i % len(vols_pin)], verts_pin) for i in range(2)):
            pass                            # allocates the staging / double-buffered pinned buffers of the stream API
    sharding.barrier(world)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    if args.no_graph:
        for i in range(args.steps):
            res = pipe.run(vols_pin[i % len(vols_pin)], geom, verts_pin)
    else:
        # the public throughput API: every knee's pinned-host volume goes H2D and its results come back D2H inside the
        # timed region; the copies of neighbouring knees overlap the compute of the current one
        for res in pipe.run_stream(((vols_pin[i % len(vols_pin)], verts_pin) for i in range(args.steps))):
            checksum = float(res["vertices_atlas"][0, 0]) + float(res["FC_atlas"][80, 192, 192])  # noqa: F841
    torch.cuda.synchronize()
    e2e_s = sharding.max_over_ranks(time.perf_counter() - t0, world)
    sharding.barrier(world)
    e2e = dict(value=world * args.steps / e2e_s, unit="volumes/s", h2d_bytes_per_step=int(res["h2d_bytes"]),
               d2h_bytes_per_step=int(res["d2h_bytes"]), ms_per_step=1e3 * e2e_s / args.steps,
               api="KneePipeline.run_stream (pinned host volume in; atlas-space maps, displacement fields and warped "
                   "vertices out; copies of neighbouring knees overlap the compute)")

    peaks = load_peaks()
    line = base_line(args, world, "full", value, "volumes/s", ms_per_step,
                     SEG_DTYPE[precision] + "; fp32 registration; fp64 warp coordinates",
                     e2e=e2e, gpu_launches=int(launches * world),
                     roofline=conv_roofline(conv_ms, conv_n, conv_fl, conv_xfl, prof_steps, ms_per_step, peaks),
                     clocks=clocks)
    line["config"]["seg_precision"] = precision
    line["config"]["seg_tflop_per_volume"] = SEG_FLOP_PER_VOLUME / 1e12
    if rank == 0:
        if world == 1:
            if e2e_dropin is not None:
                line["e2e_dropin"] = e2e_dropin
            if not args.no_library_bar:
                import gc
                del vols_d, verts_d, res
                pipe.release_graph()   # the graph's private pool (activation workspace) goes back to the allocator
                del pipe
                gc.collect()
                torch.cuda.empty_cache()
                line["library_bar"] = library_bar(vols_h[0], "full")
            if not args.no_cpu_baseline:
                line["cpu_baseline"] = cpu_reference_sample(vols_h[0], "full", seg_batches=2)
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def dropin_e2e(pipe, vols_h, geom):
    """The calls a reference user makes, one knee at a time, host objects in and out (analysis_object.py:43-49,
    dask_processing.py:95-111): AnalysisObject.segment -> (FC, TC) float64 images; AnalysisObject.register -> transform;
    deform_probmap x 2 -> float64 images on the atlas grid.  Synchronous, no overlap across knees."""
    import torch

    from oai_analysis_2_b200 import itk_compat
    from oai_analysis_2_b200.analysis_object import AnalysisObject
    from oai_analysis_2_b200.dask_processing import deform_probmap
    from oai_analysis_2_b200.registration import ICON_Registration
    sp = tuple(float(v) for v in geom.spacing)
    atlas = itk_compat.Image(pipe.atlas.cpu().numpy(), spacing=sp)
    obj = AnalysisObject(segmenter_config=pipe.segmenter.config, registerer=ICON_Registration(model=pipe.reg_model),
                         atlas_image=atlas)
    obj.segmenter = pipe.segmenter   # same weights (and the already packed layers) as the device-timed arm
    times = []
    devnull = open(os.devnull, "w")
    for rep in range(3):
        img = itk_compat.Image(vols_h[rep % len(vols_h)], spacing=sp)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fc, tc = obj.segment(img)
        stdout, sys.stdout = sys.stdout, devnull   # ICON_Registration.register prints the intensity ranges (as the reference does)
        try:
            phi_AB = obj.register(img)
        finally:
            sys.stdout = stdout
        fc_w = deform_probmap(phi_AB, img, atlas, fc, "FC")
        tc_w = deform_probmap(phi_AB, img, atlas, tc, "TC")
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    nvox = int(np.prod(vols_h[0].shape))
    return dict(value=1.0 / min(times[1:]), unit="volumes/s", ms_per_step=1e3 * min(times[1:]),
                api="AnalysisObject.segment + AnalysisObject.register + deform_probmap x2 (reference signatures; float64 "
                    "host images out, as the reference returns them)",
                h2d_bytes_per_step=4 * nvox * 2 + 2 * 4 * nvox, d2h_bytes_per_step=2 * 4 * nvox + 2 * 4 * nvox,
                checksum=float(itk_compat.array_from_image(fc_w)[80, 192, 192] + itk_compat.array_from_image(tc_w)[80, 192, 192]))


# ----------------------------------------------------------------------------------------------- library bar (GPU)
def library_bar(vol, config):
    """The reference's own torch-CUDA path on THIS GPU, timed with CUDA events (SURVEY §2.2: "the bar to beat").
    Segmentation: the same torch ops the reference's UNet issues (networks.py:109-149: cuDNN conv3d / conv_transpose3d /
    batch_norm / max_pool3d / cat) over the 160 tiles at batch 4 (segmenter.py:109-119, analysis_object.py:23), tiles
    resident on the device, with torch's defaults (cuDNN TF32 on) and under fp16 autocast.  Registration: the oracle's
    module-for-module restatement of icon_registration on cuda (8 tallUNet2 forwards + the closures' grid_samples).
    Warps: F.grid_sample of the two class maps through a dense 160x384x384 grid (ATen's trilinear gather; ITK's own
    resampler is CPU-only)."""
    import torch
    import torch.nn.functional as F

    from oracle import reg_oracle, seg_oracle
    dev = torch.device("cuda")
    out = {}

    def timed(fn, reps=1):
        fn()   # warm-up (cuDNN heuristics / autotune)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    if config in ("full", "seg"):
        sd = {k: v.to(dev) for k, v in seg_oracle.make_unet_state_dict(1234, 1, 2, True, True, False).items()}
        tiles, _ = seg_oracle.partition(vol, PATCH, OVERLAP)
        tiles = tiles.to(dev)

        def seg_pass(n_tiles=None):
            n = tiles.shape[0] if n_tiles is None else n_tiles
            with torch.no_grad():
                for i in range(0, n, 4):
                    torch.sigmoid(seg_oracle.unet_forward(sd, tiles[i:i + 4], True))

        for name, tf32, autocast in (("cudnn_tf32 (torch defaults)", True, False), ("fp16_autocast", True, True),
                                     ("fp32 (TF32 off)", False, False)):
            torch.backends.cudnn.allow_tf32 = tf32
            try:
                with torch.autocast("cuda", dtype=torch.float16, enabled=autocast):
                    seg_pass(8)
                    ms = timed(seg_pass)
            finally:
                torch.backends.cudnn.allow_tf32 = True
            out["seg_forward_ms " + name] = ms
            out["seg_tflops " + name] = SEG_FLOP_PER_VOLUME / ms / 1e9
        del tiles, sd
        torch.cuda.empty_cache()
    if config in ("full", "reg"):
        nets = {k: {kk: vv.to(dev) for kk, vv in v.items()}
                for k, v in reg_oracle.split_state_dict(reg_oracle.make_gradicon_state_dict(4321)).items()}
        A = reg_oracle.resize_to_network(vol).to(dev)
        B = reg_oracle.resize_to_network(vol[:, ::-1, :].copy()).to(dev)
        _ident = reg_oracle.identity_map
        reg_oracle.identity_map = lambda shape, dtype=torch.float32: _ident(shape, dtype).to(dev)

        def reg_pass():
            with torch.no_grad():
                for a, b in ((A, B), (B, A)):
                    reg_oracle.final_map(reg_oracle.regis_net_forward(nets, a, b), reg_oracle.INPUT_SHAPE)

        try:
            out["reg_forward_ms (icon modules restated in torch, cuda, both directions)"] = timed(reg_pass, 2)
        finally:
            reg_oracle.identity_map = _ident
        del nets, A, B
        torch.cuda.empty_cache()
    if config in ("full",):
        prob = torch.rand(1, 2, *vol.shape, device=dev)
        grid = torch.rand(1, *vol.shape, 3, device=dev) * 2 - 1
        out["warp_grid_sample_ms (2 class maps, 160x384x384)"] = timed(
            lambda: F.grid_sample(prob, grid, mode="bilinear", padding_mode="zeros", align_corners=True), 3)
        del prob, grid
        torch.cuda.empty_cache()
    total = sum(v for k, v in out.items() if k.startswith(("seg_forward_ms cudnn_tf32", "reg_forward_ms", "warp_grid")))
    best = sum(v for k, v in out.items() if k.startswith(("seg_forward_ms fp16_autocast", "reg_forward_ms", "warp_grid")))
    out["ms_per_volume (torch defaults: cuDNN TF32)"] = total
    out["volumes_per_s (torch defaults: cuDNN TF32)"] = 1e3 / total if total else None
    out["volumes_per_s (fp16 autocast)"] = 1e3 / best if best else None
    out["note"] = ("device-resident inputs, CUDA events, no host round trips: a lower bound on the reference's GPU "
                   "wall time (its segment() also moves every tile batch H2D/D2H and assembles on the host)")
    return out


# ----------------------------------------------------------------------------------------------- CPU reference arm
def cpu_reference_sample(vol, config, seg_batches=1):
    """Time the oracle (CPU restatement of the reference path) on a bounded sample and scale to the config's unit.
    Segmentation runs `seg_batches` batches of 4 tiles (the reference's batch_size, analysis_object.py:23);
    registration runs both directions of the lean cascade (the reference additionally evaluates loss terms that
    register_pair discards); the ITK-style warp runs a 2^20-voxel sample of one map."""
    import torch

    from oracle import reg_oracle, seg_oracle, warp_oracle

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    parts, t_volume = [], 0.0
    nvox = int(np.prod(vol.shape))
    phi = None
    if config in ("full", "seg", "batch64"):
        sd = seg_oracle.make_unet_state_dict(1234, 1, 2, True, True, False)
        tiles, g = seg_oracle.partition(vol, PATCH, OVERLAP)
        n_tiles = tiles.shape[0]
        with torch.no_grad():
            t0 = time.perf_counter()
            for i in range(seg_batches):
                torch.sigmoid(seg_oracle.unet_forward(sd, tiles[4 * i:4 * i + 4], True))
            t_seg_tile = (time.perf_counter() - t0) / (4 * seg_batches)
        t_volume += t_seg_tile * n_tiles
        parts.append(f"{4 * seg_batches} of {n_tiles} UNet tiles at batch 4 ({t_seg_tile:.2f} s/tile)")
    if config in ("full", "reg", "batch64"):
        rsd = reg_oracle.make_gradicon_state_dict(4321)
        nets = reg_oracle.split_state_dict(rsd)
        A = reg_oracle.resize_to_network(vol)
        B = reg_oracle.resize_to_network(vol[:, ::-1, :].copy())
        with torch.no_grad():
            t0 = time.perf_counter()
            phi = reg_oracle.final_map(reg_oracle.regis_net_forward(nets, A, B), reg_oracle.INPUT_SHAPE)
            reg_oracle.final_map(reg_oracle.regis_net_forward(nets, B, A), reg_oracle.INPUT_SHAPE)
            t_reg = time.perf_counter() - t0
            if config == "reg":
                t0 = time.perf_counter()
                reg_oracle.sample(A, phi)
                t_reg += time.perf_counter() - t0
        t_volume += t_reg
        parts.append(f"both GradICON directions, lean ({t_reg:.1f} s)")
    if config in ("full", "batch64"):
        geom = warp_oracle.Geometry(vol.shape[::-1], (0.3646, 0.3646, 0.7))
        tr = warp_oracle.CompositeTransform(reg_oracle.displacement_field_xyz(phi), geom, geom)
        sample = 1 << 20
        W, H = vol.shape[2], vol.shape[1]
        lin = np.arange(sample) * (nvox // sample)
        j = np.stack([lin % W, (lin // W) % H, lin // (W * H)], -1)
        t0 = time.perf_counter()
        q = tr.transform_points(geom.index_to_physical(j))
        idx = geom.physical_to_index(q)
        warp_oracle._trilinear_clamped(vol.astype(np.float64), idx[..., ::-1])
        t_warp = (time.perf_counter() - t0) / sample
        t0 = time.perf_counter()
        tr.transform_points(geom.index_to_physical(j[:85370]))
        t_pts = time.perf_counter() - t0
        t_volume += 2 * nvox * t_warp + t_pts
        parts.append(f"2^20 of {nvox} warp voxels of one of the two maps, 85370 vertices")
    unit = "pairs/s" if config == "reg" else "volumes/s"
    return dict(value=1.0 / t_volume, unit=unit, cores=cores, kind="port", seconds_per_unit=t_volume,
                sample=f"oracle (torch fp32 / numpy f64 port of the reference path) on {cores} host threads: "
                       + "; ".join(parts) + "; scaled to one " + ("pair" if config == "reg" else "knee"))


def cpu_warp_sample(n=128):
    """CPU leg of the warp sweep: the float64 ITK-semantics oracle on one n^3 single-channel case."""
    from oracle import warp_oracle
    rng = np.random.default_rng(7)
    img = rng.random((n, n, n))
    geom = warp_oracle.Geometry((n, n, n))
    disp = rng.standard_normal((n, n, n, 3)) * 2.0
    tr = warp_oracle.CompositeTransform(disp, geom, geom)
    sample = min(n ** 3, 1 << 20)
    lin = np.arange(sample) * (n ** 3 // sample)
    j = np.stack([lin % n, (lin // n) % n, lin // (n * n)], -1)
    t0 = time.perf_counter()
    q = tr.transform_points(geom.index_to_physical(j))
    warp_oracle._trilinear_clamped(img, geom.physical_to_index(q)[..., ::-1])
    dt = time.perf_counter() - t0
    gbs = 20.0 * sample / dt / 1e9
    return dict(value=gbs, unit="GB/s", cores=os.cpu_count() or 1, kind="port",
                sample=f"float64 ITK-semantics oracle (numpy) on {sample} voxels of a {n}^3 single-channel warp, "
                       f"20 algorithmic bytes per voxel")


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    from oai_analysis_2_b200 import synthetic
    vol = synthetic.synthetic_knee(synthetic.OAI_SHAPE, seed=100)
    vals = []
    for i in range(args.warmup + args.steps):
        r = cpu_warp_sample() if args.config == "warp-sweep" else cpu_reference_sample(vol, args.config, seg_batches=1)
        if i >= args.warmup:
            vals.append(r)
    v = float(np.mean([r["value"] for r in vals]))
    cb = dict(vals[-1], value=v)
    cfg = "full" if args.config == "batch64" else args.config
    line = base_line(args, args.gpus, args.config, v, cb["unit"], 1e3 / v if cb["unit"] != "GB/s" else None,
                     "fp32 (torch CPU) / fp64 (ITK-style warps)", impl="reference", cpu_baseline=cb,
                     e2e=dict(value=v, unit=cb["unit"], h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    line["config"]["note"] = ("icon_registration / itk are not installable offline, so the registration and warp legs run "
                              "the oracle port; the UNet leg is the reference's own torch ops.  Each step times a bounded "
                              "sample of the " + cfg + " workload and scales it to one unit: an EXTRAPOLATED CPU figure, "
                              "not a full run")
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- config: seg
def run_seg(args):
    import torch

    from oai_analysis_2_b200 import _lib, sharding
    rank, world, local = sharding.init_process_group()
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    seg = build_segmenter(device, args.tiles_per_batch)
    vols_h, _ = make_inputs(rank)
    vols_d = [torch.from_numpy(v).to(device) for v in vols_h]
    out = torch.empty((2,) + tuple(vols_d[0].shape), dtype=torch.float32, device=device)
    for i in range(args.warmup):
        seg.segment_device(vols_d[i % 2], True, out=out)
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sharding.barrier(world)
    if rank == 0:
        sampler.start()
    n0 = _lib.launch_count()
    _lib.lib.oai_profile_begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        seg.segment_device(vols_d[i % 2], True, out=out)
    e1.record()
    torch.cuda.synchronize()
    conv_ms, conv_n, conv_fl, conv_xfl = conv_profile_end(_lib.lib, _lib.check)
    launches = _lib.launch_count() - n0
    sharding.barrier(world)
    clocks = sampler.stop() if rank == 0 else None
    ms = sharding.max_over_ranks(e0.elapsed_time(e1), world)
    # e2e: the drop-in entry point, host image in, two float64 host maps out (segmenter.py:100-131)
    seg.segment(vols_h[0], if_output_prob_map=True, if_output_itk=False)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(args.steps):
        fc, tc = seg.segment(vols_h[i % 2], if_output_prob_map=True, if_output_itk=False)
    e2e_s = sharding.max_over_ranks(time.perf_counter() - t0, world)
    nvox = int(np.prod(vols_h[0].shape))
    peaks = load_peaks()
    line = base_line(args, world, "seg", world * args.steps / (ms * 1e-3), "volumes/s", ms / args.steps,
                     SEG_DTYPE[seg.model.precision],
                     e2e=dict(value=world * args.steps / e2e_s, unit="volumes/s", h2d_bytes_per_step=4 * nvox,
                              d2h_bytes_per_step=8 * nvox, ms_per_step=1e3 * e2e_s / args.steps,
                              api="Segmenter3DInPatchClassWise.segment (numpy volume in, FC/TC float64 numpy out)"),
                     gpu_launches=int(launches * world),
                     roofline=conv_roofline(conv_ms, conv_n, conv_fl, conv_xfl, args.steps, ms / args.steps, peaks),
                     clocks=clocks)
    line["config"]["seg_precision"] = seg.model.precision
    if rank == 0:
        if world == 1:
            if not args.no_library_bar:
                del seg
                torch.cuda.empty_cache()
                line["library_bar"] = library_bar(vols_h[0], "seg")
            if not args.no_cpu_baseline:
                line["cpu_baseline"] = cpu_reference_sample(vols_h[0], "seg", seg_batches=2)
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


# ----------------------------------------------------------------------------------------------- config: reg
def run_reg(args):
    import torch

    from oai_analysis_2_b200 import _lib, itk_compat, ops, sharding
    from oai_analysis_2_b200.icon_registration import itk_wrapper
    rank, world, local = sharding.init_process_group()
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    reg = build_reg_model().to(device)
    vols_h, _ = make_inputs(rank)
    A = torch.from_numpy(vols_h[0]).to(device)
    B = torch.from_numpy(vols_h[1]).to(device)
    shape = tuple(reg.identity_map.shape[2:])
    img80 = torch.empty(shape, dtype=torch.float32, device=device)

    def step():
        # register_pair up to the maps (resize of both volumes, 8 tallUNet2 forwards batched over the two directions, the
        # intermediate warps, the final composition) + the warp of image A by phi_AB (config 2's "image warp")
        phi_AB, phi_BA = itk_wrapper.register_pair_device(reg, A, B)
        reg.warp_image(ops.resize_trilinear(A, shape), 0, out=img80)
        return phi_AB, phi_BA

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    graph = None
    if not args.no_graph:
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            step()
        graph.replay()
        torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sharding.barrier(world)
    if rank == 0:
        sampler.start()
    n0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        if graph is not None:
            graph.replay()
        else:
            step()
    e1.record()
    torch.cuda.synchronize()
    if graph is None:
        launches = _lib.launch_count() - n0
    else:
        n1 = _lib.launch_count()
        step()
        launches = (_lib.launch_count() - n1) * args.steps
        torch.cuda.synchronize()
    sharding.barrier(world)
    clocks = sampler.stop() if rank == 0 else None
    ms = sharding.max_over_ranks(e0.elapsed_time(e1), world)
    ms_per_step = ms / args.steps
    # e2e: the reference's call, host images in, two transforms out with their float64 displacement fields on the host
    sp = (0.3646, 0.3646, 0.7)
    imA, imB = itk_compat.Image(vols_h[0], spacing=sp), itk_compat.Image(vols_h[1], spacing=sp)
    itk_wrapper.register_pair(reg, imA, imB)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        tAB, tBA = itk_wrapper.register_pair(reg, imA, imB)
        fa, fb = tAB.displacement_field_array(), tBA.displacement_field_array()
    e2e_s = sharding.max_over_ranks(time.perf_counter() - t0, world)
    peaks = load_peaks()
    gbs = REG_BYTES_PER_PAIR / (ms_per_step * 1e-3) / 1e9
    roof = dict(bound="hbm", kernel="registration stage (tallUNet2 x8 + compositions + warps; ~100 launches)",
                achieved=gbs, peak=peaks["hbm"], unit="GB/s", frac=gbs / peaks["hbm"], peak_source=peaks["source"],
                traffic=None, stage_ms=ms_per_step,
                note="achieved = SURVEY §8(d)'s ideal 2.6 GB of fp32 traffic per pair / stage time: the whole stage "
                     "against the HBM roofline (its kernels are small-channel convolutions, latency- and issue-bound)")
    nvox = int(np.prod(vols_h[0].shape))
    line = base_line(args, world, "reg", world * args.steps / (ms * 1e-3), "pairs/s", ms_per_step,
                     "fp32 (CUDA-core convs; split-fp16 mma.sync transposed convs with fp32-level accuracy)",
                     e2e=dict(value=world * args.steps / e2e_s, unit="pairs/s", h2d_bytes_per_step=8 * nvox,
                              d2h_bytes_per_step=int(fa.size + fb.size) * 4, ms_per_step=1e3 * e2e_s / args.steps,
                              api="icon_registration.itk_wrapper.register_pair + displacement_field_array x2"),
                     gpu_launches=int(launches * world), roofline=roof, clocks=clocks)
    if rank == 0:
        if world == 1:
            if not args.no_library_bar:
                line["library_bar"] = library_bar(vols_h[0], "reg")
            if not args.no_cpu_baseline:
                line["cpu_baseline"] = cpu_reference_sample(vols_h[0], "reg")
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


# ----------------------------------------------------------------------------------------------- config: warp-sweep
def run_warp_sweep(args):
    import torch

    from oai_analysis_2_b200 import _lib, ops, sharding
    rank, world, local = sharding.init_process_group()
    torch.cuda.set_device(local)
    peaks = load_peaks()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > L2, rewritten between cases
    eye = (np.eye(3), np.zeros(3))
    sizes, chans = (64, 96, 128, 192, 256, 384), (1, 2, 3, 4, 8)

    def smooth_disp(n, sigma_vox=2.0, seed=7):
        g = torch.Generator(device="cuda").manual_seed(seed)
        lo = torch.randn(1, 3, max(2, n // 8), max(2, n // 8), max(2, n // 8), generator=g, device="cuda")
        d = torch.nn.functional.interpolate(lo, size=(n, n, n), mode="trilinear", align_corners=True)[0]
        return (d * sigma_vox).contiguous()

    cases = []
    for n in sizes:
        disp = smooth_disp(n)
        field = disp.permute(1, 2, 3, 0).flip(-1).contiguous()   # [n,n,n,3] x,y,z components, voxels
        for C in chans:
            src = torch.rand(C, n, n, n, device="cuda")
            out = torch.empty_like(src)
            cases.append(dict(op="warp_volume", n=n, C=C, bytes=(12 + 8 * C) * n ** 3,
                              fn=(lambda s=src, f=field, o=out, n=n: ops.warp_volume(s, f, eye, eye, (n, n, n), out=o))))
        u = [(disp / (n - 1)).contiguous(), (smooth_disp(n, 2.0, 8) / (n - 1)).contiguous()]
        phi = torch.empty(3, n, n, n, device="cuda")
        cases.append(dict(op="compose2", n=n, C=3, bytes=36 * n ** 3,
                          fn=(lambda u=u, p=phi, n=n: ops.compose((n, n, n), u, False, phi_out=p))))
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in cases]
    acc = np.zeros(len(cases))

    def one_pass(record):
        for k, c in enumerate(cases):
            flush.zero_()
            if record:
                ev[k][0].record()
            c["fn"]()
            if record:
                ev[k][1].record()
        if record:
            torch.cuda.synchronize()
            for k in range(len(cases)):
                acc[k] += ev[k][0].elapsed_time(ev[k][1])

    for _ in range(max(args.warmup, 3)):
        one_pass(False)
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    n0 = _lib.launch_count()
    for _ in range(args.steps):
        one_pass(True)
    launches = _lib.launch_count() - n0
    clocks = sampler.stop() if rank == 0 else None
    sweep = []
    for k, c in enumerate(cases):
        ms = acc[k] / args.steps
        sweep.append(dict(op=c["op"], n=c["n"], C=c["C"], ms=ms, gbs=c["bytes"] / ms / 1e6,
                          frac=c["bytes"] / ms / 1e6 / peaks["hbm"]))
    tot_b, tot_ms = sum(c["bytes"] for c in cases), float(acc.sum() / args.steps)
    big = [s for s in sweep if s["n"] == 384]
    dom = max(big, key=lambda s: s["ms"])
    roof = dict(bound="hbm", kernel=f"{'warp_volume_kernel' if dom['op'] == 'warp_volume' else 'chain_kernel'} "
                                    f"({dom['op']} {dom['n']}^3 C={dom['C']}: the longest case of the sweep)",
                achieved=dom["gbs"], peak=peaks["hbm"], unit="GB/s", frac=dom["frac"], peak_source=peaks["source"],
                traffic=None, min_frac_384=min(s["frac"] for s in big), max_frac_384=max(s["frac"] for s in big),
                note="algorithmic bytes per voxel (SURVEY §8d): warp 12 + 8 C, composition 36")
    line = base_line(args, world, "warp-sweep", tot_b / tot_ms / 1e6, "GB/s", tot_ms,
                     "fp32 data, fp64 coordinate arithmetic (ITK semantics)",
                     e2e=None, gpu_launches=int(launches), roofline=roof, clocks=clocks, sweep=sweep)
    # e2e for a microbenchmark: the public resample call with host arrays in and out (one 384^3 single-channel warp)
    from oai_analysis_2_b200.transforms import CompositeTransform, Geometry
    n = 384
    g = Geometry((n, n, n))
    tr = CompositeTransform(smooth_disp(n // 2).permute(1, 2, 3, 0).flip(-1).contiguous(), g, g)
    host = torch.rand(1, n, n, n).pin_memory()
    res = torch.empty(1, n, n, n).pin_memory()
    for rep in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res.copy_(tr.resample_device(host.cuda(non_blocking=True), g, g), non_blocking=True)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    line["e2e"] = dict(value=20.0 * n ** 3 / dt / 1e9, unit="GB/s", h2d_bytes_per_step=4 * n ** 3,
                       d2h_bytes_per_step=4 * n ** 3, ms_per_step=1e3 * dt,
                       api="CompositeTransform.resample_device on a pinned host volume (H2D + warp + D2H), 384^3 C=1")
    if rank == 0:
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_warp_sample()
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


# ----------------------------------------------------------------------------------------------- config: batch64
def run_batch64(args):
    import torch

    from oai_analysis_2_b200 import _lib, sharding, synthetic
    rank, world, local = sharding.init_process_group()
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    knees = args.knees
    pipe, geom = build_pipeline(device, args.tiles_per_batch)
    verts = np.concatenate([synthetic.synthetic_vertices(synthetic.N_VERTS_FC, seed=0),
                            synthetic.synthetic_vertices(synthetic.N_VERTS_TC, seed=1000)])
    mark = {}

    def on_record():
        mark["n0"] = _lib.launch_count()
    pipe.capture(synthetic.OAI_SHAPE, geom, verts.shape[0], on_record)
    per_knee = _lib.launch_count() - mark["n0"]
    bases = [synthetic.synthetic_knee(synthetic.OAI_SHAPE, seed=200 + k) for k in range(2)]

    def knee_volume(i):
        b = bases[i % len(bases)]
        v = b[:, ::-1, :] if (i // len(bases)) % 2 else b
        return np.ascontiguousarray(np.roll(v, 7 * (i // (2 * len(bases))) + 3 * i, axis=2))

    mine = sharding.shard_indices(knees, rank, world)    # knee i -> rank i % world (static round-robin)
    pins = [torch.from_numpy(knee_volume(i)).pin_memory() for i in mine[:4]]
    vp = torch.from_numpy(verts).pin_memory()

    def items():
        for k, i in enumerate(mine):
            slot = pins[k % len(pins)]
            if k >= len(pins):
                slot.copy_(torch.from_numpy(knee_volume(i)))   # host-side producer (would be the image reader)
            yield slot, vp

    for _ in pipe.run_stream((pins[k % len(pins)], vp) for k in range(max(2, args.warmup))):
        pass
    sampler = ClockSampler(local)
    sharding.barrier(world)
    if rank == 0:
        sampler.start()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    recs = []
    for _ in range(args.steps):
        recs = []
        for i, res in zip(mine, pipe.run_stream(items())):
            recs.append(dict(index=i, rank=rank, fc_sum=float(res["FC_atlas"].sum(dtype=np.float64)),
                             tc_sum=float(res["TC_atlas"].sum(dtype=np.float64)),
                             vert_sum=float(res["vertices_atlas"].sum())))
    torch.cuda.synchronize()
    dt = sharding.max_over_ranks(time.perf_counter() - t0, world)
    clocks = sampler.stop() if rank == 0 else None
    merged = sharding.gather_records(recs, rank, world)   # host-side gather of small records: the only communication
    value = knees * args.steps / dt
    line = base_line(args, world, "batch64", value, "volumes/s", 1e3 * dt / args.steps,
                     SEG_DTYPE[pipe.segmenter.model.precision] + "; fp32 registration; fp64 warp coordinates",
                     e2e=dict(value=value, unit="volumes/s", h2d_bytes_per_step=int(res["h2d_bytes"]) * knees,
                              d2h_bytes_per_step=int(res["d2h_bytes"]) * knees, ms_per_step=1e3 * dt / args.steps,
                              api="KneePipeline.run_stream over the rank's shard; host-side gather of per-knee records"),
                     gpu_launches=int(per_knee * knees * args.steps), roofline=None, clocks=clocks)
    line["config"]["knees"] = knees
    if rank == 0:
        assert [r["index"] for r in merged] == list(range(knees))
        line["checksum"] = float(sum(r["fc_sum"] + r["tc_sum"] + r["vert_sum"] for r in merged))
        line["roofline"] = dict(bound="tensor", kernel="conv_igemm_kernel", achieved=None, peak=load_peaks()["tflops"],
                                unit="TFLOP/s", frac=None, traffic=None,
                                note="wall-clocked host API run; see --config full for the kernel's roofline line")
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--config", choices=sorted(WORKLOADS), default="full")
    ap.add_argument("--knees", type=int, default=64, help="--config batch64: knees in the batch")
    ap.add_argument("--tiles-per-batch", type=int, default=None)
    ap.add_argument("--precision", default=None, choices=["fp16", "mixed", "fp16x2", "fp16x3", "bf16"],
                    help="segmentation precision plan (default: the product default, 'mixed')")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library-bar", action="store_true")
    ap.add_argument("--no-dropin", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying the CUDA graph")
    ap.add_argument("--overlap-registration", action="store_true",
                    help="A/B: record the registration as a parallel branch of the per-knee graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="--config full: write what the last timed step computed (rank 0) to DIR/<name>.npy: the FC/TC "
                         "probability maps (prob), the maps on the atlas grid (warped), the displacement fields of both "
                         "directions (phi_AB, phi_BA) and the warped vertices; arrays over 8 MB as a fixed-seed sample")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.config != "full"):
        ap.error("--dump-outputs is implemented for --impl b200 --config full")
    if args.precision:
        os.environ["OAI_B200_SEG_PRECISION"] = args.precision
    if args.impl == "reference":
        run_reference(args)
    else:
        {"full": run_full, "seg": run_seg, "reg": run_reg, "warp-sweep": run_warp_sweep, "batch64": run_batch64}[
            args.config](args)


if __name__ == "__main__":
    main()
