#!/usr/bin/env python
"""bench.py -- hair-swap hot-path throughput on B200 (contract: see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--triples T]

A *step* = the SURVEY-8 hot path of T HairFast.swap() triples (SURVEY.md Appendix B census), the T triples'
calls batched together (independent triples, BASELINE config 5):
  * the eight Generator.forward calls of a triple (full x3 [FSE recon], 3->3 x3, 0->3 x3, full x1, 0->3 x2,
    full x1, 4->8 x1, 5->8 x1: 1057.6 GFLOP, 1024^2, randomize_noise=True like the reference),
  * e4e Encoder4Editing on 3 + 2 images and FeatureStyleEncoder fs_encoder_v2 on 3 images at 256^2
    (720.5 + 208.7 GFLOP),
  * the PostProcess conv stack (SURVEY 8f-1): FeatureEncoderMult on 2 images at 256^2 and FeatureiResnet on the
    concatenated 1024-channel 64^2 content maps (180.2 + 594.3 GFLOP),
  * BiSeNet face parsing (SURVEY 8f-3) on 3 images at 512^2 and 2 at 1024^2 (302.5 GFLOP),
i.e. 3063.8 algorithmic GFLOP per triple.  Not in the step: stage glue (resizes, masks, lerps) and the out-of-scope
nets (SEAN / CLIP / mask nets).  `value` times the step with inputs resident in HBM;
`e2e` times it through the public Python API with HOST (pinned) inputs copied in and the T final images
copied out inside the timed region.

One JSON line on stdout (rank 0).  Multi-GPU: one process per GPU under torchrun, weights broadcast from
rank 0 over NCCL at init, no collective in the step; time = max over ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GFLOP_FULL, GFLOP_0_3, GFLOP_3_3, GFLOP_4_8, GFLOP_5_8 = 148.52, 8.007, 6.043, 140.51, 116.34
GFLOP_GEN_PER_TRIPLE = 3 * GFLOP_FULL + 3 * GFLOP_3_3 + 3 * GFLOP_0_3 + GFLOP_FULL + 2 * GFLOP_0_3 + GFLOP_FULL \
    + GFLOP_4_8 + GFLOP_5_8                               # = 1057.6 (SURVEY Appendix B)
GFLOP_E4E_IMG, GFLOP_FSE_IMG = 144.1, 69.6                # SURVEY 8a rows a13 / a14
GFLOP_ENC_PER_TRIPLE = 5 * GFLOP_E4E_IMG + 3 * GFLOP_FSE_IMG
GFLOP_PP_ENC_IMG, GFLOP_PP_RES = 90.1, 594.3              # SURVEY 8d config 3: PostProcess FeatureEncoderMult / FeatureiResnet
GFLOP_PP_PER_TRIPLE = 2 * GFLOP_PP_ENC_IMG + GFLOP_PP_RES
GFLOP_SEG_512 = 27.5                                      # BiSeNet (ResNet-18 context path + heads) on one 512^2 image
GFLOP_SEG_PER_TRIPLE = 3 * GFLOP_SEG_512 + 2 * 4 * GFLOP_SEG_512      # 3 calls at 512^2, 2 at 1024^2 (SURVEY 8f-3)
GFLOP_PER_TRIPLE = GFLOP_GEN_PER_TRIPLE + GFLOP_ENC_PER_TRIPLE + GFLOP_PP_PER_TRIPLE + GFLOP_SEG_PER_TRIPLE   # = 3063.8
ROOFLINE_US_PER_IMG = 142.5                               # SURVEY Appendix A, sum of per-layer maxima


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sustained": d["bf16_tflops_sustained"],
                "src": "measured"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def mark(self):
        return len(self.rows)

    def stop(self, first: int = 0):
        if self.proc:
            self.proc.terminate()
        rows = self.rows[first:] or self.rows
        sm = sorted(int(float(r[0])) for r in rows if r and r[0].replace(".", "").isdigit())
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        smax = int(float(rows[0][1])) if rows else None
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def census(T: int):
    """(start_layer, end_layer, batch, layer_in resolution) of the 8 generator calls of T batched triples."""
    return [(0, 8, 3 * T, None), (3, 3, 3 * T, 16), (0, 3, 3 * T, None), (0, 8, T, None), (0, 3, 2 * T, None),
            (0, 8, T, None), (4, 8, T, 32), (5, 8, T, 64)]


def make_host_inputs(T: int, seed: int):
    """Pinned host inputs of one step of T triples (seeded: rank r of an N-GPU run uses seed 100 + r, so any rank's
    batch can be rebuilt anywhere for the output-equality check)."""
    import torch
    calls = census(T)
    g = torch.Generator(device="cpu").manual_seed(seed)
    lat = [torch.randn(b, 18, 512, generator=g).pin_memory() for (_, _, b, _) in calls]
    lin = [None if r is None else torch.randn(b, 512, r, r, generator=g).pin_memory() for (_, _, b, r) in calls]
    # 256^2 network inputs: e4e (3T), e4e (2T), FSE (3T), PostProcess source (T) and target (T)
    img = [(torch.rand(n * T, 3, 256, 256, generator=g) * 2 - 1).pin_memory() for n in (3, 2, 3, 1, 1)]
    # BiSeNet inputs: the three 512^2 images of a triple (Embedding.py:81) and two 1024^2 ones (Alignment / Blending)
    img += [(torch.rand(3 * T, 3, 512, 512, generator=g) * 2 - 1).pin_memory(),
            (torch.rand(T, 3, 1024, 1024, generator=g) * 2 - 1).pin_memory()]
    return {"T": T, "calls": calls, "lat": lat, "lin": lin, "img": img}


def to_device(inp, dev):
    return {"T": inp["T"], "calls": inp["calls"], "lat": [t.to(dev) for t in inp["lat"]],
            "lin": [None if t is None else t.to(dev) for t in inp["lin"]], "img": [t.to(dev) for t in inp["img"]]}


def image_checksums(final):
    """Two 64-bit integer checksums per image over the raw fp32 bit patterns (bit-exact comparison across ranks)."""
    import torch
    v = final.contiguous().view(torch.int32).view(final.shape[0], -1).to(torch.int64)
    w = (torch.arange(v.shape[1], device=v.device, dtype=torch.int64) % 65521) + 1
    return torch.stack([v.sum(1), (v * w).sum(1)], 1)


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from hairfastgan_b200 import _lib, graphs, sharding
    import hairfastgan_b200.model as M
    import hairfastgan_b200.encoders as E
    torch.set_grad_enabled(False)
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    lib = _lib.lib()                                  # raises if the CUDA library is missing: no fallback
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    T = args.triples

    # ---- synthetic networks: seeded random weights of the reference architectures (no checkpoints exist)
    torch.manual_seed(0)
    gen = M.Generator(1024, 512, 8).to(dev).eval()
    for name, prm in gen.named_parameters():
        if name.endswith("noise.weight") or name.endswith("activate.bias") or name == "to_rgb1.bias" \
                or (name.startswith("to_rgbs.") and name.endswith(".bias") and name.count(".") == 2):
            prm.data.normal_(0, 0.1)
    # the dominant kernel is timed ALONE and first (burst peak in the denominator): later in the run the board sits at
    # its power cap (nvidia-smi: sw_power_cap, ~1.76 GHz) and the same launch measures ~15 % lower
    roofline = roofline_b4 = None
    if rank == 0 and world == 1:
        roofline_b4 = time_dominant_kernel(gen, dev, 4)
        roofline = time_dominant_kernel(gen, dev, 3 * args.triples)      # the batch the step's full forwards use
    e4e = E.Encoder4Editing(50, "ir_se", types.SimpleNamespace(stylegan_size=1024)).to(dev).eval()
    fse = E.fs_encoder_v2(n_styles=18, opts=None, stride=(2, 2)).to(dev).eval()
    import hairfastgan_b200.postprocess as PP
    pp_enc = PP.FeatureEncoderMult(fs_layers=[9], opts=None).to(dev).eval()          # models/Encoders.py:109
    pp_res = PP.FeatureiResnet([[1024, 2], [768, 2], [512, 2]]).to(dev).eval()       # models/Encoders.py:113
    for name, prm in pp_res.named_parameters():      # keep the 6 stacked residual blocks O(1) with random weights
        if name.endswith("bn3.weight") or name.endswith("downsample.1.weight"):
            prm.data.mul_(0.3)
    import hairfastgan_b200.bisenet as SEG
    seg = SEG.BiSeNet(n_classes=19).to(dev).eval()    # my_parsing_util.py:42
    for net in (e4e, fse, pp_enc, pp_res, seg):       # non-trivial BatchNorm statistics
        for m in net.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_var.uniform_(0.5, 1.5)
                m.running_mean.normal_(0, 0.1)
    bcast_bytes = 0
    if world > 1:                                     # weights replicated: one coalesced NCCL broadcast per net at init
        for net in (gen, e4e, fse, pp_enc, pp_res, seg):
            bcast_bytes += sharding.broadcast_module_(net, src=0)
    host = make_host_inputs(T, 100 + rank)
    devin = to_device(host, dev)
    host_out = torch.empty(T, 3, 1024, 1024).pin_memory()
    launches = [0]

    def compute(inp, skip_fse_recon=False, full_seg=False, outs=None):
        """The hot path of T triples through the public module API (what swap()'s stages call).  `outs`, if given,
        receives every network output of the step by name."""
        def keep(name, out):
            if outs is not None:
                outs[name] = out
            return out
        img, lats, lins, calls = inp["img"], inp["lat"], inp["lin"], inp["calls"]
        n0 = lib.hf_total_launch_count() + graphs.stats()["replayed_kernels"]   # eager launches + kernels inside replayed graphs
        for name, net, x in (("e4e_a", e4e, img[0]), ("e4e_b", e4e, img[1]), ("fse", fse, img[2])):   # Embedding.py:71,74 / :51
            keep(name, net(x))
        final = None
        for i, (s, e, b, r) in enumerate(calls):
            if i == 0 and skip_fse_recon:              # opt-in 8f-2 fast path: same RNG draws, no reconstruction
                gen.consume_noise(b)
                continue
            out = keep(f"gen{i}_{s}_{e}", gen([lats[i]], input_is_latent=True, start_layer=s, end_layer=e,
                                              layer_in=lins[i]))                                   # random noise
            if i == len(calls) - 1:
                final = out[0]
        _, (f_face,) = keep("pp_enc_face", pp_enc(img[3]))   # PostProcessModel.forward, models/Encoders.py:120-139
        _, (f_hair,) = keep("pp_enc_hair", pp_enc(img[4]))
        keep("pp_res", pp_res(torch.cat((f_face, f_hair), dim=1)))
        # get_segmentation x3 at 512^2 and twice at 1024^2 (models/Net.py:108-115).  Under install()'s defaults the
        # reference's FaceParsing_tensor.parsing_img runs the label-only path (parsing_fast.py: bit-identical labels,
        # aux heads + full-resolution logits not materialised); `full_seg=True` = the module's three-logit forward
        parse = seg if full_seg else seg.parse_labels
        keep("seg_512", parse(img[5]))
        keep("seg_1024_a", parse(img[6])); keep("seg_1024_b", parse(img[6]))
        launches[0] += lib.hf_total_launch_count() + graphs.stats()["replayed_kernels"] - n0
        return final

    def step(outs=None):
        return compute(devin, outs=outs)

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2

    def timed(steps: int, warmup: int, outs=None):
        for _ in range(warmup):
            step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        launches[0] = 0
        total_ms = 0.0
        for k in range(steps):
            flush.fill_(1)                                             # L2 flush between timed iterations
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step(outs if k == steps - 1 else None)
            e1.record()
            e1.synchronize()
            total_ms += e0.elapsed_time(e1)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        return sharding.max_over_ranks(total_ms, dev), launches[0]

    # ---- end to end: HOST inputs in, HOST images out, every step.  The way a caller would drive the public API:
    # uploads on one side stream, the result download on another, double-buffered, so that the copies of step k+1 / k-1
    # overlap the kernels of step k.  The timed region is ONE event pair around all K steps (L2 flushes included) and
    # ends only after the last download has finished.
    h2d_stream, d2h_stream = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    main_stream = torch.cuda.current_stream(dev)
    host_all = host["img"] + host["lat"] + [t for t in host["lin"] if t is not None]
    dbuf = [[torch.empty(t.shape, device=dev) for t in host_all] for _ in range(2)]
    hout = [host_out, torch.empty(T, 3, 1024, 1024).pin_memory()]
    ev_ready = [torch.cuda.Event() for _ in range(2)]
    ev_done = [torch.cuda.Event() for _ in range(2)]
    n_img, n_lat = len(host["img"]), len(host["lat"])

    def e2e_step(k: int):
        s = k & 1
        with torch.cuda.stream(h2d_stream):
            h2d_stream.wait_event(ev_done[s])          # step k-2 no longer reads this buffer set
            for d, h in zip(dbuf[s], host_all):
                d.copy_(h, non_blocking=True)
            ev_ready[s].record(h2d_stream)
        main_stream.wait_event(ev_ready[s])
        it = iter(dbuf[s][n_img + n_lat:])
        lins = [None if t is None else next(it) for t in host["lin"]]
        final = compute({"T": T, "calls": host["calls"], "img": dbuf[s][:n_img], "lat": dbuf[s][n_img:n_img + n_lat],
                         "lin": lins})
        ev_done[s].record(main_stream)
        final.record_stream(d2h_stream)
        with torch.cuda.stream(d2h_stream):
            d2h_stream.wait_event(ev_done[s])
            hout[s].copy_(final, non_blocking=True)

    def timed_e2e(steps: int, warmup: int):
        for k in range(warmup):
            e2e_step(k)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(main_stream)
        for k in range(steps):
            flush.fill_(1)
            e2e_step(k)
        main_stream.wait_stream(d2h_stream)            # the last image is on the host when the clock stops
        main_stream.wait_stream(h2d_stream)
        e1.record(main_stream)
        e1.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        return sharding.max_over_ranks(e0.elapsed_time(e1), dev)

    if args.profile_step:                             # for `ncu --profile-from-start off`: exactly one step
        os.environ["HAIRFAST_CUDA_GRAPHS"] = "0"       # eager launches only: a capture inside the window would list a forward twice
        step()
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStart()
        step()
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStop()
        return None

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(2):
        step()                                        # also gives nvidia-smi time to start sampling
    torch.cuda.synchronize()
    first = sampler.mark()
    outs = {} if args.dump_outputs and rank == 0 else None
    ms, n_launch = timed(args.steps, args.warmup, outs)
    if outs is not None:
        dump_outputs(outs, args.dump_outputs)
        del outs
    ms_e2e = timed_e2e(args.steps, max(3, args.warmup // 2))
    clocks = sampler.stop(first) if rank == 0 else None

    extra = {"nccl_broadcast_bytes_at_init": bcast_bytes}

    # ---- SURVEY 8d config 5: per-triple outputs of the N-GPU run must equal the 1-GPU run bit for bit.  After the
    # timed region every rank recomputes its step under swap()'s seed (utils/seed.py:22-28, 3407) and checksums each
    # triple's final image; rank 0 rebuilds every other rank's batch from its seed, computes it on ITS GPU under the same
    # seed, and compares the checksums gathered over NCCL.
    if world > 1:
        torch.manual_seed(3407)
        mine = image_checksums(compute(devin))
        gathered = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(gathered, mine)
        ok = True
        if rank == 0:
            for r in range(1, world):
                other = to_device(make_host_inputs(T, 100 + r), dev)
                torch.manual_seed(3407)
                ok = ok and bool(torch.equal(image_checksums(compute(other)), gathered[r]))
                del other
        flag = torch.tensor([int(ok)], device=dev)
        dist.broadcast(flag, src=0)
        extra["shard_output_equality"] = {"checked_ranks": world - 1, "triples_per_rank": T,
                                          "bit_identical_to_single_gpu": bool(flag.item())}
        if not bool(flag.item()):
            raise RuntimeError("N-GPU per-triple outputs differ from the single-GPU computation")

    def avg_ms(fn, n=5):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        tot = 0.0
        for _ in range(n):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record(); e1.synchronize()
            tot += e0.elapsed_time(e1)
        return tot / n

    if rank == 0 and world == 1:
        # single-triple latency: the census exactly as ONE swap() issues it (B = 3 / 2 / 1 per call, Appendix B)
        one = to_device(make_host_inputs(1, 7), dev)
        ms_t1 = avg_ms(lambda: compute(one), n=10)
        extra["latency_T1"] = {"latency_ms_per_triple": round(ms_t1, 3), "triples_per_s": round(1e3 / ms_t1, 2),
                               "note": "hot path of ONE triple, calls at B=3/2/1 as swap() issues them, HBM-resident"}
        del one
    if rank == 0 and world == 1 and args.no_extras:
        extra["roofline"] = roofline
        extra["roofline_b4"] = roofline_b4
    elif rank == 0 and world == 1:
        # opt-in SURVEY 8f-2 fast path (install(skip_fse_reconstruction=True)): the step without the FSE reconstruction
        # forward that swap() discards (445.6 GFLOP/triple), the noise still drawn
        ms_skip = avg_ms(lambda: compute(devin, skip_fse_recon=True))
        extra["fse_recon_skipped"] = {"value": round(T / (ms_skip * 1e-3), 3), "unit": "triples/s",
                                      "ms_per_step": round(ms_skip, 3),
                                      "note": "same outputs for swap(); not the default, see INTEGRATION.md"}
        ms_full = avg_ms(lambda: compute(devin, full_seg=True))
        extra["bisenet_full_logits_step"] = {"value": round(T / (ms_full * 1e-3), 3), "unit": "triples/s",
                                             "ms_per_step": round(ms_full, 3),
                                             "note": "the step with BiSeNet.forward's three [B,19,H,W] fp32 logit "
                                                     "outputs instead of the label-only path install() uses"}
        # configs[1]: full 1024^2 generator forward, B=4
        lat4 = torch.randn(4, 18, 512, device=dev)
        us_img = avg_ms(lambda: gen([lat4], input_is_latent=True)) / 4 * 1e3
        extra["generator_b4"] = {"img_per_s": round(1e6 / us_img, 1), "us_per_img": round(us_img, 1),
                                 "frac_of_roofline_142.5us": round(ROOFLINE_US_PER_IMG / us_img, 4),
                                 "tflops_algorithmic": round(GFLOP_FULL / us_img * 1e3, 1)}
        # configs[3]: e4e + FSE inversion, 256^2, batch 32
        x32 = torch.rand(32, 3, 256, 256, device=dev) * 2 - 1
        ms_e4e, ms_fse = avg_ms(lambda: e4e(x32)), avg_ms(lambda: fse(x32))
        extra["encoders_b32"] = {"e4e_img_per_s": round(32e3 / ms_e4e, 1), "fse_img_per_s": round(32e3 / ms_fse, 1),
                                 "e4e_tflops_algorithmic": round(32 * GFLOP_E4E_IMG / ms_e4e, 1),
                                 "fse_tflops_algorithmic": round(32 * GFLOP_FSE_IMG / ms_fse, 1)}
        # PostProcess conv stack at B=16 (SURVEY 8f-1)
        xr = torch.randn(16, 1024, 64, 64, device=dev)
        ms_ppe, ms_ppr = avg_ms(lambda: pp_enc(x32[:16])), avg_ms(lambda: pp_res(xr))
        extra["postprocess_b16"] = {"feature_encoder_mult_tflops_algorithmic": round(16 * GFLOP_PP_ENC_IMG / ms_ppe, 1),
                                    "feature_iresnet_tflops_algorithmic": round(16 * GFLOP_PP_RES / ms_ppr, 1),
                                    "feature_iresnet_ms": round(ms_ppr, 3)}
        del xr
        # BiSeNet at 512^2, B=16 (SURVEY 8f-3)
        xs = torch.rand(16, 3, 512, 512, device=dev) * 2 - 1
        ms_seg = avg_ms(lambda: seg(xs))
        ms_lab = avg_ms(lambda: seg.parse_labels(xs))
        extra["bisenet_b16_512"] = {"img_per_s": round(16e3 / ms_seg, 1),
                                    "tflops_algorithmic": round(16 * GFLOP_SEG_512 / ms_seg, 1),
                                    "labels_only_img_per_s": round(16e3 / ms_lab, 1),
                                    "labels_only_tflops_algorithmic": round(16 * GFLOP_SEG_512 / ms_lab, 1),
                                    "note": "forward = three fp32 logit maps; labels_only = BiSeNet.parse_labels, the "
                                            "path face parsing takes under install() (same labels; FLOPs counted in "
                                            "the reference's three-head formulation)"}
        del xs
        # SURVEY 8d metric (3): the standalone HBM-bound operators (module-level API a6 / a7), GB/s = (in + out) / time
        import hairfastgan_b200.op as OP
        hbm = peaks()["hbm_gbs"]
        xa = torch.randn(4, 64, 1024, 1024, device=dev); ba = torch.randn(64, device=dev)
        ms_a = avg_ms(lambda: OP.fused_leaky_relu(xa, ba))
        kern = torch.tensor([1., 3., 3., 1.], device=dev)
        k2 = kern[None, :] * kern[:, None]; k2 = k2 / k2.sum()
        xu = torch.randn(1, 256, 1025, 1025, device=dev)
        ms_u1 = avg_ms(lambda: OP.upfirdn2d(xu, k2 * 4, pad=(1, 1)))
        xs3 = torch.randn(48, 3, 512, 512, device=dev)
        ms_u2 = avg_ms(lambda: OP.upfirdn2d(xs3, k2 * 4, up=2, pad=(2, 1)))
        xd = torch.randn(64, 3, 1024, 1024, device=dev)
        ms_d2 = avg_ms(lambda: OP.upfirdn2d(xd, k2, down=2, pad=(1, 1)))
        gbs = {"fused_leaky_relu_4x64x1024x1024": 2 * xa.numel() * 4 / ms_a / 1e6,
               "upfirdn2d_up1_k4_pad11_256x1025x1025": (xu.numel() + 256 * 1024 * 1024) * 4 / ms_u1 / 1e6,
               "upfirdn2d_up2_k4_pad21_144x512x512": (xs3.numel() * 5) * 4 / ms_u2 / 1e6,
               "upfirdn2d_down2_k4_pad11_192x1024x1024": (xd.numel() * 1.25) * 4 / ms_d2 / 1e6}
        extra["ops_hbm"] = {k: {"GB/s": round(v, 1), "frac_of_measured_copy_peak": round(v / hbm, 3)}
                            for k, v in gbs.items()}
        del xa, xu, xs3, xd
        extra["roofline"] = roofline
        extra["roofline_b4"] = roofline_b4
    if world > 1:
        dist.destroy_process_group()
    h2d = sum(t.numel() * 4 for t in host["lat"]) + sum(t.numel() * 4 for t in host["lin"] if t is not None) \
        + sum(t.numel() * 4 for t in host["img"])
    return ms, ms_e2e, n_launch, clocks, extra, h2d


DUMP_BYTES = 64 << 20


def dump_outputs(outs, path):
    """Write every tensor in `outs` (name -> tensor or nested tuple / list; None entries skipped) as
    path/<name>[.<index>...].npy in float32.  A tensor larger than its even share of DUMP_BYTES is written as a fixed
    sample of its flattened elements (indices drawn from a generator seeded by the name, sorted), so that two builds
    run with the same arguments write files that compare element for element."""
    import zlib
    import numpy as np
    import torch
    leaves = []

    def walk(name, v):
        if torch.is_tensor(v):
            leaves.append((name, v))
        elif isinstance(v, (list, tuple)):
            for j, u in enumerate(v):
                walk(f"{name}.{j}", u)
    for name, v in outs.items():
        walk(name, v)
    share = (DUMP_BYTES - 4096 * len(leaves)) // (4 * len(leaves))      # 4096: room for each .npy header
    os.makedirs(path, exist_ok=True)
    for name, t in leaves:
        t = t.detach()
        if t.numel() > share:
            g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
            idx = torch.randint(t.numel(), (share,), generator=g).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.float().cpu().numpy())


def _json_tail(stdout: str):
    for line in reversed(stdout.splitlines()):
        line = line.strip()
        if line.startswith("{"):
            return json.loads(line)
    raise RuntimeError("no JSON line in: " + stdout[-500:])


def comparator_legs(args):
    """Side measurements that need OTHER processes (the GPU is free: our own run has finished): the stock reference on
    the same B200 (`reference_gpu`), the full HairFast.swap() under the overlay vs the stock one (`full_swap`), and our
    own step with every network in bf16 / fp16 (`value_by_dtype`).  Each is a bounded child run; a failure is reported
    in the line, never hidden."""
    from baseline import refenv
    out = {}
    env = dict(os.environ)
    env.pop("OMP_NUM_THREADS", None)

    def child(cmd, timeout, extra_env=None):
        e = dict(env)
        e.update(extra_env or {})
        p = subprocess.run(cmd, capture_output=True, text=True, env=e, timeout=timeout, cwd=ROOT)
        if p.returncode != 0:
            raise RuntimeError(p.stderr[-600:])
        return _json_tail(p.stdout)

    by_dtype = {}
    for dt in ("bf16", "fp16"):
        try:
            d = child([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "5", "--warmup", "3", "--triples",
                       str(args.triples), "--no-extras", "--no-cpu-baseline", "--no-comparators"], 900,
                      {"HAIRFAST_DTYPE": dt, "HAIRFAST_ENC_DTYPE": dt})
            by_dtype[dt] = {"value": d["value"], "e2e": d["e2e"]["value"], "latency_T1_ms": d["latency_T1"]["latency_ms_per_triple"]}
        except Exception as ex:   # noqa: BLE001
            by_dtype[dt] = {"error": str(ex)[-300:]}
    out["value_by_dtype"] = {"unit": "triples/s", "note": "every network in that operand type (HAIRFAST_DTYPE=...)",
                             **by_dtype}
    if not refenv.available():
        out["reference_gpu"] = {"unavailable": "reference checkout not staged (tools/stage_reference.sh)"}
        out["full_swap"] = {"unavailable": "reference checkout not staged (tools/stage_reference.sh)"}
        return out
    census_py = os.path.join(ROOT, "baseline", "ref_census.py")
    ref = {}
    # T = 1 (latency) and the largest batching the stock modules survive: at T = 32 (B = 96 in the full forwards) the
    # reference dies with a CUDA error inside its own kernels (index overflow past 2^31 elements), so the sweep walks
    # down from our T until a census completes
    t_try = [1] + [t for t in (args.triples, 16, 8) if t > 1]
    done_big = False
    for T in dict.fromkeys(t_try):
        if T > 1 and done_big:
            break
        try:
            d = child([sys.executable, census_py, "--device", "cuda", "--triples", str(T), "--steps", "3", "--warmup",
                       "2"], 1500)
            ref[f"T{T}"] = {"triples_per_s": round(d["triples_per_s"], 3), "ms_per_step": round(d["ms_per_step"], 2),
                            "peak_mem_gb": d["peak_mem_gb"]}
            ref["arith"] = d["arith"]
            done_big = done_big or T > 1
        except Exception as ex:   # noqa: BLE001
            msg = str(ex)
            ref[f"T{T}"] = {"error": ("CUDA error inside the stock reference at this batch: " if "CUDA" in msg else "")
                            + msg.strip().splitlines()[-1][-160:] if msg.strip() else "failed"}
    ref["what"] = ("the SAME census on the stock reference modules on this B200: F.conv2d(groups=B)/conv_transpose2d "
                   "through cuDNN + its two JIT kernels (models/stylegan2/model.py:238-279), baseline/ref_census.py")
    out["reference_gpu"] = ref
    swap = {}
    work = os.environ.get("HAIRFAST_WORK", "/tmp/hairfast_work")
    for mode in ("reference", "overlay", "overlay_fast"):
        try:
            d = child([sys.executable, os.path.join(ROOT, "baseline", "run_swap.py"), "--mode", mode, "--work", work,
                       "--reps", "7", "--warmup", "3"], 1500)
            ts = d["timings"]

            def med(vals):
                v = sorted(vals)
                return v[len(v) // 2]
            swap[mode] = {"full_swap_ms": round(med([t["gpu_ms"] for t in ts]), 2),
                          "hot_path_ms": round(med([t["hot_path_ms"] for t in ts]), 2),
                          "out_of_scope_ms": round(med([t["out_of_scope_ms"] for t in ts]), 2),
                          "per_module_ms": {k: round(med([t["per_module_ms"].get(k, 0.0) for t in ts]), 2)
                                            for k in ts[-1]["per_module_ms"]},
                          "full_swap_ms_all_reps": [round(t["gpu_ms"], 1) for t in ts], "stat": "median of the reps",
                          "dtype": d["dtype"], "deterministic": d["deterministic"]}
        except Exception as ex:   # noqa: BLE001
            swap[mode] = {"error": str(ex)[-300:]}
    swap["what"] = ("BASELINE configs[2]: the unmodified HairFast(get_parser().parse_args([])).swap() on one synthetic "
                    "1024^2 triple, synthetic checkpoints (baseline/run_swap.py): stock reference vs the same checkout "
                    "under hairfastgan_b200.install(); hot path = generator + e4e + FS encoder + PostProcess conv "
                    "stack + BiSeNet (forward hooks, CUDA events); out of scope = SEAN, CLIP stand-in, mask nets, glue")
    out["full_swap"] = swap
    return out


def time_dominant_kernel(gen, dev, B=4):
    """The 512->512 3x3 @64^2 convolution (BASELINE configs[0] shape), the layer class that carries most of the
    tensor-core time, at batch B (the step runs it at B = 3T and T; configs[1] is B = 4).  Algorithmic FLOPs =
    2*512*512*9*64^2 per sample (SURVEY 8d)."""
    import ctypes as C
    import torch
    from hairfastgan_b200 import _lib
    import hairfastgan_b200.model as M
    lib = _lib.lib()
    conv = gen.convs[7].conv                       # convs.7 = 512->512 @64^2
    desc, blob = conv._packed.get(conv, M.default_dtype())
    x = torch.randn(B, 512, 64, 64, device=dev); st = torch.randn(B, 512, device=dev)
    y = torch.empty(B, 512, 64, 64, device=dev)
    ws = torch.empty(lib.hf_conv_workspace_bytes(C.byref(desc), B, 64, 64), dtype=torch.uint8, device=dev)
    io = _lib.hf_conv_io()
    io.batch, io.height, io.width = B, 64, 64
    io.x, io.style, io.style_dim, io.style_stride = x.data_ptr(), st.data_ptr(), 512, 512
    mw, mb = conv.modulation.weight.data, conv.modulation.bias.data
    io.mod_weight, io.mod_bias, io.demodulate = mw.data_ptr(), mb.data_ptr(), 1
    io.y, io.workspace = y.data_ptr(), ws.data_ptr()
    ms = C.c_float(0)
    _lib.check(lib.hf_conv_time_kernel(C.byref(desc), blob.data_ptr(), C.byref(io), 20, C.byref(ms),
                                       torch.cuda.current_stream().cuda_stream), "hf_conv_time_kernel")
    plan = (C.c_int * 12)()
    lib.hf_conv_plan_query(C.byref(desc), B, 64, 64, plan)
    kname = {0: "conv_igemm_kernel", 1: "conv_halo_kernel", 2: "conv_halo2_kernel (cta_group::2)"}[plan[0]]
    flops = 2.0 * 512 * 512 * 9 * 64 * 64 * B
    achieved = flops / (ms.value * 1e-3) / 1e12
    pk = peaks()
    traffic = None
    for tp in (f"ncu_dominant_kernel_r2_b{B}.json", "ncu_dominant_kernel_r1.json" if B == 4 else
               f"ncu_dominant_kernel_r1_b{B}.json"):                 # one `ncu --set full` capture per batch size
        tp = os.path.join(ROOT, "profiles", tp)
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get("dram_bytes_per_launch")
            break
    return {"kernel": f"{kname}<bf16> 512->512 3x3 @64^2 B={B} (+fp32 NCHW store)", "bound": "tensor",
            "achieved": round(achieved, 1), "peak": pk["tf_burst"], "unit": "TFLOP/s",
            "frac": round(achieved / pk["tf_burst"], 4), "peak_source": pk["src"] + " burst (kernel timed alone)",
            "launch_ms": round(ms.value, 4), "traffic": traffic}


CENSUS_COUNTS = {"gen_full": 5, "gen_0_3": 5, "gen_3_3": 3, "gen_4_8": 1, "gen_5_8": 1, "e4e": 5, "fse": 3,
                 "pp_enc": 2, "pp_res": 1, "seg_512": 3, "seg_1024": 2}          # SURVEY Appendix B, per triple
CPU_SAMPLE = ("every distinct call of the SURVEY App. B census once at B=1 (generator full / 0->3 / 3->3 / 4->8 / 5->8, "
              "e4e, FSE, FeatureEncoderMult, FeatureiResnet, BiSeNet 512^2 and 1024^2); per-triple time = "
              "sum(count x time) = the whole census, nothing FLOP-scaled")


def cpu_threads():
    """Physical host cores, stated.  torchrun exports OMP_NUM_THREADS=1 to its workers (round 1: 64 threads at N=1, one
    thread under torchrun -> a 4.5x swing of the denominator), and os.cpu_count() counts hyper-threads (128 on the B200
    hosts: measured 40x SLOWER than 64 threads on these B=1 convolutions), so neither is inherited silently."""
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
    except Exception:   # noqa: BLE001
        n = None
    n = n or os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except AttributeError:
        pass
    return max(1, n)


def cpu_census_reference(steps: int, warmup: int):
    """The STOCK reference modules (staged checkout, baseline/_ref) on the host cores: baseline/ref_census.py."""
    env = dict(os.environ)
    env.pop("OMP_NUM_THREADS", None)
    cmd = [sys.executable, os.path.join(ROOT, "baseline", "ref_census.py"), "--device", "cpu", "--steps", str(steps),
           "--warmup", str(warmup), "--threads", str(cpu_threads())]
    p = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=3000)
    if p.returncode != 0:
        raise RuntimeError("ref_census.py failed: " + p.stderr[-2000:])
    d = json.loads([l for l in p.stdout.splitlines() if l.strip()][-1])
    return d["s_per_triple"], d["cores"], "reference", d["per_call_s"]


def cpu_census_port(steps: int, warmup: int):
    """Same census on the oracle port (used only when the reference checkout is not staged)."""
    import torch
    from oracle import stylegan2_oracle as O
    from oracle import encoders_oracle as EO
    from oracle import bisenet_oracle as BO
    import hairfastgan_b200.encoders as E          # parameter containers only (CPU); the math below is the oracle's
    import hairfastgan_b200.postprocess as PP
    import hairfastgan_b200.bisenet as SEG
    torch.set_grad_enabled(False)
    torch.set_num_threads(cpu_threads())
    g = torch.Generator().manual_seed(0)
    p = O.synth_generator_params(size=1024, seed=0)
    lat = torch.randn(1, 18, 512, generator=g)
    noise = O.synth_noise(1024, batch=1, seed=1)
    li = {r: torch.randn(1, 512, r, r, generator=g) for r in (16, 32, 64)}
    pe = EO.synth_params_like(E.Encoder4Editing(50, "ir_se", types.SimpleNamespace(stylegan_size=1024)), 11)
    pf = EO.synth_params_like(E.fs_encoder_v2(n_styles=18, opts=None, stride=(2, 2)), 21)
    pm = EO.synth_params_like(PP.FeatureEncoderMult(fs_layers=[9], opts=None), 31)
    pr = EO.synth_params_like(PP.FeatureiResnet([[1024, 2], [768, 2], [512, 2]]), 41)
    ps = EO.synth_params_like(SEG.BiSeNet(n_classes=19), 51)
    x = torch.rand(1, 3, 256, 256, generator=g) * 2 - 1
    xr = torch.randn(1, 1024, 64, 64, generator=g)
    x512, x1024 = torch.rand(1, 3, 512, 512, generator=g) * 2 - 1, torch.rand(1, 3, 1024, 1024, generator=g) * 2 - 1
    calls = {"gen_full": lambda: O.generator_ref(p, lat, noise), "gen_0_3": lambda: O.generator_ref(p, lat, noise, 0, 3),
             "gen_3_3": lambda: O.generator_ref(p, lat, noise, 3, 3, li[16]),
             "gen_4_8": lambda: O.generator_ref(p, lat, noise, 4, 8, li[32]),
             "gen_5_8": lambda: O.generator_ref(p, lat, noise, 5, 8, li[64]),
             "e4e": lambda: EO.e4e_ref(pe, x), "fse": lambda: EO.fse_ref(pf, x),
             "pp_enc": lambda: EO.feature_encoder_mult_ref(pm, x), "pp_res": lambda: EO.feature_iresnet_ref(pr, xr),
             "seg_512": lambda: BO.bisenet_ref(ps, x512), "seg_1024": lambda: BO.bisenet_ref(ps, x1024)}
    tot, last = [], {}
    for it in range(warmup + steps):
        t = 0.0
        for name, fn in calls.items():
            t0 = time.perf_counter()
            fn()
            dt = time.perf_counter() - t0
            last[name] = round(dt, 4)
            t += CENSUS_COUNTS[name] * dt
        if it >= warmup:
            tot.append(t)
    return sum(tot) / len(tot), torch.get_num_threads(), "port", last


def cpu_census(steps: int = 1, warmup: int = 0):
    """(seconds per triple, threads, kind, per-call seconds) of the hot-path census on the host cores."""
    from baseline import refenv
    if refenv.available() and os.environ.get("HAIRFAST_CPU_ARM", "reference") != "port":
        return cpu_census_reference(steps, warmup)
    return cpu_census_port(steps, warmup)


WORKLOAD = ""


def dtype_string():
    gen = os.environ.get("HAIRFAST_DTYPE", "bf16")
    enc = os.environ.get("HAIRFAST_ENC_DTYPE") or os.environ.get("HAIRFAST_DTYPE", "fp16")
    return f"generator {gen} / encoders {enc} operands, f32 accumulate"


def config_of(T: int, world: int):
    """`config` of the JSON line -- identical for our arm and the reference arm (the driver compares them)."""
    return {"workload": WORKLOAD, "triples_per_step_per_gpu": T, "size": 1024,
            "parallelism": f"dp{world} (independent triples per rank, no step collective)",
            "l2": "256 MiB flush write between timed steps; value: per-step CUDA events summed; e2e: one event "
                  "pair around all steps, uploads/downloads double-buffered on side streams"}


_REAL_STDOUT = None


def _quiet_stdout():
    """The contract is ONE JSON line on stdout.  Libraries (NCCL's version banner, ...) write to fd 1 from C, so
    point fd 1 at stderr for the whole run and keep the real stdout for the final line."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(obj):
    sys.stdout.flush()
    _REAL_STDOUT.write(json.dumps(obj) + "\n")
    _REAL_STDOUT.flush()


def main():
    _quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--triples", type=int, default=32, help="independent triples batched per step and GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the per-network / per-operator side measurements")
    ap.add_argument("--profile-step", action="store_true", help="run one step between cudaProfilerStart/Stop, no JSON")
    ap.add_argument("--no-comparators", action="store_true",
                    help="skip the child-process legs (reference_gpu, full_swap, value_by_dtype)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the network outputs of the last timed step as DIR/<name>.npy (float32, 64 MB in all: "
                         "larger outputs as a fixed seeded sample); same arguments, same inputs")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    workload = ("SURVEY-8 hot path of HairFast.swap(): 8 Generator.forward calls (1024^2, randomize_noise=True) + "
                "e4e on 5 and FSE on 3 images (256^2) + PostProcess conv stack (FeatureEncoderMult x2, FeatureiResnet "
                "@64^2) + BiSeNet face parsing (labels, as install() runs it) on 3 images at 512^2 and 2 at 1024^2 "
                "per triple = 3063.8 GFLOP/triple in the reference's formulation (SURVEY App. B / 8d config 3 / 8f-3), "
                "synthetic weights; out-of-scope nets (SEAN/CLIP/mask) and stage glue "
                "excluded")
    global WORKLOAD
    WORKLOAD = workload

    if args.impl == "reference":
        if rank != 0:
            return
        s_per_triple, thr, kind, per_call = cpu_census(args.steps, args.warmup)
        val = 1.0 / s_per_triple
        emit(({
            "impl": "reference", "metric": "hair_swap_triples_per_sec", "value": val, "unit": "triples/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": s_per_triple * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_of(args.triples, world),
            "cpu_baseline": {"value": val, "unit": "triples/s", "cores": thr, "kind": kind, "sample": CPU_SAMPLE,
                             "per_call_s": per_call},
            "e2e": {"value": val, "unit": "triples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}))
        return

    res = run_ours(args, rank, world, local_rank)
    if res is None:
        return
    ms, ms_e2e, n_launch, clocks, extra, h2d = res
    if rank != 0:
        return
    T = args.triples
    step_ms = ms / args.steps
    value = world * T / (step_ms * 1e-3)
    e2e_value = world * T / (ms_e2e / args.steps * 1e-3)
    out = {
        "metric": "hair_swap_triples_per_sec", "value": round(value, 3), "unit": "triples/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(step_ms, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None,
        "dtype": dtype_string(), "data": "synthetic",
        "config": config_of(T, world),
        "tflops_algorithmic": round(GFLOP_PER_TRIPLE * value / 1e3, 1),
        # whole-step fraction of the conv roofline: algorithmic FLOP/s over all GPUs / (N x measured bf16 peak)
        "frac_of_tensor_peak": round(GFLOP_PER_TRIPLE * value / 1e3 / (world * peaks()["tf_burst"]), 4),
        "e2e": {"value": round(e2e_value, 3), "unit": "triples/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": T * 3 * 1024 * 1024 * 4},
        "gpu_launches": n_launch, "clocks": clocks,
    }
    out.update(extra)
    if world == 1 and not args.no_extras and not args.no_comparators:
        out.update(comparator_legs(args))
    if world == 1 and not args.no_cpu_baseline:
        s_per_triple, thr, kind, per_call = cpu_census(1, 0)
        out["cpu_baseline"] = {"value": round(1.0 / s_per_triple, 5), "unit": "triples/s", "cores": thr, "kind": kind,
                               "sample": f"{s_per_triple:.1f} s per triple: " + CPU_SAMPLE, "per_call_s": per_call}
    emit(out)


if __name__ == "__main__":
    main()
