"""One process = one arm of the full `HairFast.swap()` comparison (BASELINE configs[2], SURVEY 8d config 3).

    python baseline/run_swap.py --mode reference|overlay|overlay_fast --work DIR --out result.pt [--reps N]

* reference     the staged, unmodified checkout: cuDNN grouped convolutions + its two JIT kernels, fp32/TF32
* overlay       the same checkout with hairfastgan_b200.install() active (this package's modules under its names)
* overlay_fast  overlay + install(skip_fse_reconstruction=True) (hairfastgan_b200/fse_fast.py)

Three synthetic images `torch.rand(3,1024,1024)` (seeds 0,1,2) are passed as tensors (hair_swap.py:63-105), synthetic
checkpoints come from baseline/synth_checkpoints.py, `swap(..., seed=3407)` is the default seed (utils/seed.py:22-28).
The result file holds the final image of every repetition, the Embedding-stage latents of the last one and the wall /
CUDA-event timings: whole swap, and the share spent inside the hot-path modules (generator, e4e, FS encoder,
PostProcess conv stack, BiSeNet) measured with forward hooks -- the hot-path / out-of-scope split of SURVEY 8d.
Harness (run by hand; bench.py's full-swap leg); not product code.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from baseline import refenv, synth_checkpoints  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", choices=["reference", "overlay", "overlay_fast"], required=True)
    ap.add_argument("--work", default="/tmp/hairfast_work")
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--seed", type=int, default=None)
    ap.add_argument("--same_shape_color", action="store_true", help="shape image is the color image (hair_swap.py:54)")
    a = ap.parse_args()
    work = os.path.abspath(a.work)

    if not os.path.exists(os.path.join(work, "pretrained_models", ".complete_seed0")):
        # the writer needs the STOCK classes: do it in a child so this process keeps a single mode
        import subprocess
        subprocess.run([sys.executable, os.path.join(HERE, "synth_checkpoints.py"), work], check=True)

    refenv.activate(overlay=a.mode != "reference", skip_fse_reconstruction=a.mode == "overlay_fast", workdir=work)
    import torch
    assert torch.cuda.is_available(), "run_swap.py needs a GPU (tools/dryrun_swap_cpu.py is the CPU dry run)"
    from hair_swap import HairFast, get_parser      # the reference's own hair_swap.py

    t0 = time.time()
    hair_fast = HairFast(get_parser().parse_args([]))
    torch.cuda.synchronize()
    init_s = time.time() - t0

    # ---- hot-path accounting: CUDA events around the forward of every in-scope module ----------------------------
    from models.CtrlHair.external_code.face_parsing.my_parsing_util import FaceParsing
    hot = {
        "generator": hair_fast.net.generator,
        "fse_generator": hair_fast.embed.encoder.StyleGAN,
        "e4e": hair_fast.embed.e4e.encoder,
        "fse_encoder": hair_fast.embed.encoder.enc,
        "pp_encoder": hair_fast.blend.post_process.encoder_face,
        "pp_to_feature": hair_fast.blend.post_process.to_feature,
        "bisenet": FaceParsing.bise_net,
    }
    spans = []

    def pre(name):
        def hook(m, inp):
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            spans.append([name, ev, None])
        return hook

    def post(m, inp, out):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        for s in reversed(spans):
            if s[2] is None:
                s[2] = ev
                break
    for name, mod in hot.items():
        mod.register_forward_pre_hook(pre(name))
        mod.register_forward_hook(post)
    seg = FaceParsing.bise_net
    if hasattr(seg, "parse_labels"):                 # the label-only path bypasses Module.__call__ (parsing_fast.py)
        orig_parse = seg.parse_labels

        def timed_parse(x):
            pre("bisenet")(seg, None)
            out = orig_parse(x)
            post(seg, None, None)
            return out
        seg.parse_labels = timed_parse

    imgs = [torch.rand(3, 1024, 1024, generator=torch.Generator().manual_seed(s)) for s in range(3)]
    if a.same_shape_color:
        imgs[2] = imgs[1]
    kw = {} if a.seed is None else {"seed": a.seed}

    # capture the Embedding-stage outputs of the last repetition (models/Embedding.py:93-101)
    captured = {}
    orig_embed = hair_fast.embed.embedding_images

    def embedding_images(*args, **kwargs):
        res = orig_embed(*args, **kwargs)
        captured.clear()
        for name, d in res.items():
            for k, v in d.items():
                captured[f"{name}.{k}"] = v.detach().float().cpu() if v.is_floating_point() else v.detach().cpu()
        return res
    hair_fast.embed.embedding_images = embedding_images

    # optional stage trace (HF_SWAP_TRACE=1): wall time of every stage call, gc collections and graph statistics per rep
    trace = os.environ.get("HF_SWAP_TRACE") in ("1", "2")           # 2: wall clock only, no synchronize
    trace_sync = os.environ.get("HF_SWAP_TRACE") == "1"
    stage_ms = {}
    if trace:
        import gc

        def wrap(obj, name, label):
            orig = getattr(obj, name)

            def timed(*args, **kwargs):
                if trace_sync:
                    torch.cuda.synchronize()
                t0 = time.time()
                out = orig(*args, **kwargs)
                if trace_sync:
                    torch.cuda.synchronize()
                stage_ms[label] = stage_ms.get(label, 0.0) + (time.time() - t0) * 1e3
                return out
            setattr(obj, name, timed)
        wrap(hair_fast.embed, "embedding_images", "embed")
        wrap(hair_fast.align, "align_images", "align")
        wrap(hair_fast.align, "shape_module", "shape_module(incl. in align)")
        wrap(hair_fast.blend, "blend_images", "blend")
    finals, timings = [], []
    for rep in range(a.warmup + a.reps):
        if trace:
            stage_ms.clear()
            gc0 = [g["collections"] for g in gc.get_stats()]
        spans.clear()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.time()
        e0.record()
        final = hair_fast.swap(*imgs, **kw)
        e1.record()
        torch.cuda.synchronize()
        wall = (time.time() - w0) * 1e3
        per = {}
        for name, s, e in spans:
            per[name] = per.get(name, 0.0) + s.elapsed_time(e)
        hot_ms = sum(per.values())
        if trace:
            line = {"rep": rep, "wall_ms": round(wall, 1), "gpu_ms": round(e0.elapsed_time(e1), 1), "stages": {k: round(v, 1) for k, v in stage_ms.items()},
                    "gc": [g["collections"] - c for g, c in zip(gc.get_stats(), gc0)]}
            try:
                from hairfastgan_b200 import graphs as _g
                line["graphs"] = _g.stats()
            except Exception:   # noqa: BLE001
                pass
            print("TRACE " + json.dumps(line), file=sys.stderr, flush=True)
        if rep >= a.warmup:
            finals.append(final.detach().float().cpu())
            timings.append({"wall_ms": wall, "gpu_ms": e0.elapsed_time(e1), "hot_path_ms": hot_ms,
                            "out_of_scope_ms": e0.elapsed_time(e1) - hot_ms, "per_module_ms": per,
                            "hot_calls": len(spans)})
    summary = {"mode": a.mode, "init_s": init_s, "timings": timings,
               "final_shape": list(finals[-1].shape), "final_min": float(finals[-1].min()),
               "final_max": float(finals[-1].max()), "finite": bool(torch.isfinite(finals[-1]).all()),
               "deterministic": bool(all(torch.equal(finals[0], f) for f in finals[1:])),
               "device": torch.cuda.get_device_name(0),
               "dtype": ("fp32/tf32" if a.mode == "reference" else
                         "generator %s, encoders %s" % (os.environ.get("HAIRFAST_DTYPE", "bf16"),
                                                        os.environ.get("HAIRFAST_ENC_DTYPE") or
                                                        os.environ.get("HAIRFAST_DTYPE", "fp16"))),
               "generator_class": type(hair_fast.net.generator).__module__,
               "cuda_alloc_retries": int(torch.cuda.memory_stats().get("num_alloc_retries", 0)),
               "cuda_reserved_gb": round(torch.cuda.memory_reserved() / 2 ** 30, 2),
               "cuda_peak_allocated_gb": round(torch.cuda.max_memory_allocated() / 2 ** 30, 2)}
    print(json.dumps(summary))
    if a.out:
        torch.save({"finals": finals, "embed": dict(captured), "summary": summary}, a.out)


if __name__ == "__main__":
    main()
