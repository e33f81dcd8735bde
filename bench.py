#!/usr/bin/env python
"""Benchmark of the HIPIE inference hot path on B200 (contract: see the task statement / DESIGN.md §6).

  python bench.py --gpus N --steps K --warmup W [--config C]          # product arm (one process per GPU under torchrun for N>1)
  python bench.py --impl reference --gpus N --steps K ... [--config C]  # reference arm: the CPU oracle of the same path, rank 0 only
  python bench.py ... --dump-outputs DIR                                # product arm, plus the last timed step's outputs as DIR/*.npy

Workloads (BASELINE.json `configs`, SURVEY.md §8d; per-GPU shards of the image-sharded global batches):
  --config 1 (default, the configuration the metric is quoted on)  ViT-H, 8 x 1024x1024, 80-class COCO vocabulary (Lt = 512), detection
  --config 2   ViT-H, 8 x 1024x1024 per GPU (64 over 8 GPUs), 150-class ADE vocabulary, Lt = 4096, max-pooled / class-agnostic-bg scoring
  --config 3   ViT-H, 4 x 1280x1280 per GPU (16 over 4 GPUs), one referring expression per image (task grounding), Lt = 512
  --config 4   ViT-H, 4 x 1024x1024 per GPU (32 over 8 GPUs), 847-class ADE vocabulary, Lt = 4096 (> 512 tokens: chunked BERT)
Synthetic images, random-init weights of that architecture, synthetic token ids.

A step = one pass of the hot path (preprocess -> ViT-H -> BERT -> VL fusion -> deformable encoder/decoder -> MaskDINO pixel
decoder/decoder + mask-embed contraction -> CondInst masks; SURVEY §8a rows a1-a19) over the per-GPU batch with inputs resident
in HBM.  `e2e` times the public API call (HIPIE_IMG.forward incl. post-processing, rows a20-a23) from pinned host images, H2D and
D2H inside the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "images/sec at 1024x1024, ViT-H HIPIE inference hot path (synthetic batch)"

CONFIGS = {
    1: dict(name="configs[1]", img=1024, batch=8, classes=80, lt=512, task="detection", max_pool=False, bg_agnostic=False,
            vit_flops=7.41e12, desc="ViT-H, batch 8 x 1024x1024 synthetic per GPU, 80-class COCO-style vocab (Lt=512), task detection"),
    2: dict(name="configs[2]", img=1024, batch=8, classes=150, lt=4096, task="detection", max_pool=True, bg_agnostic=True,
            vit_flops=7.41e12, desc="ViT-H, batch 8 x 1024x1024 synthetic per GPU (64 over 8 GPUs), 150-class ADE vocab (Lt=4096), task detection"),
    3: dict(name="configs[3]", img=1280, batch=4, classes=1, lt=512, task="grounding", max_pool=False, bg_agnostic=False,
            vit_flops=13.33e12, desc="ViT-H, batch 4 x 1280x1280 synthetic per GPU (16 over 4 GPUs), one referring expression per image, task grounding"),
    4: dict(name="configs[4]", img=1024, batch=4, classes=847, lt=4096, task="detection", max_pool=True, bg_agnostic=True,
            vit_flops=7.41e12, desc="ViT-H, batch 4 x 1024x1024 synthetic per GPU (32 over 8 GPUs), 847-class ADE vocab (Lt=4096, chunked BERT), task detection"),
}


def vit_h_hp(cfg):
    bert = dict(vocab=30522, hidden=768, layers=12, heads=12, inter=3072, max_pos=512)
    return dict(backbone="vit",
                vit=dict(embed_dim=1280, depth=32, num_heads=16, window_size=14, window_block_indexes=(0, 1, 3, 4, 6, 7, 9, 10),
                         img_size=1024, patch_size=16, pretrain_img_size=224),
                hidden_dim=256, enc_layers=6, dec_layers=6, dim_ff=2048, num_queries=900, num_bg=10, vl_hidden=2048, lang_dim=768,
                md_queries=300, md_dec_layers=9, md_enc_layers=6, md_dim_ff=2048, bert=bert, max_query_len=cfg["lt"],
                max_pool=cfg["max_pool"], bg_cls_agnostic=cfg["bg_agnostic"])


def synth_text(num_classes, max_len, seed=0):
    """[CLS] + per-class 1-3 random word-piece ids joined by '.' (1012) + [SEP], zero padded (SURVEY §8d)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    ids, pos_map = [101], {}
    for c in range(1, num_classes + 1):
        n = int(torch.randint(1, 4, (1,), generator=g))
        if len(ids) + n + 2 > max_len:
            n = 1
        toks = torch.randint(1996, 30000, (n,), generator=g).tolist()
        pos_map[c] = list(range(len(ids), len(ids) + n))
        ids += toks + [1012]
    ids.append(102)
    assert len(ids) <= max_len
    input_ids = torch.zeros(max_len, dtype=torch.long)
    input_ids[:len(ids)] = torch.tensor(ids)
    attn = torch.zeros(max_len, dtype=torch.long)
    attn[:len(ids)] = 1
    n_thing = -(-num_classes * 6 // 10)
    return input_ids, attn, pos_map, {c: c <= n_thing for c in range(1, num_classes + 1)}


def synth_expression(max_len, seed):
    """a referring expression of 5-12 random word pieces: [CLS] w1 .. wn [SEP]"""
    import torch
    g = torch.Generator().manual_seed(seed)
    n = int(torch.randint(5, 13, (1,), generator=g))
    ids = [101] + torch.randint(1996, 30000, (n,), generator=g).tolist() + [102]
    input_ids = torch.zeros(max_len, dtype=torch.long)
    input_ids[:len(ids)] = torch.tensor(ids)
    attn = torch.zeros(max_len, dtype=torch.long)
    attn[:len(ids)] = 1
    return input_ids, attn


def batch_text(cfg, B, seed_base=0):
    """-> ids (B, Lt), am (B, Lt), positive map, is_thing.  Detection: one vocabulary prompt for the whole batch; grounding: a
    different expression per image (the text encoder really runs on B rows)."""
    import torch
    if cfg["task"] == "grounding":
        rows = [synth_expression(cfg["lt"], seed_base + b) for b in range(B)]
        return torch.stack([r[0] for r in rows]), torch.stack([r[1] for r in rows]), {1: [0]}, {1: True}
    ids, am, pos_map, is_thing = synth_text(cfg["classes"], cfg["lt"])
    return ids.unsqueeze(0).repeat(B, 1), am.unsqueeze(0).repeat(B, 1), pos_map, is_thing


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0, enabled=True):
        self.index, self.samples, self._stop, self.enabled = index, [], threading.Event(), enabled
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([v.strip() for v in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        if self.enabled:
            self.t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self.enabled:
            self.t.join(timeout=6)

    def summary(self):
        sm = sorted(float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit())
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        mx = max(float(s[1]) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[3 + i].lower().startswith("active") for s in self.samples if len(s) >= 7)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": reasons, "samples": len(sm)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


# ------------------------------------------------------------------------------------------ CPU oracle arm
def cpu_oracle_seconds_per_image(cfg, verbose=False):
    """Times the CPU oracle (oracle/, the restatement of the reference eval forward; the unmodified reference cannot run on CPU:
    its MSDeformAttn op throws and detectron2/fvcore/timm are absent -- DESIGN.md) on ONE image of the workload: the whole hot path
    a1-a19 in full (all 32 ViT-H blocks, BERT, VL fusion, deformable encoder/decoder, MaskDINO, CondInst), no extrapolation.
    Threads: min(32, cores) -- on the 128-core boxes more threads are slower for this B=1 problem size."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from hipie_oracle import hparams, synth
    from hipie_oracle.model import HipieOracle
    threads = min(32, os.cpu_count() or 8)
    torch.set_num_threads(threads)
    hp = hparams.get("vit_h")
    hp.update(max_query_len=cfg["lt"], max_pool=cfg["max_pool"], bg_cls_agnostic=cfg["bg_agnostic"])
    torch.manual_seed(0)
    model = HipieOracle(hp).eval()
    synth.perturb_(model)
    inputs, ids, am = synth.make_batch(1, cfg["img"], cfg["img"], cfg["classes"], cfg["lt"], task=cfg["task"])
    with torch.no_grad():
        tensor, mask, sizes = model.preprocess([x["image"] for x in inputs])
        t0 = time.perf_counter()
        lang = model.forward_text(ids, am)
        model.coco_inference(tensor, mask, sizes, lang, task=cfg["task"])
        total = time.perf_counter() - t0
    if verbose:
        print(f"[cpu oracle] {cfg['name']}: {total:.1f} s/img on {threads} threads", file=sys.stderr)
    sample = f"1 image {cfg['img']}^2 of {cfg['name']}: the whole hot path a1-a19 in full (32 ViT-H blocks, BERT, VL fusion, deformable enc/dec, " \
             f"MaskDINO, CondInst), {threads} torch threads"
    return total, threads, sample


def run_reference(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    secs, sample, threads = [], "", 0
    t_start = time.perf_counter()
    warm = 1 if (args.warmup > 0 and args.ref_budget_s >= 150) else 0      # one untimed sample warms the allocator / thread pool
    for i in range(warm + args.steps):
        total, threads, sample = cpu_oracle_seconds_per_image(cfg, verbose=True)
        if i >= warm:
            secs.append(total)
        if secs and time.perf_counter() - t_start + 1.2 * total > args.ref_budget_s:
            break                        # keep the whole reference run within a few minutes
    spi = sorted(secs)[len(secs) // 2]
    val = 1.0 / spi
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "images/s", "n_gpus": args.gpus, "steps": len(secs),
            "warmup": warm, "ms_per_step": spi * 1000.0, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{cfg['name']}: {cfg['desc']} -- CPU oracle of the reference path, one image per step",
                       "note": f"{len(secs)} timed samples (median) of {args.steps} requested within a {args.ref_budget_s:.0f}s wall-clock budget, "
                               f"{warm} warm-up sample; each sample = the full hot path on one image (no extrapolation)"},
            "cpu_baseline": {"value": val, "unit": "images/s", "cores": threads, "kind": "port", "sample": sample,
                             "host_cores": os.cpu_count()},
            "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ product arm
def ncu_traffic(kernel_tag):
    """DRAM bytes per launch of the dominant kernel class from the committed `ncu --set full` capture of THIS round
    (profiles/r02_ncu_summary.json, keyed by the same tags the live profiler uses); None when no capture of that class is committed."""
    p = os.path.join(ROOT, "profiles", "r02_ncu_summary.json")
    try:
        d = json.load(open(p))
        e = d.get(kernel_tag)
        if e:
            return e["dram_bytes_per_launch"], f"committed ncu capture profiles/r02_ncu_summary.json[{kernel_tag}] ({e.get('launch', '')}, commit {d.get('_commit', '?')}): " \
                                               f"dram__bytes_read.sum + dram__bytes_write.sum of one launch; not re-measured in this run"
    except Exception:
        pass
    return None, None


DUMP_CAP = 1 << 18          # elements kept per array; a larger array is dumped as a fixed, seeded sample of this many elements
DUMP_BUDGET = 64 << 20      # bytes of all dumped arrays together


def dump_outputs(out, path):
    """Writes every tensor of the hot path's result (nested dicts / lists flattened to dotted names, e.g. aux.hs.5) as
    <path>/<name>.npy: floating point and bool as float32, integers (top-k indices) as float64.  An array of more than DUMP_CAP
    elements is replaced by its elements at DUMP_CAP flat positions drawn with seed 0 and sorted, the same positions in every run,
    so that the dumps of two builds compare element for element."""
    import numpy as np
    import torch
    tensors = {}

    def walk(name, v):
        if torch.is_tensor(v):
            tensors[name] = v
        elif isinstance(v, dict):
            for k, x in v.items():
                walk(f"{name}.{k}" if name else str(k), x)
        elif isinstance(v, (list, tuple)):
            for i, x in enumerate(v):
                walk(f"{name}.{i}", x)
    walk("", out)
    arrays = {}
    for name, t in sorted(tensors.items()):
        t = t.detach()
        if t.numel() > DUMP_CAP:
            idx = torch.randint(t.numel(), (DUMP_CAP,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        exact_ints = not t.is_floating_point() and t.dtype != torch.bool
        arrays[name] = (t.double() if exact_ints else t.float()).cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BUDGET:
        raise RuntimeError(f"--dump-outputs: {len(arrays)} arrays take {total} bytes, more than {DUMP_BUDGET}")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)
    print(f"[bench] dumped {len(arrays)} arrays ({total / 2**20:.1f} MiB) of the last timed step to {path}", file=sys.stderr)


def run_product(args, cfg):
    import torch
    import torch.distributed as dist
    from hipie_b200 import _lib, ops
    from hipie_b200.modeling import params as P
    from hipie_b200.modeling.hipie_img import HIPIE_IMG
    from hipie_b200.parallel import PackedAllGather
    from hipie_b200.hostio import PinnedArena

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (product arm) needs a CUDA device: there is no CPU fallback for the hot path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    prec = 1 if args.precision == "bf16" else 3
    ops.set_precision(prec)
    hp = vit_h_hp(cfg)
    model = HIPIE_IMG(hp=hp, state_dict=P.random_state_dict(hp, seed=0), device=str(dev))
    model.engine.bf16_value_map = prec == 1
    B, IMG, task = cfg["batch"], cfg["img"], cfg["task"]
    g = torch.Generator().manual_seed(1234 + rank)
    host_imgs = [(torch.rand(3, IMG, IMG, generator=g) * 255.0).pin_memory() for _ in range(B)]
    ids, am, pos_map, is_thing = batch_text(cfg, B, seed_base=100 * rank)
    same_rows = task == "detection"
    dev_imgs = torch.stack(host_imgs).to(dev)
    ids_d, am_d = ids.to(dev), am.to(dev)
    pad_mask = torch.zeros(B, IMG, IMG, dtype=torch.bool, device=dev)
    sizes = [(IMG, IMG)] * B
    gather_keys = ["pred_logits", "pred_boxes", "pred_boxious", "pred_logits_maskdino", "pred_boxes_maskdino"]

    graphed = None
    if not args.no_graph:
        with torch.no_grad():
            graphed = model.capture_hot_path(dev_imgs, pad_mask, sizes, ids_d, am_d, task=task, same_rows=same_rows)
    gather = PackedAllGather() if world > 1 else None

    def hot_step():
        if graphed is not None:
            out = graphed()
        else:
            lang = model.forward_text_async(ids_d, am_d, same_rows=same_rows)
            out = model.coco_inference(dev_imgs, pad_mask, sizes, lang, task=task)
        if gather is not None:     # the only collective of the data-parallel path: ONE all-gather of the packed fixed-shape outputs
            gather(out, gather_keys)
        return out

    arena = PinnedArena(96 << 20)      # results land in ONE persistent page-locked arena (hipie_b200/hostio.py)

    def e2e_step():
        batched = [dict(image=im, height=IMG, width=IMG, task=task, is_thing=is_thing, positive_map_label_to_token=pos_map,
                        input_ids=ids[b], attention_mask=am[b]) for b, im in enumerate(host_imgs)]
        res = model(batched)
        arena.reset()
        to_host = (lambda t: t.cpu()) if os.environ.get("HIPIE_BENCH_PAGEABLE_D2H") == "1" else arena.to_host
        host = []
        for r in res:
            inst = r["instances"]
            item = [to_host(inst.pred_boxes.tensor), to_host(inst.scores), to_host(inst.pred_classes)]
            if task == "detection":
                sem = r["sem_seg"].argmax(0)
                item += [to_host(r["panoptic_seg"][0]), to_host(sem.to(torch.uint8 if r["sem_seg"].shape[0] <= 256 else torch.int16))]
            else:
                item.append(to_host(inst.pred_masks))
            host.append(tuple(item))
        torch.cuda.synchronize()      # all copies were queued before this one synchronize
        return host

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        for _ in range(args.warmup):
            hot_step()
        barrier()
        launches0 = _lib.launch_count()
        with ClockSampler(local, enabled=rank == 0) as clk:      # one nvidia-smi poller per job, not per rank
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(args.steps):
                out = hot_step()
            e.record()
            barrier()
        ms = s.elapsed_time(e)
        if args.dump_outputs and rank == 0:      # before the steps below can reuse any buffer of the last timed step
            dump_outputs(out, args.dump_outputs)
        launches = _lib.launch_count() - launches0
        if graphed is not None:          # replayed launches are not re-counted by the library: kernels per capture x replays
            launches = graphed.launches_per_replay * args.steps
        # per-kernel live event timing (separate, identical steps so the events do not perturb the headline number)
        ops.profiler.start()
        prof_steps = max(1, min(2, args.steps))
        overlap, model.overlap_branches = model.overlap_branches, False      # one stream: a kernel's events must bracket that kernel alone
        for _ in range(prof_steps):      # eager (un-graphed) so that each launch can be bracketed by events
            lang = model.engine.forward_text(ids_d, am_d, same_rows=same_rows)
            model.coco_inference(dev_imgs, pad_mask, sizes, lang, task=task)
        prof = ops.profiler.stop()
        model.overlap_branches = overlap
        # the ViT-H forward on its own (north-star: tensor fraction ON THE ViT-H FORWARD): CUDA events around engine.vit alone
        vit_ms = None
        if hp["backbone"] == "vit":
            for _ in range(2):
                model.engine.vit(dev_imgs)
            vs, ve = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            vs.record()
            for _ in range(3):
                model.engine.vit(dev_imgs)
            ve.record()
            torch.cuda.synchronize()
            vit_ms = vs.elapsed_time(ve) / 3.0
        # end-to-end through the public API with host buffers
        e2e_iters = max(1, min(args.steps, 5))
        model.enable_cuda_graphs(not args.no_graph)      # serving mode of the public API: forward() replays its own graph
        e2e_step()
        e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_iters):
            host = e2e_step()
        torch.cuda.synchronize()
        e2e_s = (time.perf_counter() - t0) / e2e_iters
    t_ms = torch.tensor([ms, e2e_s * 1000.0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_max, e2e_ms_max = float(t_ms[0]), float(t_ms[1])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk = peaks()
    imgs_total = world * B * args.steps
    value = imgs_total / (ms_max / 1000.0)
    h2d = B * 3 * IMG * IMG * 4 + 2 * B * hp["max_query_len"] * 8
    d2h = sum(sum(t.numel() * t.element_size() for t in h) for h in host)
    tot_prof = sum(v["ms"] for v in prof.values()) or 1.0
    top = max(prof.items(), key=lambda kv: kv[1]["ms"])
    kernels = {}

    def mma_passes(tag):
        """bf16-rate pass-equivalents one algorithmic MAC costs in this kernel class (DESIGN.md 3): p3 = three bf16 passes; f16x2 = two fp16
        passes; f16+e4m3 = one fp16 pass + ONE e4m3 pass over 2K at twice the 16-bit rate = two; f16x1 / p1 = one."""
        if "[p3]" in tag:
            return 3
        if "[f16x2]" in tag or "[f16+e4m3]" in tag:
            return 2
        return 1
    for tag, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"]):
        per = v["ms"] / v["launches"]
        entry = {"share_of_timed_kernels": v["ms"] / tot_prof, "launches_per_step": v["launches"] / prof_steps, "avg_ms": per}
        if v["work"] > 0:
            rate = v["work"] / v["launches"] / (per / 1000.0)
            if tag.startswith(("msda", "condinst", "layernorm", "row_softmax", "seg_postprocess")) or "mask_embed" in tag:
                entry.update(bound="hbm", achieved=rate / 1e9, unit="GB/s", frac=rate / 1e9 / pk["hbm"])
            else:
                entry.update(bound="tensor", achieved=rate / 1e12, unit="TFLOP/s", frac=rate / 1e12 / pk["tf_sustained"],
                             mma_pass_equivalents=mma_passes(tag), executed_frac=rate / 1e12 * mma_passes(tag) / pk["tf_sustained"])
        kernels[tag] = entry
    # all dense contractions of the step together (every gemm_tc class except the HBM-bound mask-embed)
    gsel = [(t, v) for t, v in prof.items() if t.startswith("gemm_tc") and "mask_embed" not in t and v["work"] > 0]
    g_ms = sum(v["ms"] for _, v in gsel) or 1.0
    g_alg = sum(v["work"] for _, v in gsel) / (g_ms / 1000.0) / 1e12
    g_exe = sum(v["work"] * mma_passes(t) for t, v in gsel) / (g_ms / 1000.0) / 1e12
    gemm_all = {"share_of_timed_kernels": g_ms / tot_prof, "achieved": g_alg, "unit": "TFLOP/s", "frac": g_alg / pk["tf_sustained"],
                "executed_tflops": g_exe, "executed_frac": g_exe / pk["tf_sustained"],
                "classes": {t: round(v["ms"] / g_ms, 4) for t, v in sorted(gsel, key=lambda kv: -kv[1]["ms"])}}
    tk = kernels[top[0]]
    traffic, traffic_note = ncu_traffic(top[0])
    roofline = {"kernel": top[0], "bound": tk.get("bound", "tensor"), "achieved": tk.get("achieved"),
                "peak": pk["hbm"] if tk.get("bound") == "hbm" else pk["tf_sustained"],
                "unit": tk.get("unit"), "frac": tk.get("frac"), "traffic": traffic, "traffic_note": traffic_note,
                "mma_passes": mma_passes(top[0]), "executed_tflops": (tk.get("achieved") or 0.0) * mma_passes(top[0]) if tk.get("bound") == "tensor" else None,
                "executed_frac": (tk.get("frac") or 0.0) * mma_passes(top[0]) if tk.get("bound") == "tensor" else None,
                "achieved_note": "algorithmic 2MNK flops / measured kernel time (CUDA events on the launching stream, eager steps after the "
                                 "timed region).  Every contraction is fp32-class: per algorithmic MAC the kernel issues mma_passes bf16-rate "
                                 "pass-equivalents (p3: Ah.Wh + Ah.Wl + Al.Wh in bf16 = 3; f16x2: A.Wh + A.Wl in fp16 = 2; f16+e4m3: one fp16 pass + "
                                 "ONE e4m3 pass over 2K at twice the rate = 2; f16x1 = 1), executed_* = achieved x mma_passes against the same "
                                 "bf16 peak (DESIGN.md 3)",
                "gemm_tc_all": gemm_all,
                "peak_source": pk["src"] + " (sustained figure: kernel timed inside a long step)",
                "vit_h_forward_tensor_frac": (cfg["vit_flops"] * B * world * args.steps / (ms_max / 1000.0)) / 1e12 / (pk["tf_sustained"] * world),
                "vit_h_forward_tensor_frac_note": "ViT-H forward flops / the WHOLE step time (detector, text encoder, MaskDINO included): a lower bound",
                "vit_h_forward_alone": None if not vit_ms else {
                    "ms": vit_ms, "tflops": cfg["vit_flops"] * B / (vit_ms / 1000.0) / 1e12, "frac": cfg["vit_flops"] * B / (vit_ms / 1000.0) / 1e12 / pk["tf_sustained"],
                    "note": "engine.vit(batch) alone on rank 0, eager launches, CUDA events, 3 calls after 2 warm-ups: algorithmic ViT-H forward flops "
                            "(linears + attention) / its own time against the sustained bf16 peak"},
                "north_star_hbm": {k: {"achieved_gbs": kernels[k]["achieved"], "frac": kernels[k]["frac"], "avg_ms": kernels[k]["avg_ms"]}
                                   for k in kernels if (k.startswith("msda_fused") or "mask_embed" in k) and "achieved" in kernels[k]},
                "kernels": kernels}
    cpu = None
    if not args.no_cpu_baseline:
        try:
            total, threads, sample = cpu_oracle_seconds_per_image(cfg, verbose=True)
            cpu = {"value": 1.0 / total, "unit": "images/s", "cores": threads, "kind": "port", "sample": sample,
                   "seconds_per_image": total, "host_cores": os.cpu_count()}
        except Exception as ex:  # the CPU leg must never take the GPU number down with it
            cpu = {"value": None, "unit": "images/s", "cores": 0, "kind": "port", "sample": f"failed: {ex}"}
    bert_rows = 1 if same_rows else B
    line = {"metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp32-class split precision on the tensor cores (operand planes per contraction: fp16 + e4m3 split, two fp16 passes, "
                     "three bf16 passes, one fp16 pass for softmax-normalised products; fp32 accumulate; DESIGN.md 3)" if prec == 3 else "bf16",
            "data": "synthetic",
            "config": {"workload": f"{cfg['name']}: {cfg['desc']}",
                       "per_gpu_batch": B, "global_batch": B * world, "parallelism": f"dp{world} (image sharding, one packed all-gather of logits / boxes)",
                       "value_scope": "SURVEY 8a rows a1-a19: preprocess, ViT-H, BERT, VL fusion, deformable enc/dec, MaskDINO + mask-embed, CondInst masks; "
                                      f"the text encoder runs on {bert_rows} row(s) per step "
                                      + ("(all images of a detection batch share one vocabulary prompt, hipie_img.py:330-332: encoded once and broadcast)"
                                         if same_rows else "(one expression per image)"),
                       "e2e_scope": "HIPIE_IMG.forward (public API) incl. post-processing rows a20-a23, pinned-host images in, results out",
                       "l2": "per-step working set (>= 1 GB activations per block) exceeds the 126 MB L2; no explicit flush",
                       "precision_mode": args.precision,
                       "launch": "eager" if graphed is None else "CUDA graph replay of the hot step (kernels captured once after warm-up)"},
            "clocks": clk.summary(),
            "e2e": {"value": world * B / (e2e_ms_max / 1000.0), "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=1, choices=sorted(CONFIGS), help="BASELINE.json configs[N] (default 1: the headline workload)")
    ap.add_argument("--precision", default="bf16x3", choices=["bf16x3", "bf16"],
                    help="bf16x3 = parity-grade split precision (default, the headline); bf16 = fast mode")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch the hot step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--ref-budget-s", type=float, default=240.0, help="wall-clock budget of the --impl reference run")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy (product arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    # stdout carries exactly one JSON line.  NCCL_DEBUG is left as the caller set it (the driver reads the NCCL log for its
    # evidence); NCCL prints its log to stdout by default, so it is routed to stderr instead of being silenced.
    if int(os.environ.get("WORLD_SIZE", "1")) > 1 and os.environ.get("NCCL_DEBUG", ""):
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    cfg = CONFIGS[args.config]
    if args.impl == "reference":
        run_reference(args, cfg)
    else:
        run_product(args, cfg)


if __name__ == "__main__":
    main()
