#!/usr/bin/env python
"""bench.py -- items/s for the BGE-base embed .map() hot path on N B200s (BASELINE.json's metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [...]                          # the CPU reference arm
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W   # N > 1: one rank per GPU

A "step" is one pass of the hot path over one batch of synthetic input: 32 waves (32 x 148 = 4736 on a B200;
BENCH_ITEMS_PER_STEP overrides) of 512-token items per GPU, presented as .map() inputs of 32 items (the reference's BATCH_SIZE,
06_gpu_and_ml/embeddings/text_embeddings_inference.py:19).  Weak scaling: every rank owns one GPU and an
equal shard of the items; the path has no data-path collective (items are independent), so ranks only
meet in the timing barrier.

  value  : device-resident throughput -- token ids already in HBM, forwards enqueued back to back through
           b200rt_embed_device on torch's current stream, timed with CUDA events on that stream.
  e2e    : the same metric through the C ABI a binding uses (b200rt_submit / b200rt_wait) with HOST buffers:
           pinned ids -> H2D -> scatter kernel -> forward -> fused gather -> D2H, copies inside the timed region.
  roofline: dominant kernel (by summed device time inside the forward, CUDA events on the compute stream)
           against the measured tensor peak in MEASURED_PEAKS.json.
  cpu_baseline: the oracle's HF-transformers fp32 path on the host cores (N=1, rank 0, bounded sample).

--dump-outputs DIR writes the embeddings the timed path returned in its last step to DIR/embeddings.npy (see dump_outputs);
weights and inputs are seeded, so two builds run with the same arguments can be compared row for row.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True  # the tree may be read-only: the benchmark writes nothing into it
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "modal-examples_b200"))

METRIC = "items/sec for BGE-base embed .map()"
SEQ = 512
MAP_INPUT_ITEMS = 32           # reference BATCH_SIZE
ITEMS_PER_STEP = int(os.environ.get("BENCH_ITEMS_PER_STEP", "0"))  # per GPU; 0 = 32 waves of the runtime's wave size (32 x 148 = 4736 on a B200)
REF_ITEMS_PER_STEP = 8         # bounded sample for the CPU arm
FLOPS_PER_ITEM = 96.64e9       # BASELINE.md §4 (2*m*n*k, all rows, 12 layers)

# per-layer algorithmic FLOPs per item of each tensor kernel (S = 512)
KERNEL_FLOPS = {
    "gemm_qkv": 2 * 512 * 768 * 2304, "gemm_attn_out": 2 * 512 * 768 * 768, "gemm_ffn1_gelu": 2 * 512 * 768 * 3072,
    "gemm_ffn2": 2 * 512 * 3072 * 768, "attention": 4 * 512 * 512 * 768,
}
# algorithmic HBM bytes per token of the row-wise kernels (DESIGN.md §4): embedding gather = one fp32 word row in, the
# residual stream out as fp16 hi + fp16 lo, six (sum, M2) partials.  (There is no LayerNorm kernel any more.)
KERNEL_BYTES = {"embed": 3072 + 1536 + 1536 + 48}
DUMP_BYTES = 64 << 20          # --dump-outputs writes at most this much


def dump_outputs(path, emb):
    """Writes `emb` (one embedding per item, in input order) as PATH/embeddings.npy in float32.  Beyond DUMP_BYTES a fixed
    sample of rows (numpy default_rng(0), kept in input order) stands in for the whole, the same rows on every run."""
    import numpy as np

    emb = np.asarray(emb, dtype=np.float32)
    keep = (DUMP_BYTES - 4096) // (emb.shape[1] * 4)  # 4096: room for the .npy header
    if len(emb) > keep:
        emb = emb[np.sort(np.random.default_rng(0).choice(len(emb), keep, replace=False))]
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "embeddings.npy"), emb)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tflops_burst=d["bf16_tflops"], tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="MEASURED_PEAKS.json (measured)")
    return dict(hbm_gbs=6650.0, tflops_burst=1590.0, tflops_sustained=1400.0, source="B200_PROFILING.md fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, line in self.lines:
            if not (t0 <= t <= t1):
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except Exception:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no sample inside the timed region"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm), "reasons": sorted(reasons)}


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


# ------------------------------------------------------------------------------------------ reference arm


def pick_threads(model, ids_one):
    """torch intra-op threads that actually run the oracle fastest on this host: `os.cpu_count()` over-subscribes
    containers whose CPU quota is smaller than the visible core count (128 threads ran 5x slower than 8 here)."""
    import torch
    from oracle import bge_ref as R

    ncpu = os.cpu_count() or 1
    try:
        ncpu = min(ncpu, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    cands = sorted({t for t in (4, 8, 16, 32, 64, ncpu) if t <= ncpu})
    best, best_t = cands[-1], float("inf")
    for t in cands:
        torch.set_num_threads(t)
        R.forward_hf(model, ids_one)  # warm
        t0 = time.perf_counter()
        R.forward_hf(model, ids_one)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = t, dt
    torch.set_num_threads(best)
    return best


def cpu_reference_run(n_items, warm_items, threads=None):
    """HF BertModel fp32 + CLS pool + L2 normalise on the host cores (oracle/bge_ref.py); returns items/s."""
    import numpy as np
    import torch
    from oracle import bge_ref as R

    g = R.BGE_BASE
    flat = R.make_weights(g, 0, "hf")
    model = R.build_hf_model(flat, g)
    ids = R.synth_ids(max(n_items, warm_items), SEQ, 0)
    threads = threads or pick_threads(model, ids[:1])
    torch.set_num_threads(threads)
    R.forward_hf(model, ids[:warm_items])
    t0 = time.perf_counter()
    out = R.forward_hf(model, ids[:n_items])
    dt = time.perf_counter() - t0
    assert np.isfinite(out).all()
    return n_items / dt, threads, dt, model, ids


def main_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return 0
    import numpy as np
    from oracle import bge_ref as R
    import torch

    g = R.BGE_BASE
    model = R.build_hf_model(R.make_weights(g, 0, "hf"), g)
    ids = R.synth_ids(REF_ITEMS_PER_STEP, SEQ, 0)
    threads = pick_threads(model, ids[:1])
    for _ in range(max(args.warmup, 1)):
        R.forward_hf(model, ids)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = R.forward_hf(model, ids)
    dt = time.perf_counter() - t0
    assert np.isfinite(out).all()
    value = args.steps * REF_ITEMS_PER_STEP / dt
    sample = f"{REF_ITEMS_PER_STEP} items x {SEQ} tokens per step (bounded sample of the 1M-item workload), HF BertModel fp32, torch {threads} threads (fastest of a sweep up to the visible cores)"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "items/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"bge-base-en-v1.5 embed, {SEQ}-token synthetic items, CPU oracle port of the TEI /embed path", "seq_len": SEQ,
                   "items_per_step": REF_ITEMS_PER_STEP},
        "cpu_baseline": {"value": value, "unit": "items/s", "cores": threads, "host_cores": os.cpu_count(), "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "items/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    GUARD.emit(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------ our arm


def _load_example():
    """examples/embed_bge_native.py (the reference script with TEI replaced by the engine): its `TextEmbeddings` class is
    what `e2e_map` drives through the `modal` shim's Function.map."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("embed_bge_native", os.path.join(ROOT, "examples", "embed_bge_native.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def run_independent_replicas(args, rank, local_rank, world, barrier, R):
    """N > 1 only, secondary figure: every rank drives its own 1-replica pool on its own GPU (no scatter, no gather, no
    shared dispatcher) -- the trivially parallel deployment the single-root pool is compared with."""
    import torch
    import b200rt

    steps = max(3, args.steps // 4)
    b200rt.init(devices=[local_rank])
    model = b200rt.EmbedModel(R.geometry_dict(R.BGE_BASE), R.pack_blob(R.make_weights(R.BGE_BASE, 0, "hf"), R.BGE_BASE))
    cap = b200rt.wave_capacity_items()
    n_step = ITEMS_PER_STEP or 32 * cap
    with torch.cuda.device(local_rank):
        d_ids = torch.from_numpy(R.synth_ids(n_step, SEQ, seed=rank)).cuda()
        d_lens = torch.full((n_step,), SEQ, dtype=torch.int32, device="cuda")
        d_out = torch.empty((n_step, 768), dtype=torch.float32, device="cuda")
        ts = torch.cuda.Stream()

        def device_step():
            for i in range(0, n_step, cap):
                model.embed_device(0, d_ids[i:].data_ptr(), d_lens[i:].data_ptr(), min(cap, n_step - i), SEQ, d_out[i:].data_ptr(), ts.cuda_stream)

        with torch.cuda.stream(ts):
            for _ in range(args.warmup):
                device_step()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(ts):
            e0.record()
            for _ in range(steps):
                device_step()
            e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
    del d_ids, d_lens, d_out
    b200rt.shutdown()
    torch.cuda.empty_cache()
    return ms, steps, n_step


def main_ours(args):
    import numpy as np
    import torch
    import b200rt
    from oracle import bge_ref as R  # weights + synthetic inputs only (shared bit-for-bit with the oracle)

    rank, local_rank, world = dist_env()
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback for the CUDA path (use --impl reference for the CPU arm)")
    N = args.gpus
    if torch.cuda.device_count() < N:
        raise SystemExit(f"--gpus {N} but only {torch.cuda.device_count()} visible")
    torch.cuda.set_device(local_rank)
    use_dist = world > 1
    host_pg = None
    if use_dist:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        # Long waits (ranks > 0 idle while rank 0 drives the pool) go through a gloo group: an NCCL barrier spins a kernel
        # on every waiting rank's GPU, which would time-slice against the pool's replicas on the same GPUs.
        host_pg = dist.new_group(backend="gloo")

    def barrier():
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()

    def host_barrier():
        if use_dist:
            dist.barrier(group=host_pg)

    # ---------------- N > 1, secondary: independent 1-replica pools, one per rank (the round-1 deployment)
    indep = None
    if use_dist:
        ms, isteps, istep_items = run_independent_replicas(args, rank, local_rank, world, barrier, R)
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)  # max over ranks, device time
        indep = {"value": isteps * istep_items * world / (float(t[0]) / 1e3), "unit": "items/s", "steps": isteps,
                 "what": "one process per GPU, each a 1-replica pool on its own shard, ids resident (no scatter/gather, peer_bytes 0)"}
        torch.cuda.synchronize()
    host_barrier()
    if rank != 0:
        # ---------------- ranks > 0: the pool is ONE process (rank 0) driving all N replicas; hold the barrier only
        host_barrier()
        dist.destroy_process_group()
        return 0

    # ================= rank 0: ONE pool of N replicas (scatter kernel -> peer HBM, fused peer gather, one dispatcher)
    b200rt.init(N)
    g = R.BGE_BASE
    flat = R.make_weights(g, 0, "hf")
    model = b200rt.EmbedModel(R.geometry_dict(g), R.pack_blob(flat, g))
    del flat
    cap = b200rt.wave_capacity_items()
    n_step = ITEMS_PER_STEP or 32 * cap          # per GPU: 32 full waves, a whole number of 32-item .map() inputs
    n_total = n_step * N                         # per step, whole pool
    ids_host = np.concatenate([R.synth_ids(n_step, SEQ, seed=r) for r in range(N)])  # replica r's shard has seed r
    peaks = load_peaks()

    # ---------------- value: device-resident (each replica's shard already in its HBM), one enqueueing thread per replica
    dev = []
    for r in range(N):
        with torch.cuda.device(r):
            d = {"ids": torch.from_numpy(ids_host[r * n_step:(r + 1) * n_step]).cuda(),
                 "lens": torch.full((n_step,), SEQ, dtype=torch.int32, device="cuda"),
                 "out": torch.empty((n_step, 768), dtype=torch.float32, device="cuda"),
                 # a dedicated (non-default) stream: the forwards are enqueued on it and the events that time them are
                 # recorded on it (handle 0 would mean "the replica's own stream" to b200rt_embed_device)
                 "stream": torch.cuda.Stream()}
            assert d["stream"].cuda_stream != 0
            dev.append(d)

    def device_step(r):
        d = dev[r]
        for i in range(0, n_step, cap):
            n = min(cap, n_step - i)
            model.embed_device(r, d["ids"][i:].data_ptr(), d["lens"][i:].data_ptr(), n, SEQ, d["out"][i:].data_ptr(), d["stream"].cuda_stream)

    def device_loop(steps, timed):
        """`steps` device steps on every replica concurrently; returns the max over replicas of the device time (ms)."""
        gate = threading.Barrier(N)
        ms = [0.0] * N
        errs = []

        def work(r):
            try:
                with torch.cuda.device(r):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    gate.wait()
                    with torch.cuda.stream(dev[r]["stream"]):
                        e0.record()
                        for _ in range(steps):
                            device_step(r)
                        e1.record()
                    dev[r]["stream"].synchronize()
                    ms[r] = e0.elapsed_time(e1)
            except Exception as e:  # noqa: BLE001
                errs.append(e)
                gate.abort()

        th = [threading.Thread(target=work, args=(r,)) for r in range(N)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        if errs:
            raise errs[0]
        return max(ms)

    def sync_all():
        for r in range(N):
            torch.cuda.synchronize(r)

    device_loop(args.warmup, False)
    sync_all()
    st0 = b200rt.stats()
    sampler = ClockSampler(0)
    sampler.start()
    time.sleep(0.25)
    t_wall0 = time.time()
    tw0 = time.perf_counter()
    dev_ms = device_loop(args.steps, True)
    sync_all()
    tw1 = time.perf_counter()
    t_wall1 = time.time()
    assert abs(dev_ms - (tw1 - tw0) * 1e3) < 0.05 * dev_ms + 10.0, f"CUDA-event time {dev_ms} and synchronised wall time {(tw1 - tw0) * 1e3} disagree"
    st1 = b200rt.stats()
    clocks = sampler.stop(t_wall0, t_wall1)
    launches = st1["kernel_launches"] - st0["kernel_launches"]
    for r in range(N):
        norms = torch.linalg.vector_norm(dev[r]["out"], dim=1)
        assert torch.allclose(norms, torch.ones_like(norms), atol=1e-3), "device path produced non-unit embeddings"

    # ---------------- per-kernel device times inside a sustained loop (same warm, power-capped chip as the timed region):
    # ~1 s of back-to-back forwards with CUDA events between the launches on replica 0's compute stream
    prof = model.profile_forward(cap, SEQ, iters=60)

    # ---------------- e2e: the C ABI with HOST buffers -- .map() inputs of 32 items lent from pinned memory
    # (b200rt_submit_ex BORROW_IDS) -> H2D -> scatter kernel -> forward -> fused gather -> D2H into the caller's pinned out
    n_inputs = n_total // MAP_INPUT_ITEMS
    pin_ids = b200rt.PinnedBuffer((n_total, SEQ), np.int32)
    pin_ids.array[:] = ids_host
    pin_out = b200rt.PinnedBuffer((n_total, 768), np.float32)

    def e2e_step():
        tickets = []
        for j in range(n_inputs):
            s = slice(j * MAP_INPUT_ITEMS, (j + 1) * MAP_INPUT_ITEMS)
            tickets.append(model.submit(pin_ids.array[s], None, out=pin_out.array[s], borrow_ids=True))
        for t in tickets:
            model.wait(t)

    for _ in range(max(1, args.warmup)):
        e2e_step()
    sync_all()
    s0 = b200rt.stats()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    sync_all()
    e2e_s = time.perf_counter() - t0
    s1 = b200rt.stats()
    e2e_out = pin_out.array.copy()
    assert np.allclose(np.linalg.norm(e2e_out, axis=1), 1.0, atol=1e-3)
    dev_out = np.concatenate([dev[r]["out"].cpu().numpy() for r in range(N)])
    assert float(np.abs(dev_out - e2e_out).max()) < 1e-5, "device-resident and host-buffer paths disagree"

    # ---------------- ragged lengths (uniform 16..512, seed 1: SURVEY.md section 8(d)'s correctness variant) at throughput: the
    # same submit/wait path; items travel in 64-token length buckets, so tokens/s should stay near the full-length figure
    rng_r = np.random.default_rng(1)
    r_lens = rng_r.integers(16, SEQ + 1, size=n_total).astype(np.int32)
    pin_lens = b200rt.PinnedBuffer((n_total,), np.int32)
    pin_lens.array[:] = r_lens

    def ragged_step():
        tk = [model.submit(pin_ids.array[j * MAP_INPUT_ITEMS:(j + 1) * MAP_INPUT_ITEMS], pin_lens.array[j * MAP_INPUT_ITEMS:(j + 1) * MAP_INPUT_ITEMS],
                           out=pin_out.array[j * MAP_INPUT_ITEMS:(j + 1) * MAP_INPUT_ITEMS], borrow_ids=True) for j in range(n_inputs)]
        for t in tk:
            model.wait(t)

    ragged_step()
    sync_all()
    t0 = time.perf_counter()
    r_steps = max(2, args.steps // 4)
    for _ in range(r_steps):
        ragged_step()
    sync_all()
    ragged_s = time.perf_counter() - t0
    assert np.allclose(np.linalg.norm(pin_out.array, axis=1), 1.0, atol=1e-3)
    ragged = {"lens": "uniform 16..512 (numpy default_rng(1))", "items_per_s": r_steps * n_total / ragged_s,
              "tokens_per_s": r_steps * float(r_lens.sum()) / ragged_s}
    pin_lens.free()

    # ---------------- the device-resident loop once more, now on chips as warm as the e2e loop saw them: separates the
    # cost of the host path from power-cap clock drift between the two timed regions
    dev_ms_after = device_loop(args.steps, True)
    sync_all()

    # ---------------- e2e_map: the same items through the `modal` shim -- examples/embed_bge_native.py's class,
    # `model.embed.map(generate_batches(), order_outputs=False)` exactly as text_embeddings_inference.py:167 calls it
    ex = _load_example()
    shim_obj = ex.TextEmbeddings(n_gpus=N)
    data = [(i, ids_host[i]) for i in range(n_total)]

    def batches(items, size):
        for j in range(0, len(items) - size + 1, size):  # remainder dropped, as the reference does (:156-163)
            yield items[j:j + size]

    def map_pass(items, size):
        done = 0
        t_0 = time.perf_counter()
        for out_batch in shim_obj.embed.map(batches(items, size), order_outputs=False):
            done += len(out_batch)
        return done, time.perf_counter() - t_0

    shim_obj.embed.remote(data[:MAP_INPUT_ITEMS])  # cold start (engine attach + weight upload) outside the timed region
    map_pass(data, MAP_INPUT_ITEMS)                # warm-up pass
    map_steps = max(2, args.steps // 4)
    e2e_map = {"api": "modal shim: TextEmbeddings().embed.map(generate_batches(), order_outputs=False) (examples/embed_bge_native.py)",
               "unit": "items/s"}
    for size, key in ((MAP_INPUT_ITEMS, "value"), (1024, "value_1024_per_input")):
        done, dt = 0, 0.0
        for _ in range(map_steps):
            d_, t_ = map_pass(data, size)
            done += d_
            dt += t_
        e2e_map[key] = done / dt
    big = 65536
    reps = -(-big // n_total)
    big_items = (data * reps)[:big]
    done, dt = map_pass(big_items, MAP_INPUT_ITEMS)
    e2e_map["pass_65536_items"] = {"items": done, "seconds": dt, "value": done / dt, "map_input_items": MAP_INPUT_ITEMS}
    e2e_map["steps"] = map_steps
    st_map = b200rt.stats()

    # ---------------- secondary (SURVEY.md section 8 f3, the next encoder on the same scheduler): CLIP ViT-B/16 image tower,
    # preprocessed pixels in pinned host memory -> per-replica H2D -> forward -> fused gather -> D2H
    vit = None
    if not args.no_vit:
        from b200rt.weights import CLIP_VIT_B16_GEOMETRY, random_vit_blob

        vmodel = b200rt.ImageEmbedModel(CLIP_VIT_B16_GEOMETRY, random_vit_blob(CLIP_VIT_B16_GEOMETRY, 0))
        n_img = 64 * N * 4
        pin_px = b200rt.PinnedBuffer((n_img, 3, 224, 224), np.float32)
        pin_px.array[:] = np.random.default_rng(0).standard_normal((1, 3, 224, 224), dtype=np.float32)
        pin_vo = b200rt.PinnedBuffer((n_img, 512), np.float32)

        def vit_step():
            tk = [vmodel.submit(pin_px.array[j:j + 64], out=pin_vo.array[j:j + 64]) for j in range(0, n_img, 64)]
            for t in tk:
                vmodel.wait(t)

        vit_step()
        sync_all()
        v_steps = max(2, args.steps // 2)
        t0 = time.perf_counter()
        for _ in range(v_steps):
            vit_step()
        sync_all()
        v_s = time.perf_counter() - t0
        assert np.allclose(np.linalg.norm(pin_vo.array, axis=1), 1.0, atol=1e-3)
        gf_per_image = 12 * (2 * 197 * 768 * 2304 + 2 * 197 * 768 * 768 + 2 * 2 * 197 * 768 * 3072 + 4 * 197 * 197 * 768) / 1e9 + 2 * 196 * 768 * 768 / 1e9
        ips = v_steps * n_img / v_s
        vit = {"what": "CLIP ViT-B/16 image tower (image_embeddings_infinity.py:76-77), 224x224 preprocessed pixels from pinned host memory through "
                       "b200rt_submit_pixels/b200rt_wait, inputs of 64 images, seeded random weights", "images_per_s": ips,
               "gflop_per_image": gf_per_image, "tflops": ips * gf_per_image / 1e3,
               "frac_of_tensor_peak": ips / N * gf_per_image / 1e3 / peaks["tflops_sustained"],
               "h2d_GBps": ips * 3 * 224 * 224 * 4 / 1e9, "images_per_step": n_img, "steps": v_steps,
               "reference_published": "> 750 images/s overall on <= 50 x L4 (image_embeddings_infinity.py:19-20; other hardware, context only)"}
        pin_px.free()
        pin_vo.free()

    # ---------------- p50 per-item latency: one 512-token item through the same C ABI, host buffers
    one_ids = pin_ids.array[:1]
    one_out = pin_out.array[:1]
    lat = []
    for i in range(1100):  # SURVEY.md section 8(d): 1 000 trials after 100 warm-ups
        t1 = time.perf_counter()
        model.wait(model.submit(one_ids, None, out=one_out, borrow_ids=True))
        if i >= 100:
            lat.append((time.perf_counter() - t1) * 1e3)
    lat.sort()
    p50_ms, p99_ms = lat[len(lat) // 2], lat[int(len(lat) * 0.99) - 1]
    lat_map = []
    one_item = data[:1]
    for i in range(300):  # the same through the shim: embed.remote([one item])
        t1 = time.perf_counter()
        shim_obj.embed.remote(one_item)
        if i >= 50:
            lat_map.append((time.perf_counter() - t1) * 1e3)
    lat_map.sort()

    total_items = args.steps * n_total
    value = total_items / (dev_ms / 1e3)
    e2e_value = total_items / e2e_s
    ragged["tokens_per_s_full_length"] = e2e_value * SEQ
    ragged["tokens_per_s_ratio"] = ragged["tokens_per_s"] / (e2e_value * SEQ)

    # ---------------- roofline of the dominant kernel (device events between launches, compute stream, sustained loop)
    top = max((k for k in prof if k in KERNEL_FLOPS), key=lambda k: prof[k])
    n_launch = g.layers
    achieved = KERNEL_FLOPS[top] * cap * n_launch / (prof[top] / 1e3) / 1e12
    traffic = None
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get(top)
    total_ms = sum(prof.values())
    roofline = {
        "bound": "tensor", "kernel": top, "achieved": achieved, "peak": peaks["tflops_sustained"], "unit": "TFLOP/s",
        "frac": achieved / peaks["tflops_sustained"], "traffic": traffic, "peak_source": peaks["source"] + ", sustained bf16/fp16 dense",
        "launch_ms": prof[top] / n_launch, "share_of_forward": prof[top] / total_ms,
        "forward": {"items_per_s_per_gpu": value / N, "tflops": value / N * FLOPS_PER_ITEM / 1e12,
                    "frac_of_tensor_peak": value / N * FLOPS_PER_ITEM / 1e12 / peaks["tflops_sustained"],
                    "frac_of_tensor_peak_burst": value / N * FLOPS_PER_ITEM / 1e12 / peaks["tflops_burst"]},
        "per_kernel_ms": prof, "per_kernel_ms_what": f"sum over {n_launch} layers of one {cap}-item wave, averaged over 60 back-to-back forwards (sustained clocks)",
        "tensor_kernels": {k: {"TFLOPs": KERNEL_FLOPS[k] * cap * n_launch / (prof[k] / 1e3) / 1e12,
                               "frac": KERNEL_FLOPS[k] * cap * n_launch / (prof[k] / 1e3) / 1e12 / peaks["tflops_sustained"]}
                           for k in KERNEL_FLOPS if k in prof},
        "hbm_kernels": {k: {"GBps": KERNEL_BYTES[k] * cap * SEQ * (n_launch if k != "embed" else 1) / (prof[k] / 1e3) / 1e9,
                            "frac": KERNEL_BYTES[k] * cap * SEQ * (n_launch if k != "embed" else 1) / (prof[k] / 1e3) / 1e9 / peaks["hbm_gbs"]}
                        for k in KERNEL_BYTES if k in prof},
    }
    cpu_baseline = None
    if N == 1 and not args.no_cpu_baseline:
        v, threads, dt, _, _ = cpu_reference_run(n_items=16, warm_items=4)
        host_cores = os.cpu_count()
        try:
            usable = len(os.sched_getaffinity(0))
        except Exception:
            usable = host_cores
        cpu_baseline = {"value": v, "unit": "items/s", "cores": threads, "host_cores": host_cores, "usable_cores": usable, "kind": "port",
                        "sample": f"16 items x {SEQ} tokens after a 4-item warm-up ({dt:.1f} s), HF BertModel fp32 (oracle), torch {threads} threads "
                                  f"(fastest of a sweep; the host shows {host_cores} cores, {usable} usable by this process)"}
    per_step = lambda a, b_, k, n: (b_[k] - a[k]) / n  # noqa: E731
    line = {
        "metric": METRIC, "value": value, "unit": "items/s", "n_gpus": N, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic",
        "config": {"workload": f"06_gpu_and_ml/embeddings: BGE-base-en-v1.5 embed, synthetic {SEQ}-token items, .map() inputs of {MAP_INPUT_ITEMS}",
                   "seq_len": SEQ, "items_per_step_per_gpu": n_step, "items_per_step": n_total, "map_input_items": MAP_INPUT_ITEMS, "device_batch_items": cap,
                   "weights": "HF default init, numpy default_rng(0), shared with the oracle",
                   "parallelism": f"ONE process, one pool of {N} replica(s): scatter kernel -> peer HBM, forward per replica, pool+normalise stores into the root's gather buffer (no NCCL on the data path)",
                   "l2": "per-step working set (218 MB fp16 weights + ~1.3 GB activations per replica) exceeds the 126 MB L2; no explicit flush",
                   "precision": "fp16 tensor-core operands, fp32 accumulate, fp32 residual/LayerNorm/softmax"},
        "pool": {"replicas": N, "driving_processes": 1, "peer_bytes_per_step": per_step(s0, s1, "peer_bytes", args.steps),
                 "waves_per_step": per_step(s0, s1, "waves", args.steps)},
        "e2e": {"value": e2e_value, "unit": "items/s", "h2d_bytes_per_step": int(per_step(s0, s1, "h2d_bytes", args.steps)),
                "d2h_bytes_per_step": int(per_step(s0, s1, "d2h_bytes", args.steps)), "peer_bytes_per_step": int(per_step(s0, s1, "peer_bytes", args.steps)),
                "ms_per_step": e2e_s / args.steps * 1e3,
                "api": "b200rt_submit_ex(BORROW_IDS)/b200rt_wait (C ABI; ids and out in b200rt_alloc_pinned memory, DMA'd in place)",
                "device_resident_rerun_after_e2e": total_items / (dev_ms_after / 1e3),
                "per_step_ms": {k: (s1[k] - s0[k]) / args.steps / 1e3 for k in ("stage_us", "dispatch_us", "h2d_scatter_us", "forward_us", "gap_us", "d2h_us", "forward_max_us", "gap_max_us")}},
        "e2e_map": e2e_map, "ragged": ragged, "secondary_clip_vit": vit,
        "gpu_launches": launches, "clocks": clocks, "roofline": roofline,
        "latency": {"p50_ms": p50_ms, "p99_ms": p99_ms, "what": "one 512-token item, b200rt_submit_ex+b200rt_wait, pinned host buffers, 1000 trials after 100 warm-ups",
                    "shim_remote_p50_ms": lat_map[len(lat_map) // 2], "shim_remote_p99_ms": lat_map[int(len(lat_map) * 0.99) - 1]},
    }
    if indep:
        line["independent_replicas"] = indep
    if cpu_baseline:
        line["cpu_baseline"] = cpu_baseline
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dev_out)  # the headline device-resident loop's last step, every replica in item order
    GUARD.emit(json.dumps(line))
    pin_ids.free()
    pin_out.free()
    shim_obj._teardown()  # runs the class's @modal.exit hook, which shuts the runtime down
    b200rt.shutdown()
    host_barrier()
    if use_dist:
        dist.destroy_process_group()
    return 0


class StdoutGuard:
    """The contract is ONE JSON line on stdout: libraries (NCCL prints its version banner on stdout) are pointed at
    stderr at the file-descriptor level for the whole run; emit() writes the line to the real stdout."""

    def __init__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, line: str):
        sys.stdout.flush()
        os.write(self.real, (line + "\n").encode())


GUARD = None


def main():
    global GUARD
    GUARD = StdoutGuard()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-vit", action="store_true", help="skip the secondary CLIP ViT-B/16 measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's embeddings to DIR/embeddings.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3  # timing rule: W >= 3
    sys.exit(main_reference(args) if args.impl == "reference" else main_ours(args))


if __name__ == "__main__":
    main()
