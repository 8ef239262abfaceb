#!/usr/bin/env python
"""Benchmark of the Issue_Embeddings encoder hot path (BASELINE.json: issues/sec to 2400-d @ seq_len 512 batch 256).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of 256 synthetic issues x 512 tokens (BASELINE.json configs[1]
shape; reference-deployed R4 encoder: L=4, E=800, H=2400, V=60000, random-init seed 1234): token ids -> per-token
input-projection table lookup (layer 0) / hoisted input-projection GEMMs (layers 1-2) / input projection fused into the
recurrent K loop (last layer) -> 4 x 512 recurrent LSTM steps -> masked [mean|max|last] pool -> (256, 2400) f32.

`batches_per_launch` (5) consecutive steps ride one ie_encoder_encode call (1280 rows): the persistent recurrent kernel
(csrc/lstm_layer.cu) deals the (timestep, batch, column-tile) work items of the five independent batches round-robin over
all 74 CTA pairs, so an item's inputs were finished two rounds earlier and the tensor pipe never waits for a step
barrier.  Each step is still one batch of 256 issues with its own result rows; `single_batch` in the JSON line is the
same measurement with one batch per launch.

* `value`      : whole-job issues/s with the token ids already resident in HBM (CUDA events on the launching stream,
                 barrier + synchronize on both sides, max over ranks; under torchrun each rank encodes its own batches
                 -- weak scaling, no data-path collective -- and the timed region ends with the ONE all-gather of the
                 2400-d outputs).  The W warm-up steps are repeated until the device has been under this load for
                 `config.preroll_s` seconds (BENCH_PREROLL_S, default 2): the board runs at its power cap, the governor
                 needs about a second after an idle -> load edge to settle, and the roofline denominator
                 (MEASURED_PEAKS.json bf16_tflops_sustained) is itself a 4-second back-to-back figure.  The timed region
                 is exactly K steps.
* `e2e`        : the same metric through the public bulk API on HOST token-id lists -- what df_to_embedding does after
                 tokenisation (py/code_intelligence/inference.py:171-229): bulk.encode_bulk_distributed(docs, ...) = global
                 length sort -> issue j to rank j mod G -> IssueEncoder.encode_id_list pipeline (pinned staging, H2D under
                 the previous batch's kernels, C-ABI ie_encoder_encode) -> one NCCL all-gather -> un-sort -> D2H of the
                 (N, 2400) result on rank 0.  Host packing, H2D, D2H are all inside the timed region (perf_counter around the call,
                 device idle before, max over ranks).
* `roofline`   : dominant kernel = lstm_layer_kernel on the 2400-wide layers.  achieved = algorithmic FLOPs per launch
                 (2*256*2400*9600 per batch-step x 512 steps x batches in the launch) / launch duration from CUDA events
                 recorded inside ie_encoder_encode around it (ie_encoder_last_phase_ms; average of the three 2400-wide
                 layers of the last timed call).  peak = MEASURED_PEAKS.json bf16_tflops_sustained.
* `cpu_baseline`: the CPU oracle (oracle/awd_lstm_ref.py, torch nn.LSTM fp32 == the modules the reference's fastai
                 model wraps) timed on this box's host cores on a bounded sample (>= 32 issues).
* `--impl reference`: times that CPU path alone (the reference's own encoder is not installable: fastai/spaCy absent,
                 no network -- see DESIGN.md); each step is a bounded sample (>= 32 issues) of the same workload.
* `extra`      : fp32-accurate mode (IE_CFG_FP32), the north star's literal 3-layer shape (N3), the device-resident MLP
                 head (configs[4]) and a var-len bulk run checked bit for bit against a single-GPU encode.

`--dump-outputs DIR` writes, after the timed steps, what the timed paths handed back (float32 .npy, 12 MB on one GPU),
so that two builds can be compared output for output; inputs and weights are seeded, so the same arguments give the
same inputs:
* `embeddings.npy`            : the (256, 2400) result of the last timed step of `value` (with G ranks: that step of
                                every rank, rank-major; above 2048 rows a fixed seeded sample of them)
* `e2e_embeddings_sample.npy` : rows of the (N, 2400) array `e2e`'s bulk call returned, a fixed seeded sample of at most
                                1024 rows in ascending row order
* `reference_embeddings.npy`  : under `--impl reference`, the first 32 rows of the last timed step (how many issues
                                that arm encodes per step depends on a host-speed probe; the ids of its first rows do not)
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

B, T = 256, 512
N_LAYERS, EMB, HID, VOCAB = 4, 800, 2400, 60000


def flop_per_token(n_layers=N_LAYERS):
    dims = [((EMB if l == 0 else HID), (HID if l != n_layers - 1 else EMB)) for l in range(n_layers)]
    return 2 * sum(4 * o * (i + o) for i, o in dims)     # R4: 266.24e6, N3: 174.08e6 (SURVEY.md section 8d)


FLOP_PER_TOKEN = flop_per_token()
STEP_FLOP_2400 = 2.0 * B * 2400 * 9600   # one recurrent step of one 2400-wide layer, one batch of 256


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.p = gpu_index, [], None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        time.sleep(0.05)
        return self.summarise(self.rows)

    @staticmethod
    def summarise(rows):
        """Median SM clock and board power over the samples taken UNDER LOAD (power >= 60 % of the highest sample: the
        sampler also sees the idle gaps between the arms, where the clock sits at its maximum)."""
        samples, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                clk, cmax = float(r[1]), float(r[2])
            except Exception:
                continue
            try:
                pw = float(r[3])
            except Exception:
                pw = None
            samples.append((clk, pw))
            mx.append(cmax)
            for nm, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        powers = [pw for _, pw in samples if pw is not None]
        if powers:
            thr = 0.6 * max(powers)
            loaded = [(c, pw) for c, pw in samples if pw is not None and pw >= thr]
        else:
            loaded = samples
        clks = sorted(c for c, _ in loaded)
        pws = sorted(pw for _, pw in loaded if pw is not None)
        return {"sm_mhz": (clks[len(clks) // 2] if clks else None), "sm_max_mhz": (max(mx) if mx else None),
                "reasons": sorted(reasons), "samples": len(samples), "samples_under_load": len(loaded),
                "power_w": (pws[len(pws) // 2] if pws else None), "power_w_max": (max(powers) if powers else None)}


def usable_cpus():
    """Host cores this process may actually use: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(p) + 0.5)))
    except Exception:
        pass
    return max(1, n)


CPU_SAMPLE_MIN = 32   # issues per CPU sample: fewer under-feed the BLAS threads (round-1 verdict: 7 issues -> 2x too slow)


def cpu_oracle_setup():
    """Build the CPU oracle encoder and pick the torch thread count that maximises its throughput on this box
    (more threads than usable cores makes it slower).  The probe has the shape of the real sample (32 issues) at a
    quarter of the length."""
    import numpy as np
    import torch
    from oracle import awd_lstm_ref as R
    enc = R.make_encoder(1234, VOCAB, EMB, HID, N_LAYERS)
    cores = usable_cpus()
    probe = np.stack(R.synthetic_ids(CPU_SAMPLE_MIN, 128, seed=1))
    best = (0.0, 1)
    cands = sorted({c for c in (cores, cores // 2, 32, 16, 8) if 1 <= c <= cores}, reverse=True)
    for th in cands:
        torch.set_num_threads(th)
        R.encode_padded(enc, probe[:8, :32], [32] * 8)   # warm the thread pool
        t0 = time.perf_counter()
        R.encode_padded(enc, probe, [128] * CPU_SAMPLE_MIN)
        rate = CPU_SAMPLE_MIN * 128 / (time.perf_counter() - t0)
        if rate > best[0]:
            best = (rate, th)
    torch.set_num_threads(best[1])
    return enc, best[1], best[0], cores


DUMP_MAX_BYTES = 64 << 20


def sample_rows(a, max_rows, seed=0):
    """A copy of `a` if it has at most `max_rows` rows, else a fixed seeded sample of them in ascending row order."""
    import numpy as np
    if a.shape[0] <= max_rows:
        return np.array(a)
    return a[np.sort(np.random.default_rng(seed).choice(a.shape[0], size=max_rows, replace=False))]


def dump_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy in float32."""
    import numpy as np
    arrays = {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    assert total <= DUMP_MAX_BYTES, f"{total} bytes of outputs exceed the {DUMP_MAX_BYTES}-byte dump limit"
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def cpu_sample_size(tok_rate, budget_s):
    return int(max(CPU_SAMPLE_MIN, min(B, tok_rate * budget_s / T)))


def cpu_oracle_rate(budget_s=20.0):
    """issues/s of the CPU oracle on a bounded sample (>= 32 issues, about `budget_s` seconds) of the step's workload."""
    import numpy as np
    from oracle import awd_lstm_ref as R
    enc, threads, tok_rate, cores = cpu_oracle_setup()
    sb = cpu_sample_size(tok_rate, budget_s)
    ids = np.stack(R.synthetic_ids(sb, T, seed=2))
    t0 = time.perf_counter()
    out = R.encode_padded(enc, ids, [T] * sb)
    dt = time.perf_counter() - t0
    assert out.shape == (sb, 3 * EMB)
    return sb / dt, dt, threads, cores, sb


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port) on this box's host cores, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np
    from oracle import awd_lstm_ref as R
    enc, threads, tok_rate, cores = cpu_oracle_setup()
    budget = 150.0 / max(1, args.steps + args.warmup)          # whole run within a few minutes
    sb = cpu_sample_size(tok_rate, budget)
    ids = np.stack(R.synthetic_ids(sb, T, seed=3))
    for _ in range(args.warmup):
        R.encode_padded(enc, ids, [T] * sb)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = R.encode_padded(enc, ids, [T] * sb)
    dt = time.perf_counter() - t0
    val = sb * args.steps / dt
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"reference_embeddings": out[:CPU_SAMPLE_MIN]})
    sample = (f"{sb} of the {B} issues of a step (seq_len {T}), torch fp32 nn.LSTM oracle, {threads} threads "
              f"(best of a thread-count probe; {cores} usable cores)")
    print(json.dumps({
        "impl": "reference", "metric": "issues/sec to 2400-d @ seq_len 512 batch 256", "value": val, "unit": "issues/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1]: R4 encoder, seq_len 512, batch 256 (CPU arm: bounded sample per step)",
                   "sample_issues_per_step": sb},
        "cpu_baseline": {"value": val, "unit": "issues/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "issues/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=15)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what they computed as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from code_intelligence_b200 import IssueEncoder, bulk
    from oracle import awd_lstm_ref as R   # weights + synthetic ids generator + cpu_baseline leg only

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    K, W = args.steps, max(args.warmup, 3)

    ref = R.make_encoder(1234, VOCAB, EMB, HID, N_LAYERS)
    emb, layers = ref.export_weights()
    enc = IssueEncoder(N_LAYERS, EMB, HID, VOCAB, 1, local).load_weights(emb, layers)
    del ref

    # distinct synthetic ids per step and per rank, resident in HBM for the `value` arm
    g = torch.Generator().manual_seed(1234 + rank)
    ids_all = torch.randint(0, VOCAB, (K + W, B, T), generator=g, dtype=torch.int64)
    ids_all[ids_all == 1] = 0
    ids_all[:, :, 0] = 2
    ids_dev = ids_all.to(dev)
    out_dev = torch.empty((K * B, 3 * EMB), dtype=torch.float32, device=dev)
    gathered = torch.empty((world * K * B, 3 * EMB), dtype=torch.float32, device=dev) if world > 1 else None
    stream = torch.cuda.current_stream(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- launch plan: steps are submitted kPerLaunch at a time (5 x 256 rows per ie_encoder_encode call) ----------
    kPerLaunch = max(1, enc.max_batch // B)
    def plan(first, count, per_launch):
        # a remainder launch (count % per_launch steps) goes first, so that the LAST launch of a region -- whose
        # phase events feed the roofline -- is a full one
        out, i = [], first
        r = count % per_launch
        if r:
            out.append((i, r))
            i += r
        while i < first + count:
            out.append((i, per_launch))
            i += per_launch
        return out

    ids_flat_dev = ids_dev.view((K + W) * B, T)
    len_dev2 = torch.full((kPerLaunch * B,), T, dtype=torch.int32, device=dev)

    def run_device(first, count, per_launch):
        for (i, n) in plan(first, count, per_launch):
            enc.encode_ids_device(ids_flat_dev[i * B:(i + n) * B], len_dev2[:n * B],
                                  out_dev[(i - W) * B:(i - W + n) * B] if i >= W else out_dev[:n * B], stream)

    preroll_s = float(os.environ.get("BENCH_PREROLL_S", "2.0"))

    def device_arm(per_launch):
        run_device(0, W, per_launch)
        torch.cuda.synchronize(dev)
        t_pre = time.perf_counter()
        while time.perf_counter() - t_pre < preroll_s:    # same W warm-up steps again: power / clock steady state
            run_device(0, W, per_launch)
            torch.cuda.synchronize(dev)
        barrier()
        l0 = enc.launch_count
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        run_device(W, K, per_launch)
        if world > 1:
            dist.all_gather_into_tensor(gathered, out_dev)          # the single collective of the bulk path
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        enc.check_errors()
        t_ms = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
        return float(t_ms.item()), enc.launch_count - l0, enc.last_phase_ms(), enc.last_phase_mhz()

    # ---- device-resident arm ------------------------------------------------------------------------
    sampler = ClockSampler(local)
    ms_single, _, _, _ = device_arm(1)               # one batch per launch (reported as `single_batch`)
    if rank == 0:
        sampler.start()
    ms_max, launches, phases, phase_mhz = device_arm(kPerLaunch)   # five batches per launch: the bulk-encode mode
    value = world * B * K / (ms_max * 1e-3)
    single_value = world * B * K / (ms_single * 1e-3)
    dumps = {}
    if args.dump_outputs and rank == 0:
        last = gathered.view(world, K, B, 3 * EMB)[:, K - 1] if world > 1 else out_dev[(K - 1) * B:]
        dumps["embeddings"] = sample_rows(last.reshape(-1, 3 * EMB).cpu().numpy(), 2048)

    # ---- end-to-end arm: HOST token-id lists through the public bulk API -----------------------------------
    # every rank holds the same global list (the reference's per-repo list of numericalised issues), as the API expects
    n_total = world * K * B
    rng = np.random.default_rng(4321)
    def make_docs(n, seed_rng):
        a = seed_rng.integers(0, VOCAB, size=(n, T), dtype=np.int64)
        a[a == 1] = 0
        a[:, 0] = 2
        return list(a)
    docs_warm = make_docs(n_total, rng)      # same shape as the timed call: buffers of the right size exist afterwards
    docs = make_docs(n_total, rng)
    local_fn = lambda d: bulk.encode_sorted_batches_device(d, enc, min_batches_rule=False, to_host=False)
    bulk.encode_bulk_distributed(docs_warm, local_fn, device=dev, to_host="rank0")
    barrier()
    t0 = time.perf_counter()
    res = bulk.encode_bulk_distributed(docs, local_fn, device=dev, to_host="rank0")   # rank 0: np.ndarray (n_total, 2400)
    if rank != 0:
        torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - t0
    assert tuple(res.shape) == (n_total, 3 * EMB)
    if rank == 0:
        assert isinstance(res, np.ndarray) and np.isfinite(res[::97]).all()
        if args.dump_outputs:
            dumps["e2e_embeddings_sample"] = sample_rows(res, 1024)
    t_e2e = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    e2e_value = n_total / float(t_e2e.item())
    clocks = sampler.stop() if rank == 0 else None
    # where the end-to-end time goes (a second, diagnostic repetition on this rank's shard; not part of `e2e.value`)
    e2e_breakdown = None
    del res                      # hands its page-locked block back to torch's cache (the repetition below reuses it)
    if world == 1:
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        loc = local_fn(docs)
        torch.cuda.synchronize(dev)
        t1 = time.perf_counter()
        host = bulk._to_numpy(loc)     # what the API does: D2H through torch's cached page-locked allocator
        t2 = time.perf_counter()
        e2e_breakdown = {"pack_h2d_encode_unsort_ms": (t1 - t0) * 1e3, "d2h_result_ms": (t2 - t1) * 1e3,
                         "device_only_ms_for_same_steps": ms_max}
        del loc, host

    # ---- extras (rank 0 reports; all ranks take part where a collective is involved) ---------------------------
    extra = {}
    if not args.no_extra:
        # var-len bulk encode, strong scaling: a FIXED list, sharded over the ranks, checked bit for bit against rank 0
        # encoding the whole list alone
        nv = 5120
        rv = np.random.default_rng(99)
        lens = rv.integers(64, T + 1, size=nv)
        vdocs = []
        for L in lens:
            a = rv.integers(0, VOCAB, size=int(L), dtype=np.int64)
            a[a == 1] = 0
            a[0] = 2
            vdocs.append(a)
        bulk.encode_bulk_distributed(vdocs[:world * 256], local_fn, device=dev)
        barrier()
        t0 = time.perf_counter()
        vres = bulk.encode_bulk_distributed(vdocs, local_fn, device=dev)
        vs = time.perf_counter() - t0
        t_v = torch.tensor([vs], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t_v, op=dist.ReduceOp.MAX)
        if rank == 0:
            alone = enc.encode_id_list(vdocs, min_batches_rule=False)
            extra["bulk_varlen"] = {"issues": nv, "lengths": "uniform in [64, 512]", "valid_tokens": int(lens.sum()),
                                    "value": nv / float(t_v.item()), "unit": "issues/s", "scaling": "strong",
                                    "valid_tokens_per_s": float(lens.sum()) / float(t_v.item()),
                                    "bit_equal_to_single_gpu": bool(np.array_equal(vres, alone))}
        barrier()
    if rank == 0 and not args.no_extra:
        try:
            extra.update(extras_rank0(enc, emb, layers, dev, R))
        except Exception as e:   # extras never take the headline down
            extra["error"] = repr(e)

    if rank == 0:
        peaks = measured_peaks()
        peak = (peaks or {}).get("bf16_tflops_sustained", 1400.0)
        peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else "fallback 1.4 PFLOP/s sustained"
        batches = kPerLaunch if K >= kPerLaunch else K   # batches riding the LAST timed launch (see plan())
        step_ms = phases["steps"][:N_LAYERS - 1]
        avg_launch_ms = sum(step_ms) / len(step_ms)
        flop_per_launch = STEP_FLOP_2400 * T * batches
        achieved = flop_per_launch / (avg_launch_ms * 1e-3) / 1e12
        traffic, traffic_src = None, None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "lstm_layer_traffic.json")))
            traffic, traffic_src = tj["dram_bytes_per_launch"], tj.get("source")
        except Exception:
            pass
        line = {
            "metric": "issues/sec to 2400-d @ seq_len 512 batch 256", "value": value, "unit": "issues/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_max / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "configs[1]: 1M-issue bulk encode shape, fixed seq_len 512, batch 256 per step, "
                                   "R4 encoder (L=4,E=800,H=2400,V=60000) random-init seed 1234",
                       "batch": B, "seq_len": T, "batches_per_launch": kPerLaunch, "preroll_s": preroll_s,
                       "parallelism": f"dp{world} (issues sharded, one all-gather of outputs)",
                       "l2": "inputs larger than L2: each step streams ~3 GB of workspace (bf16 Gx, hidden-state rings) "
                             "and new ids",
                       "operands": "bf16 weights/activations/Gx, f32 accumulate, f32 cell state and pooling"},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "issues/s", "h2d_bytes_per_step": B * T * 8 + B * 4,
                    "d2h_bytes_per_step": world * B * 3 * EMB * 4,
                    "api": "bulk.encode_bulk_distributed(host id lists) -> np.ndarray (N, 2400) on rank 0",
                    "note": "host packing and H2D run under the previous batch's kernels and the result leaves through "
                            "page-locked memory, so e2e tracks `value` to within the +-2 % clock variation between the two "
                            "arms (it can land on either side)",
                    "breakdown_ms": e2e_breakdown},
            "single_batch": {"value": single_value, "unit": "issues/s", "ms_per_step": ms_single / K,
                             "note": "same measurement with one batch of 256 per launch"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "kernel": "lstm_layer_kernel (persistent recurrent kernel, 2400-wide layers, "
                                   "%d batches in the last timed launch)" % batches,
                         "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "avg_launch_us": avg_launch_ms * 1e3, "flop_per_launch": flop_per_launch,
                         "whole_step_tflops": FLOP_PER_TOKEN * B * T / (ms_max / K * 1e-3) / 1e12,
                         "whole_step_frac": FLOP_PER_TOKEN * B * T / (ms_max / K * 1e-3) / 1e12 / peak,
                         "phase_ms_last_call": phases, "phase_sm_mhz": {k: [round(x) for x in v] for k, v in phase_mhz.items()}},
            "extra": extra,
        }
        if world == 1 and not args.no_cpu_baseline:
            rate, dt, threads, cores, sb = cpu_oracle_rate()
            line["cpu_baseline"] = {"value": rate, "unit": "issues/s", "cores": threads, "kind": "port",
                                    "sample": f"{sb} issues x seq_len {T} ({sb}/{B} of a step), torch fp32 nn.LSTM "
                                              f"oracle, {threads} threads of {cores} usable cores, {dt:.1f} s"}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dumps)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def extras_rank0(enc, emb, layers, dev, R):
    """Secondary measurements on one GPU (device-resident inputs, CUDA events, after a warm-up call each)."""
    import numpy as np
    import torch
    from code_intelligence_b200 import IssueEncoder, _lib
    from code_intelligence_b200.mlp import MLPHead
    out = {}
    g = torch.Generator().manual_seed(7)

    def time_encoder(e, rows, iters, flop_tok):
        ids = torch.randint(2, VOCAB, (rows, T), generator=g, dtype=torch.int64).to(dev)
        lens = torch.full((rows,), T, dtype=torch.int32, device=dev)
        o = torch.empty((rows, 3 * EMB), dtype=torch.float32, device=dev)
        e.encode_ids_device(ids, lens, o)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            e.encode_ids_device(ids, lens, o)
        e1.record()
        torch.cuda.synchronize(dev)
        e.check_errors()
        ms = e0.elapsed_time(e1) / iters
        return {"value": rows / ms * 1e3, "unit": "issues/s", "rows_per_call": rows, "ms_per_256": ms * 256 / rows,
                "tflops": flop_tok * rows * T / ms / 1e9}

    # the reference's online entry (flask_app /text, Issue_Embeddings/flask_app/app.py:49-76): ONE issue per call.  Latency of
    # ie_encoder_encode with B = 1 (device-resident ids; the recurrence is a chain of T x L dependent steps, so this is a
    # latency figure, not a throughput one)
    lat = {}
    for t_len in (128, 512):
        ids1 = torch.randint(2, VOCAB, (1, t_len), generator=g, dtype=torch.int64).to(dev)
        len1 = torch.full((1,), t_len, dtype=torch.int32, device=dev)
        o1 = torch.empty((1, 3 * EMB), dtype=torch.float32, device=dev)
        for _ in range(2):
            enc.encode_ids_device(ids1, len1, o1)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            enc.encode_ids_device(ids1, len1, o1)
        e1.record()
        torch.cuda.synchronize(dev)
        lat[f"T{t_len}_ms"] = e0.elapsed_time(e1) / 5
    lat["note"] = "one issue per call (the /text endpoint's shape), device-resident ids, mean of 5 calls"
    out["online_b1"] = lat
    # BASELINE configs[1] as written ("fp32"): split-bf16 products, f32 Gx, IEEE gates; parity in tests/test_gpu_parity.py
    e32 = IssueEncoder(N_LAYERS, EMB, HID, VOCAB, 1, dev.index, _lib.IE_CFG_FP32).load_weights(emb, layers)
    r = time_encoder(e32, e32.max_batch, 2, FLOP_PER_TOKEN)
    r["note"] = ("IE_CFG_FP32: every product as three bf16 tensor-core passes (hi*hi + lo*hi + hi*lo), f32 accumulate; "
                 "tflops counts the algorithmic (single-pass) FLOPs; rel-L2 vs the fp32 oracle <= 2e-5")
    out["fp32_mode"] = r
    e32.close()
    # the north star's literal 3-layer shape
    ref3 = R.make_encoder(1234, VOCAB, EMB, HID, 3)
    emb3, layers3 = ref3.export_weights()
    e3 = IssueEncoder(3, EMB, HID, VOCAB, 1, dev.index).load_weights(emb3, layers3)
    out["n3"] = time_encoder(e3, e3.max_batch, 3, flop_per_token(3))
    out["n3"]["note"] = "L=3 (800->2400->2400->800), same metric; 174.08 MFLOP/token"
    e3.close()
    # Label_Microservice head (configs[4]): (D_in -> 600 -> 600 -> 256), device-resident X, n = 2^20 rows
    rng = np.random.default_rng(0)
    for d_in in (1600, 2400):
        dims = [d_in, 600, 600, 256]
        coefs = [(rng.standard_normal((dims[i], dims[i + 1])) / np.sqrt(dims[i])).astype(np.float32) for i in range(3)]
        ints = [(rng.standard_normal(dims[i + 1]) * 0.1).astype(np.float32) for i in range(3)]
        head = MLPHead(coefs, ints, device=dev.index)
        n = 1 << 20
        X = torch.randn((n, d_in), generator=g).mul_(0.1).to(dev)
        P = torch.empty((n, 256), dtype=torch.float32, device=dev)
        head.predict_proba_device(X, P)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            head.predict_proba_device(X, P)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / 3
        flop = 2.0 * n * (d_in * 600 + 600 * 600 + 600 * 256)
        byt = n * (d_in * 4 + 256 * 4)
        peaks = measured_peaks() or {}
        hbm = peaks.get("hbm_gbs", 6500.0)
        tf = peaks.get("bf16_tflops_sustained", 1400.0)
        t_hbm, t_tensor = byt / hbm / 1e6, flop / tf / 1e9          # ms at the measured peaks
        # the binding roofline is the slower of the two: at D_in >= 1600 the three bf16 GEMMs (tensor) outlast the
        # f32 X read + probability write (HBM)
        if t_tensor >= t_hbm:
            roof = {"bound": "tensor", "achieved": flop / ms / 1e9, "peak": tf, "unit": "TFLOP/s", "frac": t_tensor / ms}
        else:
            roof = {"bound": "hbm", "achieved": byt / ms / 1e6, "peak": hbm, "unit": "GB/s", "frac": t_hbm / ms}
        roof["hbm_frac"] = t_hbm / ms
        roof["note"] = ("algorithmic FLOPs 2 n (D_in 600 + 600 600 + 600 256); algorithmic bytes = f32 X in + f32 "
                        "probabilities out; peaks from MEASURED_PEAKS.json")
        out[f"mlp_{d_in}"] = {"rows_per_s": n / ms * 1e3, "labels_per_s": n * 256 / ms * 1e3, "ms": ms,
                              "tflops": flop / ms / 1e9, "hbm_gbs": byt / ms / 1e6, "roofline": roof}
        head.close()
    return out


if __name__ == "__main__":
    main()
