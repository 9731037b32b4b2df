#!/usr/bin/env python
"""bench.py -- Score() prompts/sec @4K tokens against a 10M-block / 256-pod index (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path (GetPodScores steps 2-4, pkg/kvcache/indexer.go:141-163) over one
batch of synthetic 4096-token prompts.  --steps sets the number of timed steps of `value`.

--dump-outputs DIR writes what the last timed step returned to its caller, as .npy files: scores.npy (dense
score rows, float64), has_keys.npy (float32) and prompt_index.npy (which prompts of the batch the rows belong to,
float64).  Batches above 16 K prompts are sampled (fixed seed, 32 MiB of rows).  The inputs depend only on the
arguments, so the files of two builds can be compared one to one.  Rank 0 writes its own batch.

  value     whole-job prompts/s with the batch already resident in HBM (kvidx_score_batch_dev)
  e2e       the same metric through the host-buffer C-ABI call (kvidx_score_batch): pinned host tokens
            -> H2D -> kernel -> D2H dense score rows, copies inside the timed region
  roofline  algorithmic bytes (SURVEY.md 8(d): A = 4T + 32*n_probe + 8P per prompt) / kernel time, against
            the measured HBM copy bandwidth in MEASURED_PEAKS.json
  cpu_baseline  the C++ restatement of the reference's Go path (oracle/, kind "port") on this box's host cores,
            on a bounded sample of the same prompts against the same 10M-block index

Multi-GPU (torchrun, one rank per GPU), "scaling": "weak" (every rank scores its own resident batch):
  value           hash-range SHARDED index (the north-star layout): tables partitioned over the ranks, probes and slot
                  updates over NVLink peer memory from the scoring kernels themselves
  value_replicas  every rank holds the full index, no exchange
  config4         (N = 8) BASELINE config #4: 100 M-block index sharded over the 8 GPUs
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "llm-d-kv-cache-manager_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

# "metric row" of SURVEY 8(d): T=4K, N=10M, P=256.  The other BASELINE configs run through the same script:
#   #3  KVIDX_BENCH_TOKENS=8192                      #4  KVIDX_BENCH_BLOCKS=100000000 KVIDX_BENCH_MODE=sharded --gpus 8
T_TOKENS = int(os.environ.get("KVIDX_BENCH_TOKENS", "4096"))
N_BLOCKS = int(os.environ.get("KVIDX_BENCH_BLOCKS", "10000000"))
N_PODS, BLOCK = 256, 16
CONFIG_ID = 6
WEIGHTS = (1.0, 0.8)


def log(*a):
    if int(os.environ.get("RANK", "0")) == 0:
        print(*a, file=sys.stderr, flush=True)


# ----------------------------------------------------------------------------------------------
# synthetic data on the device (same SplitMix64 counter streams as kvidx/synth.py, in torch int64)
# ----------------------------------------------------------------------------------------------
def _i64(v):
    v &= (1 << 64) - 1
    return v - (1 << 64) if v >= (1 << 63) else v


def t_mix(z):
    import torch
    def lsr(x, k):
        return (x >> k) & ((1 << (64 - k)) - 1)
    z = (z ^ lsr(z, 30)) * _i64(0xBF58476D1CE4E5B9)
    z = (z ^ lsr(z, 27)) * _i64(0x94D049BB133111EB)
    return z ^ lsr(z, 31)


def t_stream(seed, start, count, device):
    import torch
    idx = torch.arange(start + 1, start + count + 1, dtype=torch.int64, device=device)
    return t_mix(idx * _i64(0x9E3779B97F4A7C15) + _i64(seed))


def t_umod(z, m):
    """unsigned (z as uint64) mod m for int64 tensors."""
    import torch
    r = torch.remainder(z, m)
    return torch.where(z < 0, torch.remainder(r + ((1 << 64) % m), m), r)


def device_queries(wl, q0, q1, device, full_depth=False, chunk=8192):
    """tokens (nq, T) int32 on `device`, plus host arrays doc, m (the generator of synth.Workload.queries)."""
    import torch
    nq = q1 - q0
    from kvidx import synth
    r = synth.stream(wl.s_q, q0 * 2, nq * 2).reshape(nq, 2)
    doc = (r[:, 0] % np.uint64(wl.D)).astype(np.int64)
    m = (r[:, 1] % np.uint64(wl.n + 1)).astype(np.int64)
    if full_depth:
        m[:] = wl.n
    out = torch.empty((nq, wl.T), dtype=torch.int32, device=device)
    col = torch.arange(wl.T, dtype=torch.int64, device=device)[None, :]
    for c0 in range(0, nq, chunk):
        c1 = min(nq, c0 + chunk)
        tail = t_umod(t_stream(wl.s_tail, (q0 + c0) * wl.T, (c1 - c0) * wl.T, device), wl.vocab).view(c1 - c0, wl.T)
        d = torch.from_numpy(doc[c0:c1]).to(device)[:, None]
        idx = d * wl.T + col + 1
        dtok = t_umod(t_mix(idx * _i64(0x9E3779B97F4A7C15) + _i64(wl.s_doc)), wl.vocab)
        mm = torch.from_numpy(m[c0:c1]).to(device)[:, None] * wl.B
        out[c0:c1] = torch.where(col < mm, dtok, tail).to(torch.int32)
    return out, doc, m


DUMP_ROWS = 16384          # 16 K dense rows of 256 float64 scores = 32 MiB


def dump_rows(n):
    """Prompts of an n-prompt batch that --dump-outputs writes: all of them up to DUMP_ROWS, else a fixed seeded sample."""
    if n <= DUMP_ROWS:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))


def dump_outputs(out_dir, rows, scores, has_keys):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("prompt_index", rows.astype(np.float64)), ("scores", np.asarray(scores, np.float64)),
                    ("has_keys", np.asarray(has_keys, np.float32))):
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log("[dump] %d score rows of the last timed step -> %s" % (len(rows), out_dir))


def algorithmic_bytes(wl, m):
    """SURVEY.md 8(d): A = 4T + 32*n_probe + 8P, n_probe = min(n, depth_of_last_active_pod + 1)."""
    n_probe = np.minimum(wl.n, m + 1)
    return 4 * wl.T + 32 * n_probe + 8 * wl.P


# ----------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        self.join(timeout=2)
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """DRAM bytes (read+write) per prompt of one default Score() step from the committed ncu captures: the range profile of the
    whole step (profiles/r2_step_range_profile.json, `ncu --replay-mode range --set full`, its kernels as one unit), else the sum
    over the per-kernel launch list (profiles/score_step_traffic.json); None if neither is committed."""
    try:
        m = json.load(open(os.path.join(ROOT, "profiles", "r2_step_range_profile.json")))["metrics"]
        unit = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
        tot = sum(float(m[k]["value"]) * unit[m[k]["unit"]] for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"))
        return tot / 1048576.0
    except Exception:
        pass
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "score_step_traffic.json")))["dram_bytes_per_prompt"]
    except Exception:
        return None


# ----------------------------------------------------------------------------------------------
def build_cpu_oracle(wl, n_docs=None):
    """The reference-path port on the host: same events, same index."""
    from oracle.kvoracle_c import COracle
    co = COracle(block_size=BLOCK, size=10 ** 8, pod_cache_size=10, tier_weights=WEIGHTS, max_pods=wl.P)
    D = wl.D if n_docs is None else n_docs
    t0 = time.time()
    for d0 in range(0, D, 2048):
        ev, hs, tk = wl.fill_events(d0, min(D, d0 + 2048))
        rc, dropped = co.apply_events(ev, hs, tk)
        assert rc == 0 and dropped == 0
    return co, time.time() - t0


def best_threads(co, tok, off, ns, wl):
    """The reference serialises on the global mutex inside lru.Cache.Get (in_memory.go:118), so more threads is
    not faster; time a short probe at several thread counts and keep the best one for the reported sample."""
    cand = sorted({1, 2, 4, 8, 16, host_threads()})
    cand = [c for c in cand if c <= host_threads()]
    probe = min(ns, 1024)
    best, best_v = 1, 0.0
    for c in cand:
        _, _, el, _ = co.score_batch(tok[: probe * wl.T], off[: probe + 1], n_threads=c, want_scores=False)
        if probe / el > best_v:
            best, best_v = c, probe / el
    ref_s, _, el, l = co.score_batch(tok[: ns * wl.T], off[: ns + 1], n_threads=best, want_latency=True)
    return best, el, l, ref_s


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port; Go cannot be built in
    this image), all host threads, same config / metric / unit."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from kvidx import synth
    wl = synth.Workload(CONFIG_ID, T_TOKENS, N_BLOCKS, N_PODS, BLOCK)
    log("[reference] building %d-block index on the host ..." % wl.n_blocks)
    co, fill_s = build_cpu_oracle(wl)
    sample = int(os.environ.get("KVIDX_REF_SAMPLE", "4096"))
    ptok, _, _ = wl.queries(10 ** 7, 10 ** 7 + 1024)
    threads, _, _, _ = best_threads(co, ptok.reshape(-1), np.arange(0, 1025 * wl.T, wl.T, dtype=np.int64), 1024, wl)
    times = []
    lat = []
    q = 0
    for step in range(args.warmup + args.steps):
        toks, doc, m = wl.queries(q, q + sample)
        q += sample
        off = np.arange(0, (sample + 1) * wl.T, wl.T, dtype=np.int64)
        scores, has, el, l = co.score_batch(toks.reshape(-1), off, n_threads=threads, want_scores=True, want_latency=True)
        if step >= args.warmup:
            times.append(el)
            lat.append(l)
    if args.dump_outputs:
        rows = dump_rows(sample)
        dump_outputs(args.dump_outputs, rows, scores[rows], has[rows])
    total = sum(times)
    value = sample * len(times) / total
    lat = np.concatenate(lat)
    out = {"metric": "score_prompts_per_sec", "value": value, "unit": "prompts/s", "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "u64", "data": "synthetic", "impl": "reference",
           "config": {"workload": "Score() %d-token prompts, %s-block / 256-pod index (SURVEY 8(d) %s)" % (
                              T_TOKENS, "%dM" % round(N_BLOCKS / 1e6), "metric row" if (T_TOKENS, N_BLOCKS) == (4096, 10_000_000) else "config variant"),
                      "prompt_tokens": wl.T, "index_blocks": wl.n_blocks, "pods": wl.P, "block_size": BLOCK,
                      "batch_prompts": sample, "query_mix": "m uniform in [0,n] matched blocks + random tail"},
           "cpu_baseline": {"value": value, "unit": "prompts/s", "cores": threads, "kind": "port",
                            "sample": "%d steps x %d prompts, one GetPodScores per call on %d threads (best of a 1..%d sweep; C++ restatement "
                                      "of the Go path; Go toolchain absent); index fill %.1fs" % (len(times), sample, threads, host_threads(), fill_s),
                            "host_cores": host_threads(),
                            "p99_latency_ms": float(np.percentile(lat, 99)) / 1e6, "p50_latency_ms": float(np.percentile(lat, 50)) / 1e6,
                            "go_probe": go_probe()},
           "e2e": {"value": value, "unit": "prompts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    emit(out)


# ----------------------------------------------------------------------------------------------
def go_probe():
    """SURVEY 8(d): "probe at run time, never assume".  If a Go toolchain AND the module the hash depends on
    (fxamacker/cbor/v2 v2.7.0) are on this box, oracle/goprobe runs the reference's own hash call shape
    (token_processor.go:94-112) over tests/golden/hash_kats.json and the result is recorded; otherwise the reason is."""
    import shutil
    import tempfile
    go = shutil.which("go")
    if not go:
        return {"go": None, "pinned": False, "why": "no go toolchain on this box"}
    try:
        ver = subprocess.run([go, "version"], capture_output=True, text=True, timeout=20).stdout.strip()
        env = dict(os.environ, GOFLAGS="-mod=mod", GOPROXY="off", GOTOOLCHAIN="local")
        with tempfile.TemporaryDirectory() as tmp:          # -mod=mod may write go.sum: run a copy, not the tree
            probe = shutil.copytree(os.path.join(ROOT, "oracle", "goprobe"), os.path.join(tmp, "goprobe"))
            r = subprocess.run([go, "run", "."], cwd=probe, capture_output=True, text=True, timeout=120, env=env,
                               input=open(os.path.join(ROOT, "tests", "golden", "hash_kats.json")).read())
        if r.returncode != 0:
            return {"go": ver, "pinned": False, "why": "go run failed (module cache without fxamacker/cbor?): " + r.stderr.strip()[-200:]}
        res = json.loads(r.stdout)
        return {"go": ver, "pinned": bool(res.get("all_equal")), "cases": res.get("cases"), "mismatches": res.get("mismatches")}
    except Exception as e:      # noqa: BLE001
        return {"go": go, "pinned": False, "why": repr(e)[:200]}


def h2d_peak_gbs(dev):
    """Measured pinned host -> device copy bandwidth of this rank (1 GiB, best of 5): the bound of the e2e number."""
    import torch
    n = 1 << 30
    h = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    h.fill_(1)
    d = torch.empty(n, dtype=torch.uint8, device=dev)
    best = 0.0
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); d.copy_(h, non_blocking=True); e1.record(); e1.synchronize()
        best = max(best, n / (e0.elapsed_time(e1) / 1e3) / 1e9)
    del h, d
    return best


def run_ours(args):
    import torch
    import torch.distributed as dist
    import kvidx
    from kvidx import synth
    from kvidx import dist as kd
    from kvidx.numa import pin_to_gpu_numa

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    numa = pin_to_gpu_numa(local) if not os.environ.get("KVIDX_BENCH_NO_NUMA") else {"pinned": False, "note": "disabled"}
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def all_ok(flag):
        if world == 1:
            return bool(flag)
        t = torch.tensor([1 if flag else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item())

    def max_ranks(v):
        if world == 1:
            return float(v)
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    wl = synth.Workload(CONFIG_ID, T_TOKENS, N_BLOCKS, N_PODS, BLOCK)
    Q = int(os.environ.get("KVIDX_BENCH_BATCH", str(1048576)))      # prompts resident in HBM per step (per GPU)
    QE = int(os.environ.get("KVIDX_BENCH_E2E_BATCH", str(65536)))  # prompts per e2e step (host buffers)
    nocheck = bool(os.environ.get("KVIDX_BENCH_NOCHECK"))          # timing experiments with ablated kernels only

    # ---- index: filled through the write path (BlockStored events) ----
    #   sharded  : the north-star layout -- request / engine tables hash-range sharded over the ranks; every rank maps its
    #              peers' shards (CUDA IPC, one 192-byte all_gather) and probes / updates them through NVLink peer memory from
    #              the same kernels; each rank ingests the events of its own pods (pod % world == rank).  `value` at N > 1.
    #   replicas : every rank holds the full index, prompts are sharded, no exchange at all.  `value_replicas` at N > 1.
    if world == 1:
        modes = ["single"]
    else:
        m_env = os.environ.get("KVIDX_BENCH_MODE", "both")
        modes = ["sharded", "replicas"] if m_env == "both" else [m_env]

    def build_index(mode, wlx):
        if mode == "sharded":
            ix = kvidx.Index(block_size=BLOCK, capacity=wlx.n_blocks + (1 << 20), max_pods=wlx.P, tier_weights=WEIGHTS, device=local,
                             shard_rank=rank, shard_count=world)
            kd.connect_shards(ix, dev)
        else:
            ix = kvidx.Index(block_size=BLOCK, capacity=wlx.n_blocks + (1 << 20), max_pods=wlx.P, tier_weights=WEIGHTS, device=local)
        t0 = time.time()
        n_ev = 0
        apply_s = 0.0                                    # time inside kvidx_apply_events (host arrays in, H2D + kernels), generation excluded
        for d0 in range(0, wlx.D, 4096):
            ev, hs, tk = wlx.fill_events(d0, min(wlx.D, d0 + 4096))
            if mode == "sharded":
                ev = kd.events_for_rank(ev, rank, world)
            ta = time.perf_counter()
            rc, dropped = ix.apply_events(ev, hs, tk)
            apply_s += time.perf_counter() - ta
            assert rc == 0 and dropped == 0, (rc, dropped, ix.last_error())
            n_ev += len(ev)
        barrier()
        fill_s = time.time() - t0
        st = ix.stats()
        if mode == "sharded":
            tot = torch.tensor([st["request_keys"]], dtype=torch.int64, device=dev)
            dist.all_reduce(tot)
            assert int(tot.item()) == wlx.n_blocks, (int(tot.item()), wlx.n_blocks)
        else:
            assert st["request_keys"] == wlx.n_blocks, st
        log("[fill %s] %d BlockStored events -> %d request keys on this rank in %.1fs (host event generation included; %.2fs inside apply_events, %d events re-hashed)"
            % (mode, n_ev, st["request_keys"], fill_s, apply_s, st["rehashed_events"]))
        return ix, {"fill_s": fill_s, "apply_s": apply_s, "events": n_ev, "keys": st["request_keys"], "slots": st["request_slots"], "rehashed": st["rehashed_events"]}

    built = {m: build_index(m, wl) for m in modes}
    primary = modes[0]
    ix, fill = built[primary]

    # ---- device-resident batch (rank r scores its own slice of the query stream) ----
    q_base = rank * (Q + QE) * 4
    d_tok, doc, m = device_queries(wl, q_base, q_base + Q, dev)
    d_off = torch.arange(0, (Q + 1) * wl.T, wl.T, dtype=torch.int64, device=dev)
    d_scores = torch.empty((Q, wl.P), dtype=torch.float64, device=dev)
    d_has = torch.empty((Q,), dtype=torch.uint8, device=dev)
    stream = torch.cuda.Stream(device=dev)          # a real (non-default) stream: the library launches on it and
    torch.cuda.set_stream(stream)                   # the CUDA events below are recorded on it
    assert stream.cuda_stream != 0
    exp = wl.expected_scores(doc[:4096], m[:4096], WEIGHTS)

    def parity_gate(ixx, qs=None, what=""):
        """closed-form expectation of the generator (bit-exact f64) on 4096 prompts + the pod-count property on the whole
        batch, on EVERY rank; the run stops unless all ranks agree."""
        torch.cuda.synchronize()
        n = Q if qs is None else qs
        ok = np.array_equal(d_scores[:min(4096, n)].cpu().numpy(), exp[:min(4096, n)])
        ok = ok and np.array_equal((d_scores[:n] >= 0).sum(dim=1).cpu().numpy(), np.where(m[:n] > 0, 4, 0))
        ok = all_ok(ok or nocheck)
        assert ok, "score mismatch vs closed form (%s)" % what
        return True

    def measure(mode):
        ixx = built[mode][0]
        ixx.set_stream(stream.cuda_stream)

        def step():
            ixx.score_batch_dev(d_tok.data_ptr(), d_off.data_ptr(), Q, d_scores.data_ptr(), d_has_keys=d_has.data_ptr())
        d_scores.fill_(-7.0)
        step()
        parity_gate(ixx, what=mode)
        sampler = ClockSampler(local)
        sampler.start()                                  # started before the warm-up: nvidia-smi needs a moment (longer with N of them)
        for _ in range(max(args.warmup, 3)):
            step()
        # keep the GPU under the same load until the sampler has produced its first rows, so that the rows taken during and
        # around the (short) timed region are rows under load
        t_wait = time.time()
        while len(sampler.rows) < 2 and time.time() - t_wait < 8.0 and not os.environ.get("KVIDX_BENCH_QUICK"):
            step()
            torch.cuda.synchronize()
        barrier()
        launches0 = ixx.stats()["kernel_launches"]
        n_before = len(sampler.rows)
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        barrier()
        t_all0 = torch.cuda.Event(enable_timing=True); t_all1 = torch.cuda.Event(enable_timing=True)
        t_all0.record(stream)
        for a, b in evs:
            a.record(stream)
            step()
            b.record(stream)
        t_all1.record(stream)
        barrier()
        if args.dump_outputs and mode == primary and rank == 0:
            rows = dump_rows(Q)
            sel = torch.from_numpy(rows).to(dev)
            dump_outputs(args.dump_outputs, rows, d_scores.index_select(0, sel).cpu().numpy(), d_has.index_select(0, sel).cpu().numpy())
        launches = ixx.stats()["kernel_launches"] - launches0
        total_ms = max_ranks(t_all0.elapsed_time(t_all1))
        t_wait = time.time()
        while len(sampler.rows) < n_before + 2 and time.time() - t_wait < 3.0 and not os.environ.get("KVIDX_BENCH_QUICK"):      # a few more rows under the same load
            step()
            torch.cuda.synchronize()
        clocks = sampler.stop()
        step_ms = np.array([a.elapsed_time(b) for a, b in evs])
        return {"value": world * Q * args.steps / (total_ms / 1e3), "total_ms": total_ms, "step_ms": step_ms, "launches": int(launches),
                "clocks": clocks, "step": step}

    res = {mode: measure(mode) for mode in modes}
    R = res[primary]
    value, total_ms, step_ms, launches, clocks, step_dev = R["value"], R["total_ms"], R["step_ms"], R["launches"], R["clocks"], R["step"]
    if os.environ.get("KVIDX_BENCH_QUICK"):                       # profiling runs (ncu): the timed steps only
        if rank == 0:
            emit({"metric": "score_prompts_per_sec", "value": value, "unit": "prompts/s", "n_gpus": world, "steps": args.steps, "ms_per_step": total_ms / args.steps,
                  "gpu_launches": int(launches), "quick": True, "mode": primary, "fill": fill,
                  "value_replicas": res["replicas"]["value"] if "replicas" in res and primary != "replicas" else None})
        if world > 1:
            dist.destroy_process_group()
        return

    # smaller batches on the same resident data (fewer chains in flight, less prefix sharing per batch): the SURVEY's
    # "64K batch" regime and half a million prompts
    def sub_batch(qs):
        qs = min(Q, qs)
        def stp():
            ix.score_batch_dev(d_tok.data_ptr(), d_off.data_ptr(), qs, d_scores.data_ptr(), d_has_keys=d_has.data_ptr())
        for _ in range(3):
            stp()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(); e0.record(stream)
        for _ in range(5):
            stp()
        e1.record(stream); barrier()
        return world * qs * 5 / (max_ranks(e0.elapsed_time(e1)) / 1e3)
    value_64k = sub_batch(65536)
    value_512k = sub_batch(524288)

    # the same resident batch with the reference's RESULT SHAPE (<= 10 (pod, score) pairs per prompt, indexer.go:134) left on the
    # device instead of a dense double[P] row: 101 B instead of 2 KB written per prompt.  Extra information: `value` stays the
    # dense-row number the metric was defined on.
    value_sparse = None
    try:
        d_sp_pods = torch.empty((Q, 10), dtype=torch.int16, device=dev)
        d_sp_sc = torch.empty((Q, 10), dtype=torch.float64, device=dev)
        d_sp_cnt = torch.empty((Q,), dtype=torch.uint8, device=dev)
        def sstp():
            ix.score_batch_sparse_dev(d_tok.data_ptr(), d_off.data_ptr(), Q, d_sp_pods.data_ptr(), d_sp_sc.data_ptr(), d_sp_cnt.data_ptr(),
                                      d_has_keys=d_has.data_ptr())
        for _ in range(3):
            sstp()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(); e0.record(stream)
        for _ in range(5):
            sstp()
        e1.record(stream); barrier()
        ms_sp = max_ranks(e0.elapsed_time(e1)) / 5
        ns = 4096
        pods = d_sp_pods[:ns].cpu().numpy().view(np.uint16); scs = d_sp_sc[:ns].cpu().numpy(); cn = d_sp_cnt[:ns].cpu().numpy()
        dense = np.full((ns, N_PODS), -1.0)
        for i in range(ns):
            dense[i, pods[i, :cn[i]]] = scs[i, :cn[i]]
        value_sparse = {"value": world * Q / (ms_sp / 1e3), "unit": "prompts/s", "ms_per_step": ms_sp,
                        "parity": "closed form, first %d prompts" % ns if np.array_equal(dense, exp[:ns]) else "MISMATCH",
                        "note": "kvidx_score_batch_sparse_dev: the reference's result shape left in HBM (101 B per prompt instead of a 2 KB dense row)"}
    except Exception as ex:                                     # noqa: BLE001 -- an extra must never cost the bench line
        value_sparse = {"error": repr(ex)[:200]}

    # ---- the two ways to run a sharded Score(): peer-memory probes from the walk (what the library does) vs the routed form
    # of SURVEY 8(e) (NCCL all-to-all of every key to its owner, slot images back), same prompts, same index, same batch ----
    alltoall = None
    if world > 1 and "sharded" in built and not os.environ.get("KVIDX_BENCH_SKIP_A2A"):
        Qa = min(Q, int(os.environ.get("KVIDX_BENCH_A2A_BATCH", "131072")))
        ix_s = built["sharded"][0]
        d_scores.fill_(-7.0)
        vol = kd.score_alltoall(ix_s, d_tok, d_off, Qa, d_scores, BLOCK, d_has=d_has)
        parity_gate(ix_s, qs=Qa, what="routed all-to-all")
        for _ in range(2):
            kd.score_alltoall(ix_s, d_tok, d_off, Qa, d_scores, BLOCK, d_has=d_has)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(); e0.record(stream)
        for _ in range(3):
            kd.score_alltoall(ix_s, d_tok, d_off, Qa, d_scores, BLOCK, d_has=d_has)
        e1.record(stream); barrier()
        a2a_ms = max_ranks(e0.elapsed_time(e1)) / 3

        def peer_step():
            ix_s.score_batch_dev(d_tok.data_ptr(), d_off.data_ptr(), Qa, d_scores.data_ptr(), d_has_keys=d_has.data_ptr())
        for _ in range(3):
            peer_step()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(); e0.record(stream)
        for _ in range(5):
            peer_step()
        e1.record(stream); barrier()
        peer_ms = max_ranks(e0.elapsed_time(e1)) / 5
        alltoall = {"batch_prompts_per_gpu": Qa, "value_alltoall": world * Qa / (a2a_ms / 1e3), "ms_per_step_alltoall": a2a_ms,
                    "value_peer_probes": world * Qa / (peer_ms / 1e3), "ms_per_step_peer_probes": peer_ms,
                    "nvlink_bytes_per_prompt_alltoall": (vol["bytes_out"] + vol["bytes_back"]) / Qa,
                    "note": "routed form: every key of every prompt hashed at the origin, 8 B to its owner and 32 B back through two NCCL "
                            "all_to_all_single calls, no early exit, no prefix sharing; peer probes: the library's sharded path (64-byte peer loads "
                            "issued by the walk for the slots it actually visits). Both bit-exact vs the closed form."}

    # ---- SURVEY config #5: Score() with the write path running BESIDE it.  A writer thread applies BlockStored batches of new
    # documents and BlockRemoved batches of the ones stored a moment ago through kvidx_apply_events (its own stream; slot
    # updates are single-image publishes the readers never wait for) at >= 100 K events/s per GPU, while this thread runs
    # Score() steps on the resident batch.  Scores of the resident batch must stay bit-exact.
    mixed = None
    if not os.environ.get("KVIDX_BENCH_SKIP_MIXED"):
        import threading
        docs_per_batch = 512                                             # ~5 K stored + ~5 K removed events per pair of calls
        n_batches = 10
        churn0 = wl.D                                                   # documents beyond the indexed ones
        batches = []
        for s_i in range(n_batches):
            ev, hs, tk = wl.fill_events(churn0 + s_i * docs_per_batch, churn0 + (s_i + 1) * docs_per_batch)
            if primary == "sharded":
                ev = kd.events_for_rank(ev, rank, world)
            rm = ev.copy(); rm["op"] = 1; rm["has_parent"] = 0; rm["n_tokens"] = 0
            batches.append((ev, rm, hs, tk))
        target_eps = float(os.environ.get("KVIDX_BENCH_EVENTS_PER_S", "100000")) / (world if primary == "sharded" else 1)
        stop = threading.Event()
        wstat = {"events": 0, "busy_s": 0.0, "err": None, "t0": None, "t1": None}

        def writer():
            try:
                i = 0
                wstat["t0"] = time.perf_counter()
                while not stop.is_set():
                    ev, rm, hs, tk = batches[i % n_batches]
                    ta = time.perf_counter()
                    rc, dropped = ix.apply_events(ev, hs, tk); assert rc == 0 and dropped == 0, ix.last_error()
                    rc, dropped = ix.apply_events(rm, hs, tk); assert rc == 0, ix.last_error()
                    wstat["busy_s"] += time.perf_counter() - ta
                    wstat["events"] += len(ev) + len(rm)
                    i += 1
                    ahead = wstat["events"] / target_eps - (time.perf_counter() - wstat["t0"])     # pace to the target rate
                    if ahead > 0:
                        stop.wait(ahead)
                wstat["t1"] = time.perf_counter()
            except Exception as e:      # noqa: BLE001
                wstat["err"] = repr(e)
                wstat["t1"] = time.perf_counter()

        th = threading.Thread(target=writer)
        torch.cuda.synchronize(); barrier()
        th.start()
        time.sleep(0.05)
        n_mixed = max(args.steps, 10)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(n_mixed):
            step_dev()
        e1.record(stream)
        torch.cuda.synchronize()
        stop.set(); th.join()
        mixed_ms = max_ranks(e0.elapsed_time(e1))
        assert wstat["err"] is None, wstat["err"]
        parity_gate(ix, what="with the write path running")
        w_el = wstat["t1"] - wstat["t0"]
        mixed = {"score_prompts_per_s": world * Q * n_mixed / (mixed_ms / 1e3), "events_per_s": (world if primary == "sharded" else 1) * wstat["events"] / w_el,
                 "blocks_per_event": wl.bpe, "vs_value": (world * Q * n_mixed / (mixed_ms / 1e3)) / value,
                 "writer_busy_frac": wstat["busy_s"] / w_el,
                 "note": "concurrent: a writer thread paces kvidx_apply_events (BlockStored then BlockRemoved batches, ~%d events per call) to the "
                         "target rate while %d Score() steps run on the resident batch (device-timed); scores stay bit-exact" % (len(batches[0][0]), n_mixed)}
        barrier()

    # roofline of the step
    A = algorithmic_bytes(wl, m)
    peak, peak_src = measured_peak()
    kern_s = float(step_ms.mean()) / 1e3
    achieved = float(A.sum()) / kern_s / 1e9
    default_cfg = (T_TOKENS, N_BLOCKS, Q) == (4096, 10_000_000, 1048576) and primary != "sharded"
    traffic = ncu_traffic() if default_cfg else None          # the committed ncu capture is of the default single-GPU step only
    roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": None if traffic is None else traffic * Q,
            "peak_source": peak_src, "algorithmic_bytes_per_prompt_mean": float(A.mean()),
            "algorithmic_bytes_per_launch": float(A.sum()), "kernel_ms": float(step_ms.mean()),
            "kernel": "one step = prefix sort + rounds x parts x (group_round [cp.async token chunks], group_lists, hash_round, walk_round, finish_round), kernel G on low-priority streams; "
                      "achieved = step's algorithmic bytes / step GPU time (CUDA events around all of its launches), i.e. a lower bound for "
                      "every kernel in it; per-kernel ncu summaries under profiles/",
            "note": "traffic = DRAM bytes of one step from the committed ncu range profile of the whole step (profiles/r2_step_range_profile.json; "
                    "per kernel: profiles/score_step_traffic.json), default single-GPU configuration only; null for any other configuration"}

    # ---- e2e: host pinned buffers through the C ABI (H2D + kernels + D2H inside the timed region) ----
    #   headline e2e: kvidx_score_batch_sparse -- the reference's result shape (a map of <= 10 pods per prompt, indexer.go:134)
    #   e2e_dense   : kvidx_score_batch (a dense double[max_pods] row per prompt)
    for mode in modes:
        built[mode][0].set_stream(0)
    h2d_peak = h2d_peak_gbs(dev)
    e_tok_d, e_doc, e_m = device_queries(wl, q_base + Q, q_base + Q + QE, dev)
    h_tok = kvidx.pinned_array((QE * wl.T,), np.uint32)
    torch.cuda.synchronize()
    h_tok[:] = e_tok_d.view(-1).cpu().numpy().view(np.uint32)
    del e_tok_d
    h_off = np.arange(0, (QE + 1) * wl.T, wl.T, dtype=np.int64)
    h_scores = kvidx.pinned_array((QE, wl.P), np.float64)
    sp = (kvidx.pinned_array((QE, 10), np.uint16), kvidx.pinned_array((QE, 10), np.float64), kvidx.pinned_array((QE,), np.uint8), kvidx.pinned_array((QE,), np.uint8))
    e_exp = wl.expected_scores(e_doc[:2048], e_m[:2048], WEIGHTS)
    e_steps = max(3, min(args.steps, 10))

    def e2e_run(sparse):
        def call():
            if sparse:
                ix.score_batch_sparse(h_tok, h_off, out=sp)
            else:
                ix.score_batch(h_tok, h_off, out=h_scores)
        for _ in range(2):
            call()
        if sparse:
            got = np.full((2048, wl.P), -1.0)
            for i in range(2048):
                got[i, sp[0][i, :sp[2][i]]] = sp[1][i, :sp[2][i]]
        else:
            got = h_scores[:2048]
        assert all_ok(nocheck or np.array_equal(got, e_exp)), "e2e score mismatch"
        barrier()
        t0 = time.perf_counter()
        for _ in range(e_steps):
            call()
        torch.cuda.synchronize()
        return max_ranks(time.perf_counter() - t0)
    h2d_b = int(QE * wl.T * 4 + (QE + 1) * 8)
    es_s = e2e_run(True)
    es_d = e2e_run(False)
    e2e = {"value": world * QE * e_steps / es_s, "unit": "prompts/s", "h2d_bytes_per_step": h2d_b,
           "d2h_bytes_per_step": int(QE * (10 * 10 + 2)), "batch_prompts": QE, "steps": e_steps,
           "h2d_peak_GBps_this_rank": h2d_peak, "pcie_frac": (h2d_b * e_steps / es_s / 1e9) / h2d_peak,
           "numa": numa,
           "note": "pinned host tokens -> kvidx_score_batch_sparse -> <= 10 (pod, score) pairs per prompt in pinned host memory "
                   "(the reference's result shape); pcie_frac = achieved H2D rate / this rank's measured pinned-copy bandwidth"}
    e2e_dense = {"value": world * QE * e_steps / es_d, "unit": "prompts/s", "h2d_bytes_per_step": h2d_b,
                 "d2h_bytes_per_step": int(QE * wl.P * 8 + QE), "pcie_frac": (h2d_b * e_steps / es_d / 1e9) / h2d_peak}

    # ---- small-batch latency (the regime a single gRPC request sees): warp-per-prompt cooperative kernel ----
    lat = {}
    for nb in (1, 1024):
        ts = []
        for _ in range(40):
            t0 = time.perf_counter()
            ix.score_batch(h_tok[: nb * wl.T], h_off[: nb + 1], out=h_scores[:nb])
            ts.append(time.perf_counter() - t0)
        ts = np.array(ts[8:]) * 1e3
        lat["batch_%d" % nb] = {"p50_ms": float(np.percentile(ts, 50)), "p99_ms": float(np.percentile(ts, 99))}
    lat["batch_1_matched_blocks"] = int(e_m[0])

    # ---- 1000 concurrent single-prompt callers (the load shape of the reference's gRPC server: one goroutine per RPC, no
    # batching anywhere, server.go:70-96) through the C ABI from a plain C++ load generator; the library's submission queue
    # turns them into shared launches.  Every returned score is verified inside the generator. ----
    clients = None
    qps_bin = os.path.join(PKG, "lib", "kvidx_qps")
    if rank == 0 and world == 1 and os.path.exists(qps_bin) and not os.environ.get("KVIDX_BENCH_SKIP_QPS"):
        clients = {}
        for nthreads in (1, 64, 1000):
            try:
                r = subprocess.run([qps_bin, str(nthreads), "2.0", "4096", str(wl.T)], capture_output=True, text=True, timeout=300)
                clients["threads_%d" % nthreads] = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 else {"error": (r.stderr or r.stdout)[-300:]}
            except Exception as e:      # noqa: BLE001
                clients["threads_%d" % nthreads] = {"error": repr(e)[:300]}
        clients["note"] = ("kvidx_qps: N OS threads, one %d-token prompt per kvidx_score_batch_sparse call, 1 M-block index; calls/s and call latency; "
                           "wrong_results must be 0" % wl.T)

    # ---- CPU baseline (rank 0, N=1 only): the reference-path port on the host cores ----
    cpu = None
    if rank == 0 and world == 1 and not os.environ.get("KVIDX_BENCH_SKIP_CPU"):
        co, cfill = build_cpu_oracle(wl)
        ns = int(os.environ.get("KVIDX_CPU_SAMPLE", "8192"))
        threads, el, l, ref_s = best_threads(co, h_tok, h_off, ns, wl)
        ix.score_batch(h_tok[: ns * wl.T], h_off[: ns + 1], out=h_scores[:ns])
        assert np.array_equal(ref_s, h_scores[:ns]), "GPU scores differ from the CPU reference port"
        cpu = {"value": ns / el, "unit": "prompts/s", "cores": threads, "kind": "port",
               "sample": "%d of the e2e prompts, one GetPodScores per call on %d threads (best of a 1..%d sweep: the path "
                         "serialises on the LRU mutex) against the same %d-block index (bit-exact vs GPU: checked); index fill %.1fs"
                         % (ns, threads, host_threads(), wl.n_blocks, cfill), "host_cores": host_threads(),
               "p50_latency_ms": float(np.percentile(l, 50)) / 1e6, "p99_latency_ms": float(np.percentile(l, 99)) / 1e6,
               "go_probe": go_probe()}
        del co

    # ---- BASELINE config #4 (100 M-block index hash-sharded over the 8 GPUs of the box), as an extra record at N = 8 ----
    config4 = None
    want_c4 = os.environ.get("KVIDX_BENCH_CONFIG4", "1" if world == 8 else "0") == "1"
    if want_c4 and world > 1:
        barrier()                                               # nobody is still probing a peer's shard
        for mode in modes:
            built[mode][0].close()
        built.clear()
        barrier()
        wl4 = synth.Workload(CONFIG_ID, T_TOKENS, int(os.environ.get("KVIDX_BENCH_CONFIG4_BLOCKS", "100000000")), N_PODS, BLOCK)
        ix4, fill4 = build_index("sharded", wl4)
        del d_tok
        torch.cuda.empty_cache()
        d_tok, doc, m = device_queries(wl4, q_base, q_base + Q, dev)
        exp = wl4.expected_scores(doc[:4096], m[:4096], WEIGHTS)
        ix4.set_stream(stream.cuda_stream)

        def step4():
            ix4.score_batch_dev(d_tok.data_ptr(), d_off.data_ptr(), Q, d_scores.data_ptr(), d_has_keys=d_has.data_ptr())
        d_scores.fill_(-7.0)
        step4()
        parity_gate(ix4, what="config #4")
        for _ in range(3):
            step4()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(); e0.record(stream)
        n4 = 5
        for _ in range(n4):
            step4()
        e1.record(stream); barrier()
        ms4 = max_ranks(e0.elapsed_time(e1))
        config4 = {"value": world * Q * n4 / (ms4 / 1e3), "unit": "prompts/s", "ms_per_step": ms4 / n4, "index_blocks": wl4.n_blocks,
                   "queries_per_document": world * Q / wl4.D, "index_fill_s": fill4["fill_s"], "apply_events_s": fill4["apply_s"], "parity": "closed form, every rank",
                   "note": "BASELINE config #4: 100 M-block / 256-pod index hash-range sharded over %d GPUs, %d resident 4K-token prompts per GPU" % (world, Q)}

    if rank == 0:
        out = {"metric": "score_prompts_per_sec", "value": value, "unit": "prompts/s", "n_gpus": world, "steps": args.steps,
               "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
               "vs_baseline": None, "dtype": "u64", "data": "synthetic",
               "config": {"workload": "Score() %d-token prompts, %s-block / 256-pod index (SURVEY 8(d) %s)" % (
                              T_TOKENS, "%dM" % round(N_BLOCKS / 1e6), "metric row" if (T_TOKENS, N_BLOCKS) == (4096, 10_000_000) else "config variant"),
                          "prompt_tokens": wl.T, "index_blocks": wl.n_blocks, "pods": wl.P, "block_size": BLOCK,
                          "batch_prompts_per_gpu": Q, "query_mix": "m uniform in [0,n] matched blocks + random tail",
                          "queries_per_document": Q / wl.D,
                          "pipeline": "prefix-class rounds: each distinct prefix is hashed and probed once per batch (batches >= 393216 prompts; "
                                      "smaller ones, and batches with little repetition, take the per-prompt round kernels, <= 2048 prompts the "
                                      "warp-per-prompt cooperative kernel)"
                                      if launches / max(args.steps, 1) > 100 else "per-prompt rounds / cooperative kernel (batch below the class pipeline's size "
                                      "threshold, or too little repetition: fewer than ~6 prompts per distinct first block)",
                          "l2_policy": "inputs (%.1f GB tokens + %.1f GB table) larger than the 126 MB L2; no flush" % (Q * wl.T * 4 / 1e9, fill["slots"] * 32 / 1e9),
                          "multi_gpu": {"single": "single GPU", "replicas": "replicas: full index per GPU, prompts sharded, no data-path collective",
                                        "sharded": "hash-range sharded tables (the north-star layout): probes and slot updates over NVLink peer memory "
                                                   "from the scoring / event kernels themselves (CUDA IPC), per-pod ingest ranks; value_replicas = "
                                                   "the replica layout on the same box"}[primary],
                          "index_fill_s": fill["fill_s"], "fill_events": fill["events"]},
               "parity": {"gate": "closed-form scores of 4096 prompts per rank bit-exact + pod-count property on every resident prompt, every rank, every "
                                  "mode, before timing and again after the concurrent write run", "modes": modes, "ok": True},
               "write_path": {"apply_events_s": fill["apply_s"], "events_per_s": fill["events"] / fill["apply_s"], "blocks_per_s": fill["keys"] / fill["apply_s"],
                              "pod_entries_per_s": fill["keys"] * 2.5 / fill["apply_s"],
                              "algorithmic_GBps": fill["keys"] * 136 / fill["apply_s"] / 1e9,
                              "roofline": {"bound": "hbm", "achieved": fill["keys"] * 136 / fill["apply_s"] / 1e9, "peak": peak, "unit": "GB/s",
                                           "frac": fill["keys"] * 136 / fill["apply_s"] / 1e9 / peak},
                              "rehashed_events": fill["rehashed"],
                              "note": "index fill through kvidx_apply_events from host arrays (BlockStored, %d blocks per event, 4 pods per document): "
                                      "host sort + H2D + hash_events_kernel + apply_events_kernel, per rank; A_ev = 136 B per block (SURVEY 8(d)); "
                                      "this rank's share of the index = %d keys" % (wl.bpe, fill["keys"])},
               "p99_step_ms": float(np.percentile(step_ms, 99)), "latency": lat, "value_at_64k_batch": value_64k, "value_at_512k_batch": value_512k, "value_sparse_result": value_sparse,
               "mixed_read_write": mixed, "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "e2e_dense": e2e_dense, "concurrent_clients": clients,
               "gpu_launches": int(launches), "clocks": clocks}
        if "replicas" in res and primary != "replicas":
            out["value_replicas"] = res["replicas"]["value"]
            out["ms_per_step_replicas"] = res["replicas"]["total_ms"] / args.steps
            out["sharded_over_replicas"] = value / res["replicas"]["value"]
        if alltoall is not None:
            out["alltoall_vs_peer_probes"] = alltoall
        if config4 is not None:
            out["config4"] = config4
        emit(out)
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def quiet_stdout():
    """Rank 0 must print exactly ONE JSON line on stdout; NCCL / torchrun helpers write banners with C-level
    printf.  Point fd 1 at stderr for the duration of the run and restore it for the final line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(obj), flush=True)


def main():
    sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree it runs from (it may be read-only)
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
