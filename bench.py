#!/usr/bin/env python3
"""bench.py — headline benchmark of the two hot paths (BASELINE.json `metric`).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

One "step" is one pass of the hot path over one batch of synthetic input:
  * BLS  (headline, BASELINE configs[2]): bls::verify_signature_sets over 100 000 aggregate attestations x 128 pubkeys per
    GPU; weak scaling — every rank verifies its own shard, one NCCL all-reduce(min) of the verdicts.
  * tree hash (object `tree_hash`, configs[1]): cold tree_hash_root of a 500 000-validator Deneb BeaconState; N > 1 = N
    independent states + one all-gather of the roots the step produced; `sharded_single_state` = one state over N GPUs.
  * `cfg0` (configs[0]): 1 024 SignatureSets — latency and sets/s, next to the CPU oracle on ONE thread.
  * `cfg3` (configs[3]): the SignatureSets of 32 full Deneb blocks (~5.2 k sets, ~1.0 M keys) strong-scaled over N GPUs.
  * `cfg4` (configs[4]): 200 000 attestations + 32 state roots strong-scaled over N GPUs.
`value` is device-resident throughput (inputs already in HBM, CUDA events on the launching stream, max over ranks);
`e2e` is the same metric through the plugin call lhb200_verify_signature_sets with pinned HOST buffers (H2D and D2H
inside the timed region; `e2e_pageable`: ordinary pageable buffers, what a Rust `Vec` is).
`roofline` is the INTEGER-pipe form (both paths are ALU-bound, SURVEY.md §8d): multiply instructions of the dominant kernel
per launch (counted by ncu, profiles/r2_counters.json) / its live CUDA-event time, against the measured IMAD.WIDE issue
peak; the HBM numbers the contract asks for sit under `roofline.hbm` / `roofline.traffic`.
`--impl reference` times the CPU oracle (oracle/, kind "port": the reference's Rust/blst path cannot be built here) on
the host cores on a bounded sample OF THE SAME WORKLOAD (same generator, same seed).
`--dump-outputs DIR` writes, after the timed steps, what the last timed step of each hot path returned to its caller
(rank 0), so that two builds can be compared output for output on the same seeded inputs:
  bls_verdict.npy     float64 [1]       verdict of the last BLS step (1.0 = every set verified)
  bls_set_status.npy  float32 [N_SETS]  per-set status of that step (0 = the set entered the batch check, else why it was rejected)
  state_root.npy      float64 [32]      bytes of the BeaconState root the last tree-hash step produced
"""
import argparse
import ctypes as C
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # before torch creates the CUDA context (see lhb200_init)

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_SETS = int(os.environ.get("LHB_BENCH_SETS", "100000"))
KEYS_PER_SET = int(os.environ.get("LHB_BENCH_KEYS", "128"))
N_VALIDATORS_BLS = 16384
N_VALIDATORS_STATE = int(os.environ.get("LHB_BENCH_VALIDATORS", "500000"))
CFG0_SETS = 1024
CFG3_BLOCKS = 32
CFG3_VALIDATORS = 524288                                  # 2^19 ~ the 500 k of SURVEY §8d (generator needs a power of two)
CFG4_SETS = int(os.environ.get("LHB_BENCH_CFG4_SETS", "200000"))
CFG4_STATES = 32
SEED_CFG2, SEED_CFG0, SEED_CFG3, SEED_CFG4 = 0x11570002, 0x11570000, 0x11570003, 0x11570004
CPU_SAMPLE_SETS = int(os.environ.get("LHB_BENCH_CPU_SAMPLE", "32768"))
BLS_BYTES_PER_SET = 96 * KEYS_PER_SET + 96 + 32 + 8      # SURVEY §8d algorithmic bytes per unit (12 424 B at k=128)
STATE_UNIT_BYTES = 96                                    # one hash32_concat: 64 B in + 32 B out
SKIP = set(filter(None, os.environ.get("LHB_BENCH_SKIP", "").split(",")))   # e.g. cfg3,cfg4 for quick runs


def load_synthetic():
    """lighthouse_b200/synthetic.py as a stand-alone module: the workload DEFINITION (numpy + hashlib) without importing the
    package, i.e. without loading liblhb200.so — the reference arm must not touch the CUDA library."""
    spec = importlib.util.spec_from_file_location("lhb200_synthetic_standalone",
                                                  os.path.join(ROOT, "lighthouse_b200", "synthetic.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def effective_cores():
    """Host threads this process may actually use: affinity mask and cgroup CPU quota (BENCH and SCALE boxes differ)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, min(n, 256))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def counters():
    """Per-launch counters of the shipped kernels from the committed ncu captures (profiles/r2_counters.json):
    {kernel: {"imad_wide_warp_inst": ..., "alu_warp_inst": ..., "dram_bytes": ..., "n_sets": ...}}."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r2_counters.json")))
    except Exception:
        return {}


def imad_peak_warp_inst_per_s():
    """Measured issue peak of the carry-chained 32x32+64 multiply-add (scripts/ubench/imad_peak.cu on this chip)."""
    try:
        for line in open(os.path.join(ROOT, "profiles", "r1_imad_peak.jsonl")):
            d = json.loads(line)
            if "carry" in d["kernel"]:
                return d["thread_inst_per_s"] / 32.0, "measured (profiles/r1_imad_peak.jsonl, IMAD.WIDE.U32.X)"
    except Exception:
        pass
    return 148 * 0.99 * 1.965e9, "fallback (148 SM x 0.99/clk x 1.965 GHz)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.mark_at = index, [], None, 0

    def mark(self):
        """the timed region starts here (nvidia-smi needs a second or two to come up on an 8-GPU box, so it is started
        before the warm-up; rows before the mark are dropped if any arrive after it)"""
        self.mark_at = len(self.rows)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        window = "timed region"
        if len(self.rows) > self.mark_at:
            self.rows = self.rows[self.mark_at:]
        elif self.rows:
            window = "warm-up (same kernels; no sample landed inside the timed region)"
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active")
                                                          for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "window": window}


def dist_env():
    ws = int(os.environ.get("WORLD_SIZE", "1"))
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), ws


class DevPtr:
    """A device pointer as a __cuda_array_interface__ object, so torch can view the library's output in place."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (int(ptr), False), "version": 2}


# ---------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    rank, local_rank, world = dist_env()
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import lighthouse_b200
    from lighthouse_b200 import bls, tree_hash as T, _ffi
    from lighthouse_b200 import synthetic as S
    lighthouse_b200.init(local_rank)
    lib = _ffi.lib
    stream = torch.cuda.Stream(device=dev)
    sp = stream.cuda_stream
    K, W = args.steps, args.warmup

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # the library's own NCCL communicator (no torch / host hops on the data path); id broadcast through torch's store
    lib_comm = False
    if world > 1 and hasattr(lib, "lhb200_comm_init"):
        ident = (C.c_uint8 * 128)()
        if rank == 0:
            _ffi.check(lib.lhb200_comm_unique_id(ident), "comm_unique_id")
        obj = [bytes(ident)]
        dist.broadcast_object_list(obj, src=0)
        ident = (C.c_uint8 * 128).from_buffer_copy(obj[0])
        _ffi.check(lib.lhb200_comm_init(rank, world, ident), "comm_init")
        lib_comm = True

    pin = lambda b: torch.frombuffer(bytearray(b), dtype=torch.uint8).pin_memory()
    vp = lambda t: C.c_void_p(t.data_ptr())
    verdict = torch.zeros(1, dtype=torch.int32, device=dev)

    def time_resident(batch, n_iter, collective=True):
        """n_iter enqueue+result passes on `stream`; returns ms per pass (CUDA events, max over ranks)."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ok = True
        with torch.cuda.stream(stream):
            e0.record(stream)
        for _ in range(n_iter):
            with torch.cuda.stream(stream):
                batch.enqueue(sp)
                ok = batch.result(sp) and ok
                verdict.fill_(1 if ok else 0)
                if world > 1 and collective:
                    dist.all_reduce(verdict, op=dist.ReduceOp.MIN)   # the one collective of the path (SURVEY §8e)
        with torch.cuda.stream(stream):
            e1.record(stream)
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / n_iter, ok

    # ------------------------------------------------------------------ cfg2: the headline BLS workload (per rank)
    pk_table = S.interop_pubkey_table(N_VALIDATORS_BLS)
    ab = S.attestation_batch(N_SETS, keys_per_set=KEYS_PER_SET, n_validators=N_VALIDATORS_BLS, seed=SEED_CFG2,
                             first_index=rank * N_SETS, pk_table=pk_table)
    n_keys = N_SETS * KEYS_PER_SET
    rng = np.random.default_rng(99 + rank)
    rands = rng.integers(1, 2 ** 63, size=N_SETS, dtype=np.uint64) * 2 + 1          # nonzero 64-bit scalars
    batch = bls.Batch(N_SETS, n_keys)
    batch.upload(ab.sigs, ab.msgs, ab.pks, ab.offsets, rands)
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(W):
        ms, ok = time_resident(batch, 1)
        assert ok, "synthetic batch must verify"
    barrier()
    sampler.mark()
    l0 = lib.lhb200_launch_count()
    dom_ms = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        e0.record(stream)
    ok = True
    for _ in range(K):
        with torch.cuda.stream(stream):
            batch.enqueue(sp)
            ok = batch.result(sp) and ok
            verdict.fill_(1 if ok else 0)
            if world > 1 and not os.environ.get("LHB_BENCH_NO_STEP_COLLECTIVE"):   # (diagnostic switch; never set by default)
                dist.all_reduce(verdict, op=dist.ReduceOp.MIN)
        dom_ms.append(batch.dominant_kernel_ms)
    with torch.cuda.stream(stream):
        e1.record(stream)
    barrier()
    bls_ms = max_over_ranks(e0.elapsed_time(e1)) / K
    bls_launches = lib.lhb200_launch_count() - l0
    clocks = sampler.stop()
    assert ok and int(verdict.item()) == 1
    bls_value = N_SETS * world / (bls_ms / 1e3)
    outputs = {}
    if args.dump_outputs:
        # reads back the device verdict and statuses of the last enqueue; the batch is reused below
        ok_last, status = batch.result(sp, want_status=True)
        outputs["bls_verdict"] = np.array([float(ok_last)], dtype=np.float64)
        outputs["bls_set_status"] = status.astype(np.float32)

    # e2e: THE PLUGIN CALL lhb200_verify_signature_sets with host buffers (H2D of every input and D2H of the verdict inside)
    offs_np = ab.offsets.copy()
    h_sigs, h_msgs, h_pks = pin(ab.sigs), pin(ab.msgs), pin(ab.pks)
    h_offs = torch.from_numpy(offs_np.copy()).pin_memory()
    h_rands = torch.from_numpy(rands.copy()).pin_memory()
    h2d = h_sigs.numel() + h_msgs.numel() + h_pks.numel() + h_offs.numel() * 4 + h_rands.numel() * 8
    okb = C.create_string_buffer(1)

    def plugin_call(ps, pm, pp, po, pr, n):
        _ffi.check(lib.lhb200_verify_signature_sets(ps, pm, pp, po, pr, n, okb, None), "verify_signature_sets")
        return okb.raw[0] == 1

    def time_wall(fn, n_iter):
        assert fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_iter):
            assert fn()
        torch.cuda.synchronize(dev)
        ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / n_iter
        barrier()
        return ms

    bls_e2e_ms = time_wall(lambda: plugin_call(vp(h_sigs), vp(h_msgs), vp(h_pks), vp(h_offs), vp(h_rands), N_SETS), K)
    # the same call on ordinary pageable memory (numpy arrays): what a shim that passes Vec<u8> pointers gets
    g_sigs, g_msgs, g_pks = (np.frombuffer(x, dtype=np.uint8).copy() for x in (ab.sigs, ab.msgs, ab.pks))
    cp = lambda a: C.c_void_p(a.ctypes.data)
    bls_e2e_pg_ms = time_wall(lambda: plugin_call(cp(g_sigs), cp(g_msgs), cp(g_pks), cp(offs_np), cp(rands), N_SETS),
                              max(1, min(K, 3)))

    # e2e with the device-resident pubkey table (SURVEY §8f-1): sets carry u32 validator indices
    table = bls.PubkeyTable(N_VALIDATORS_BLS)
    table.append(pk_table.tobytes())
    h_idx = torch.from_numpy(np.ascontiguousarray(ab.committees.reshape(-1).astype(np.uint32))).pin_memory()
    h2d_idx = h_sigs.numel() + h_msgs.numel() + h_idx.numel() * 4 + h_offs.numel() * 4 + h_rands.numel() * 8

    def bls_e2e_idx_step():
        _ffi.check(lib.lhb200_bls_batch_upload_indexed(batch._h, table._h, vp(h_sigs), vp(h_msgs), vp(h_idx),
                                                       vp(h_offs), vp(h_rands), N_SETS), "upload_indexed")
        batch.enqueue(sp)
        return batch.result(sp)

    bls_e2e_idx_ms = time_wall(bls_e2e_idx_step, K)

    # ------------------------------------------------------------------ cfg0: 1 024 sets (latency) — BASELINE configs[0]
    cfg0 = None
    if "cfg0" not in SKIP:
        a0 = S.attestation_batch(CFG0_SETS, keys_per_set=KEYS_PER_SET, n_validators=N_VALIDATORS_BLS, seed=SEED_CFG0,
                                 pk_table=pk_table)
        r0 = np.random.default_rng(7).integers(1, 2 ** 63, size=CFG0_SETS, dtype=np.uint64) * 2 + 1
        b0 = bls.Batch(CFG0_SETS, CFG0_SETS * KEYS_PER_SET)
        b0.upload(a0.sigs, a0.msgs, a0.pks, a0.offsets, r0)
        time_resident(b0, 3, collective=False)
        ms0, ok0 = time_resident(b0, max(K, 10), collective=False)
        assert ok0
        p0 = [pin(a0.sigs), pin(a0.msgs), pin(a0.pks), torch.from_numpy(a0.offsets.copy()).pin_memory(),
              torch.from_numpy(r0.copy()).pin_memory()]
        ms0_e2e = time_wall(lambda: plugin_call(*[vp(t) for t in p0], CFG0_SETS), max(K, 10))
        cfg0 = {"workload": f"verify_signature_sets on {CFG0_SETS} attestation SignatureSets x {KEYS_PER_SET} keys, one GPU "
                            "(BASELINE configs[0])", "latency_ms_resident": ms0, "sets_per_s_resident": CFG0_SETS / ms0 * 1e3,
                "latency_ms_e2e": ms0_e2e, "sets_per_s_e2e": CFG0_SETS / ms0_e2e * 1e3, "launches": int(b0.launches),
                "verdict": True}
        b0.destroy()
        # the reference's steady state: gossip batches of <= 64 sets (beacon_processor/src/lib.rs:202-203), here 64 single-key
        # sets (unaggregated attestations) and 64 aggregates of 128 keys, through the plugin call with pinned buffers
        gossip = {}
        for label, kps in (("64_sets_x_1_key", 1), ("64_sets_x_128_keys", KEYS_PER_SET)):
            ag = S.attestation_batch(64, keys_per_set=kps, n_validators=N_VALIDATORS_BLS, seed=SEED_CFG0 + kps, pk_table=pk_table)
            rg = np.random.default_rng(9).integers(1, 2 ** 63, size=64, dtype=np.uint64) * 2 + 1
            bg = bls.Batch(64, 64 * kps)
            bg.upload(ag.sigs, ag.msgs, ag.pks, ag.offsets, rg)
            time_resident(bg, 3, collective=False)
            msg_, okg = time_resident(bg, max(K, 10), collective=False)
            assert okg
            pg = [pin(ag.sigs), pin(ag.msgs), pin(ag.pks), torch.from_numpy(ag.offsets.copy()).pin_memory(),
                  torch.from_numpy(rg.copy()).pin_memory()]
            msg_e2e = time_wall(lambda: plugin_call(*[vp(t) for t in pg], 64), max(K, 10))
            gossip[label] = {"latency_ms_resident": msg_, "latency_ms_e2e": msg_e2e, "launches": int(bg.launches)}
            bg.destroy()
        cfg0["gossip_batch"] = gossip
        # ... and the same from several blocking workers at once (beacon_processor/src/lib.rs:256): throughput of the boundary
        conc = {}
        gb = [S.attestation_batch(64, keys_per_set=1, n_validators=N_VALIDATORS_BLS, seed=SEED_CFG0 + 100 + t, pk_table=pk_table)
              for t in range(16)]
        for T_ in (8, 16):
            def one(t):
                return bls.verify_signature_sets_raw(gb[t].sigs, gb[t].msgs, gb[t].pks, gb[t].offsets)
            warm = [threading.Thread(target=one, args=(t,)) for t in range(T_)]
            [w.start() for w in warm]; [w.join() for w in warm]
            counts, t_end = [0] * T_, time.perf_counter() + 1.0

            def work(t):
                while time.perf_counter() < t_end:
                    assert one(t)
                    counts[t] += 1
            t0 = time.perf_counter()
            th = [threading.Thread(target=work, args=(t,)) for t in range(T_)]
            [x.start() for x in th]; [x.join() for x in th]
            dt = time.perf_counter() - t0
            conc[f"{T_}_workers"] = {"batches_per_s": sum(counts) / dt, "sets_per_s": sum(counts) * 64 / dt,
                                     "mean_latency_ms": dt * T_ / max(sum(counts), 1) * 1e3}
        cfg0["gossip_concurrent"] = {"workload": "T host threads, each verifying its own 64-set x 1-key batch through "
                                                 "lhb200_verify_signature_sets back to back (pooled handles)", **conc}

    # ------------------------------------------------------------------ tree-hash workload (per rank)
    ssz = S.beacon_state_deneb_ssz(N_VALIDATORS_STATE, seed=42 + rank)
    st = T.ResidentState(ssz)
    root0 = st.root()
    roots_all = torch.zeros(world * 32, dtype=torch.uint8, device=dev)

    def state_step():
        with torch.cuda.stream(stream):
            d_root = st.enqueue(sp)
            if world > 1:   # one all-gather of the 32-byte roots THIS step produced (device pointer, no host hop)
                mine = torch.as_tensor(DevPtr(d_root, 32), device=dev)
                dist.all_gather_into_tensor(roots_all, mine)
        return d_root

    for _ in range(W):
        state_step()
    barrier()
    l0 = lib.lhb200_launch_count()
    with torch.cuda.stream(stream):
        e0.record(stream)
    for _ in range(K):
        d_root = state_step()
    with torch.cuda.stream(stream):
        e1.record(stream)
    barrier()
    if args.dump_outputs:
        outputs["state_root"] = torch.as_tensor(DevPtr(d_root, 32), device=dev).cpu().numpy().astype(np.float64)
    st_dom = st.dominant_kernel_ms
    st_ms = max_over_ranks(e0.elapsed_time(e1)) / K
    st_launches = lib.lhb200_launch_count() - l0
    assert st.root() == root0
    if world > 1:
        assert bytes(roots_all[32 * rank:32 * rank + 32].cpu().tolist()) == root0, "gathered root != this rank's root"

    # one state sharded over all ranks (SURVEY §8e): per-rank leaf ranges, all-gather of subtree roots, combine
    sharded = None
    if world > 1 and (world & (world - 1)) == 0:
        common = S.beacon_state_deneb_ssz(N_VALIDATORS_STATE, seed=4242)          # the same state on every rank
        sh = T.ShardedState(common, rank, world)
        use_lib = lib_comm and hasattr(sh, "root_collective")

        def sharded_step():
            if use_lib:
                return sh.root_collective(sp)          # shard roots -> ncclAllGather -> combine, one stream, no host hop
            mine = sh.shard_roots()
            t = torch.frombuffer(bytearray(mine), dtype=torch.uint8).to(dev)
            out = torch.empty(world * len(mine), dtype=torch.uint8, device=dev)
            dist.all_gather_into_tensor(out, t)
            return sh.combine(bytes(out.cpu().tolist()))

        r_sh = sharded_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(K):
            r_sh = sharded_step()
        torch.cuda.synchronize(dev)
        sh_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / K
        full = T.beacon_state_root_deneb(common) if rank == 0 else None
        sharded = {"ms_per_root": sh_ms, "roots_per_s": 1e3 / sh_ms,
                   "matches_single_gpu_root": (r_sh == full) if rank == 0 else None,
                   "collective": "ncclAllGather inside liblhb200 (device buffers, one stream)" if use_lib
                   else "torch all_gather + host combine",
                   "note": "one 500k-validator state split by leaf range over all ranks; wall clock per root incl. the collective"}
        sh.release()
        barrier()

    h_ssz = pin(ssz)
    out32 = C.create_string_buffer(32)

    def state_e2e_step():
        _ffi.check(lib.lhb200_beacon_state_root_deneb(vp(h_ssz), len(ssz), out32, None), "state root")

    state_e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        state_e2e_step()
    st_e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / K
    assert out32.raw == root0
    units = st.hash_units

    # ------------------------------------------------------------------ cfg3: 32 blocks' SignatureSets over N GPUs (strong)
    cfg3 = None
    if "cfg3" not in SKIP:
        from lighthouse_b200 import parallel as PAR
        kc = S.block_signature_key_counts(CFG3_BLOCKS, CFG3_VALIDATORS)
        offs_all = np.concatenate([[0], np.cumsum(kc)]).astype(np.uint64)
        lo, hi = PAR.shard_ranges_by_keys(offs_all, world)[rank]
        tab3 = S.interop_pubkey_table(CFG3_VALIDATORS)
        w3 = S.sets_workload(kc[lo:hi], CFG3_VALIDATORS, seed=SEED_CFG3, first_index=lo)
        a3 = S.materialize_sets(w3, tab3, bls.sign)
        n3, k3 = hi - lo, int(w3["offsets"][-1])
        b3 = bls.Batch(max(n3, 1), max(k3, 1))
        r3 = np.random.default_rng(3 + rank).integers(1, 2 ** 63, size=max(n3, 1), dtype=np.uint64) * 2 + 1
        if n3:
            b3.upload(a3.sigs, a3.msgs, a3.pks, a3.offsets, r3[:n3])
        time_resident(b3, 2)
        ms3, ok3 = time_resident(b3, max(K, 5))
        assert ok3
        cfg3 = {"workload": f"BlockSignatureVerifier batch of {CFG3_BLOCKS} full Deneb blocks: {len(kc)} SignatureSets, "
                            f"{int(offs_all[-1])} keys ({CFG3_VALIDATORS} validators), key-balanced contiguous shards over "
                            f"{world} GPU(s), one all-reduce(min) (BASELINE configs[3])",
                "sets": int(len(kc)), "keys": int(offs_all[-1]), "ms_per_segment": ms3, "scaling": "strong",
                "sets_per_s": len(kc) / ms3 * 1e3, "blocks_per_s": CFG3_BLOCKS / ms3 * 1e3, "verdict": True}
        b3.destroy()
        del tab3, a3, w3

    # ------------------------------------------------------------------ cfg4: 200 k attestations + 32 state roots (strong)
    cfg4 = None
    if "cfg4" not in SKIP:
        per = (CFG4_SETS + world - 1) // world
        lo4, hi4 = min(CFG4_SETS, rank * per), min(CFG4_SETS, (rank + 1) * per)
        a4 = S.attestation_batch(hi4 - lo4, keys_per_set=KEYS_PER_SET, n_validators=N_VALIDATORS_BLS, seed=SEED_CFG4,
                                 first_index=lo4, pk_table=pk_table)
        r4 = np.random.default_rng(40 + rank).integers(1, 2 ** 63, size=hi4 - lo4, dtype=np.uint64) * 2 + 1
        b4 = bls.Batch(hi4 - lo4, (hi4 - lo4) * KEYS_PER_SET)
        b4.upload(a4.sigs, a4.msgs, a4.pks, a4.offsets, r4)
        my_states = [i for i in range(CFG4_STATES) if i % world == rank]       # whole states round-robin (SURVEY §8e)
        roots4 = torch.zeros(CFG4_STATES * 32, dtype=torch.uint8, device=dev)
        stream2 = torch.cuda.Stream(device=dev)

        def cfg4_step():
            stream2.wait_stream(stream)          # after the previous step's root all-reduce on `stream`
            with torch.cuda.stream(stream):
                b4.enqueue(sp)
            with torch.cuda.stream(stream2):     # the state roots run beside the BLS kernels on a second stream
                roots4.zero_()
                for i in my_states:
                    d_root = st.enqueue(stream2.cuda_stream)
                    roots4[32 * i:32 * i + 32].copy_(torch.as_tensor(DevPtr(d_root, 32), device=dev), non_blocking=True)
            stream.wait_stream(stream2)
            with torch.cuda.stream(stream):
                okk = b4.result(sp)
                verdict.fill_(1 if okk else 0)
                if world > 1:
                    dist.all_reduce(verdict, op=dist.ReduceOp.MIN)
                    dist.all_reduce(roots4.view(torch.int32), op=dist.ReduceOp.SUM)   # each rank fills only its slots
            return okk

        assert cfg4_step()
        barrier()
        with torch.cuda.stream(stream):
            e0.record(stream)
        n4 = max(1, min(K, 3))
        for _ in range(n4):
            assert cfg4_step()
        with torch.cuda.stream(stream):
            e1.record(stream)
        barrier()
        ms4 = max_over_ranks(e0.elapsed_time(e1)) / n4
        torch.cuda.synchronize()
        got4 = bytes(roots4.cpu().tolist())
        want4 = [root0]                          # rank r hashes its own state (seed 42 + r): slot i holds rank (i % world)'s root
        if world > 1:
            mine = torch.tensor(list(root0), dtype=torch.uint8, device=dev)
            allr = torch.zeros(world * 32, dtype=torch.uint8, device=dev)
            dist.all_gather_into_tensor(allr, mine)
            flat = bytes(allr.cpu().tolist())
            want4 = [flat[32 * r:32 * r + 32] for r in range(world)]
        for i in range(CFG4_STATES):             # every slot: mine and the ones the all-reduce brought
            if got4[32 * i:32 * i + 32] != want4[i % world]:
                raise RuntimeError(f"cfg4: state root slot {i} on rank {rank} is {got4[32 * i:32 * i + 32].hex()}, "
                                   f"expected {want4[i % world].hex()}")
        ideal_bls = CFG4_SETS / bls_value * 1e3 * 1.0          # ms at the cfg2 rate of this run (all ranks)
        cfg4 = {"workload": f"mixed epoch: {CFG4_SETS} aggregate attestations x {KEYS_PER_SET} keys + {CFG4_STATES} cold "
                            f"{N_VALIDATORS_STATE}-validator state roots, sets sharded and whole states round-robin over "
                            f"{world} GPU(s); one verdict all-reduce + one root all-reduce(sum of disjoint slots) (BASELINE configs[4])",
                "ms_per_epoch_workload": ms4, "scaling": "strong", "sets_per_s": CFG4_SETS / ms4 * 1e3,
                "state_roots_per_s": CFG4_STATES / ms4 * 1e3,
                "frac_of_cfg2_rate": (CFG4_SETS / bls_value * 1e3 + 0.0) / ms4,
                "roofline_note": "BLS kernels at the cfg2 integer-pipe fraction; the 32 state roots (~0.85 ms each) hide "
                                 "under them on a second stream"}
        b4.destroy()
        del a4

    # ------------------------------------------------------------------ CPU baseline (rank 0, N = 1 only)
    cpu_bls = cpu_state = cpu_cfg0 = None
    if rank == 0 and world == 1:
        from tests import oracle_lib as O
        cores = effective_cores()
        O.set_threads(cores)
        sample = min(N_SETS, CPU_SAMPLE_SETS)
        t0 = time.perf_counter()
        ok_cpu = O.bls_verify_signature_sets(ab.sigs[:96 * sample], ab.msgs[:32 * sample],
                                             ab.pks[:96 * KEYS_PER_SET * sample], ab.offsets[:sample + 1], rands[:sample])
        dt = time.perf_counter() - t0
        assert ok_cpu, "CPU oracle disagrees with the GPU verdict"
        cpu_bls = {"value": sample / dt, "unit": "sets/s", "cores": cores, "kind": "port",
                   "sample": f"first {sample} of the {N_SETS} sets of this run, C oracle (oracle/bls12_381.c), {cores} threads, {dt:.1f} s"}
        O.set_threads(1)
        s1 = min(CFG0_SETS, 192)
        t0 = time.perf_counter()
        assert O.bls_verify_signature_sets(ab.sigs[:96 * s1], ab.msgs[:32 * s1], ab.pks[:96 * KEYS_PER_SET * s1],
                                           ab.offsets[:s1 + 1], rands[:s1])
        dt1 = time.perf_counter() - t0
        cpu_cfg0 = {"value": s1 / dt1, "unit": "sets/s", "cores": 1, "kind": "port",
                    "sample": f"{s1} sets x {KEYS_PER_SET} keys, C oracle, ONE thread (configs[0] names blst single-threaded), {dt1:.1f} s"}
        O.set_threads(cores)
        t0 = time.perf_counter()
        want, _ = O.beacon_state_root_deneb(ssz)
        dt = time.perf_counter() - t0
        assert want == root0, "CPU oracle root differs from the GPU root"
        cpu_state = {"value": 1.0 / dt, "unit": "roots/s", "cores": cores, "kind": "port",
                     "sample": f"1 full {N_VALIDATORS_STATE}-validator state, C oracle with SHA-NI, {cores} threads, {dt*1e3:.1f} ms"}
        O.set_threads(1)
        if cfg0:
            cfg0["cpu_baseline"] = cpu_cfg0

    if rank == 0:
        peak, peak_src = measured_peaks()
        ipeak, ipeak_src = imad_peak_warp_inst_per_s()
        ctr = counters()
        dom = sorted(x for x in dom_ms if x > 0)
        dom_bls = dom[len(dom) // 2] if dom else None
        dom_st = st_dom if st_dom and st_dom > 0 else None
        kname = "k_miller_coop"
        kc_ = ctr.get(kname, {})
        scale = N_SETS / kc_["n_sets"] if kc_.get("n_sets") else None
        imad = kc_.get("imad_wide_warp_inst") * scale if scale else None
        ach = imad / (dom_bls * 1e-3) if (imad and dom_bls) else None
        bls_hbm = BLS_BYTES_PER_SET * N_SETS / (dom_bls * 1e-3) / 1e9 if dom_bls else None
        step_imad = sum(v.get("imad_wide_warp_inst", 0) * (N_SETS / v["n_sets"]) for k, v in ctr.items()
                        if v.get("path") == "bls" and v.get("n_sets"))
        st_units_dom = 8 * N_VALIDATORS_STATE                       # k_validator_roots: 8 hash32_concat per validator
        st_ach = STATE_UNIT_BYTES * st_units_dom / (dom_st * 1e-3) / 1e9 if dom_st else None
        vr = ctr.get("k_validator_roots", {})
        st_alu = vr.get("alu_warp_inst") / (dom_st * 1e-3) if (vr.get("alu_warp_inst") and dom_st) else None
        alu_peak = 148 * 2.0 * (clocks.get("sm_mhz") or 1965) * 1e6   # 64 lanes/clk/SM on the alu pipe
        line = {
            "metric": "bls_sig_sets_verified_per_sec", "value": bls_value, "unit": "sets/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": bls_ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs (381-bit Montgomery integers)", "data": "synthetic",
            "config": {"workload": f"verify_signature_sets: {N_SETS} aggregate attestations x {KEYS_PER_SET} pubkeys per GPU "
                                   f"(BASELINE configs[2]), mainnet spec, interop keys over {N_VALIDATORS_BLS} validators, "
                                   "every message distinct", "sets_per_gpu": N_SETS, "keys_per_set": KEYS_PER_SET,
                       "l2": f"inputs per step {ab.input_bytes/1e6:.0f} MB > 126 MB L2 (no flush needed)",
                       "collective": "ncclAllReduce(min) of 1 x int32 verdict per step" if world > 1 else "none (1 GPU)"},
            "clocks": clocks,
            "e2e": {"value": N_SETS * world / (bls_e2e_ms / 1e3), "unit": "sets/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": 1, "ms_per_step": bls_e2e_ms,
                    "call": "lhb200_verify_signature_sets (the plugin entry point), pinned host buffers",
                    "timer": "perf_counter around synchronised calls"},
            "e2e_pageable": {"value": N_SETS * world / (bls_e2e_pg_ms / 1e3), "unit": "sets/s", "ms_per_step": bls_e2e_pg_ms,
                             "h2d_bytes_per_step": int(h2d), "call": "lhb200_verify_signature_sets, pageable host buffers (keys staged by the library's pinned ring + copy threads)"},
            "e2e_indexed": {"value": N_SETS * world / (bls_e2e_idx_ms / 1e3), "unit": "sets/s",
                            "h2d_bytes_per_step": int(h2d_idx), "d2h_bytes_per_step": 1, "ms_per_step": bls_e2e_idx_ms,
                            "note": "keys referenced by u32 index into the device-resident pubkey table (ValidatorPubkeyCache mirror)"},
            "gpu_launches": int(bls_launches),
            "roofline": {"kernel": kname, "bound": "alu", "pipe": "fmaheavy (32x32+64 multiply-add, IMAD.WIDE)",
                         "achieved": ach / 1e9 if ach else None, "peak": ipeak / 1e9, "unit": "G warp-inst/s",
                         "frac": (ach / ipeak) if ach else None, "peak_source": ipeak_src, "kernel_ms": dom_bls,
                         "imad_wide_warp_inst_per_launch": imad,
                         "counter_source": "ncu source-level instruction counts of this kernel (profiles/r2_counters.json)",
                         "traffic": kc_.get("dram_bytes") * scale if scale and kc_.get("dram_bytes") else None,
                         "hbm": {"achieved": bls_hbm, "peak": peak, "unit": "GB/s", "frac": (bls_hbm / peak) if bls_hbm else None,
                                 "peak_source": peak_src,
                                 "note": "whole-step algorithmic bytes (12 424 B/set) over this kernel's time, as the contract "
                                         "defines it; ~0.7 % by construction — the path is integer-ALU bound"},
                         "step": {"imad_wide_warp_inst": step_imad or None,
                                  "frac_of_peak": (step_imad / (bls_ms * 1e-3) / ipeak) if step_imad else None,
                                  "note": "all BLS kernels of a step / step time: the whole-step integer-pipe fraction"}},
            "cpu_baseline": cpu_bls,
            "cfg0": cfg0, "cfg3": cfg3, "cfg4": cfg4,
            "tree_hash": {
                "metric": "beacon_state_tree_hash_root_per_sec", "value": world / (st_ms / 1e3), "unit": "roots/s",
                "ms_per_step": st_ms, "scaling": "weak (one independent state per GPU)",
                "config": {"workload": f"cold tree_hash_root of a synthetic {N_VALIDATORS_STATE}-validator Deneb BeaconState "
                                       "(BASELINE configs[1]), resident in HBM", "hash32_concat_units": int(units),
                           "l2": "state (72 MB) fits L2; k_init-free re-hash each step reads the same buffers "
                                 "(ALU-bound kernel, HBM traffic is 2% of time)",
                           "collective": "all-gather of the 32-byte root each step produced (device pointer)" if world > 1 else "none"},
                "e2e": {"value": world / (st_e2e_ms / 1e3), "unit": "roots/s", "h2d_bytes_per_step": len(ssz),
                        "d2h_bytes_per_step": 32, "ms_per_step": st_e2e_ms},
                "gpu_launches": int(st_launches),
                "roofline": {"kernel": "k_validator_roots", "bound": "alu", "pipe": "alu (SHF/LOP3/IADD3)",
                             "achieved": st_alu / 1e9 if st_alu else None, "peak": alu_peak / 1e9, "unit": "G warp-inst/s",
                             "frac": (st_alu / alu_peak) if st_alu else None, "kernel_ms": dom_st,
                             "traffic": vr.get("dram_bytes"),
                             "hbm": {"achieved": st_ach, "peak": peak, "unit": "GB/s", "frac": (st_ach / peak) if st_ach else None,
                                     "peak_source": peak_src},
                             "whole_root": {"units_per_s": units / (st_ms / world * 1e-3) if st_ms else None,
                                            "note": "hash32_concat units of the whole root / step time"}},
                "cpu_baseline": cpu_state,
                "sharded_single_state": sharded,
            },
        }
        print(json.dumps(line))
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in outputs.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    if lib_comm:
        lib.lhb200_comm_destroy()
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference's CPU implementation of the path, timed on the host cores.  The reference (Rust + blst/sha2
    asm) cannot be built in this image, so this is the CPU oracle ("port"), all usable host threads, on the first
    CPU_SAMPLE_SETS sets of THE SAME workload the GPU arm verifies (same generator, seed and keys) — built with the
    oracle's own sk_to_pk / sign, so this arm never loads liblhb200.so."""
    rank, _, world = dist_env()
    if rank != 0:
        return
    import numpy as np
    from concurrent.futures import ThreadPoolExecutor
    from tests import oracle_lib as O
    S = load_synthetic()
    cores = effective_cores()
    K, W = args.steps, args.warmup
    sample = min(N_SETS, CPU_SAMPLE_SETS)
    work = S.sets_workload(np.full(sample, KEYS_PER_SET), N_VALIDATORS_BLS, seed=SEED_CFG2, first_index=0)
    pool = ThreadPoolExecutor(max_workers=cores)             # ctypes calls release the GIL
    sks = work["sks"]
    tab = np.frombuffer(b"".join(pool.map(lambda s: O.bls_sk_to_pk(s.to_bytes(32, "big")), sks)),
                        dtype=np.uint8).reshape(len(sks), 96)
    msgs = work["msgs"]
    sign_one = lambda j: O.bls_sign(work["agg_sk"][j].to_bytes(32, "big"), msgs[32 * j:32 * j + 32])
    sigs = b"".join(pool.map(sign_one, range(sample)))
    pks = tab[work["committees"]].tobytes()
    offs = work["offsets"]
    rands = np.random.default_rng(99).integers(1, 2 ** 63, size=sample, dtype=np.uint64) * 2 + 1
    O.set_threads(cores)
    for _ in range(min(W, 1)):
        assert O.bls_verify_signature_sets(sigs, msgs, pks, offs, rands)
    t0 = time.perf_counter()
    for _ in range(K):
        assert O.bls_verify_signature_sets(sigs, msgs, pks, offs, rands)
    dt = (time.perf_counter() - t0) / K
    value = sample / dt
    O.set_threads(1)
    s1 = min(sample, 192)
    t0 = time.perf_counter()
    assert O.bls_verify_signature_sets(sigs[:96 * s1], msgs[:32 * s1], pks[:96 * KEYS_PER_SET * s1], offs[:s1 + 1], rands[:s1])
    dt1 = time.perf_counter() - t0
    O.set_threads(cores)
    ssz = S.beacon_state_deneb_ssz(N_VALIDATORS_STATE, seed=42)
    O.beacon_state_root_deneb(ssz)
    t0 = time.perf_counter()
    for _ in range(K):
        O.beacon_state_root_deneb(ssz)
    dts = (time.perf_counter() - t0) / K
    O.set_threads(1)
    desc = (f"sets [0, {sample}) of the {N_SETS}-set cfg2 workload (same generator, seed and keys as the GPU arm) per step, "
            f"C oracle, {cores} threads")
    print(json.dumps({
        "impl": "reference", "metric": "bls_sig_sets_verified_per_sec", "value": value, "unit": "sets/s",
        "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64 limbs (381-bit Montgomery integers)", "data": "synthetic",
        "config": {"workload": f"verify_signature_sets: {N_SETS} aggregate attestations x {KEYS_PER_SET} pubkeys per GPU "
                               f"(BASELINE configs[2]), mainnet spec, interop keys over {N_VALIDATORS_BLS} validators, "
                               "every message distinct", "sets_per_gpu": N_SETS, "keys_per_set": KEYS_PER_SET,
                   "sample": desc, "same_workload_as_gpu_arm": True},
        "cpu_baseline": {"value": value, "unit": "sets/s", "cores": cores, "kind": "port", "sample": desc},
        "cpu_single_thread": {"value": s1 / dt1, "unit": "sets/s", "cores": 1, "kind": "port",
                              "sample": f"{s1} sets of the same workload, one thread, {dt1:.1f} s"},
        "e2e": {"value": value, "unit": "sets/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "tree_hash": {"metric": "beacon_state_tree_hash_root_per_sec", "value": 1.0 / dts, "unit": "roots/s",
                      "ms_per_step": dts * 1e3, "cpu_baseline": {"value": 1.0 / dts, "unit": "roots/s", "cores": cores,
                                                                   "kind": "port", "sample": "full 500k-validator state per step, SHA-NI"}},
        "note": "reference (Rust, blst 0.3.12 / sha2 asm) is unbuildable in this image (no cargo/rustc, crates not vendored); "
                "this is the from-spec C restatement in oracle/ ('port'), ~2-2.5x slower per core than blst",
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed BLS steps and timed tree-hash steps (>= 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (GPU arm, rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU arm; it does not apply to --impl reference")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
