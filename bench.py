#!/usr/bin/env python
"""Benchmark of the SGD hot path: rating updates/s on synthetic Netflix-shaped ratings.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU kernels

A *step* is one epoch of ``train_linear_kernel`` semantics (kmf_train.pyx:195-277) over the
whole rating set.  ``value`` times K epochs with everything resident in HBM (CUDA events on the
library's stream); ``e2e`` is the median of >= 10 calls of the drop-in
``train_linear_kernel(nbr_epochs=1)`` with host numpy buffers (pinned; the same with pageable
arrays and one 200-epoch call beside it), i.e. H2D of ratings + factors, layout, one epoch, D2H
of the factors inside the timed region.  At N > 1 the line's value is STRONG scaling (the same
100M-rating problem cut into N user slices, with a parity block against the one-GPU run); the
weak-scaling run is the secondary key ``weak``.  One JSON line on stdout (rank 0).
``--dump-outputs DIR`` also writes what the last timed step returned as ``.npy`` files (the model
after the last epoch; with ``--workload topn`` the last call's items and scores); the inputs are
seeded, so two builds run with the same arguments can be compared output for output.  It needs
``--gpus 1``: the ring at N > 1 leaves the model spread over the ranks and is not dumped.
"""
import argparse
import functools
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "rating_updates_per_s"
UNIT = "updates/s"
HP = dict(lr=0.005, K_users=0.05, K_items=0.05, K_bias=0.007)


def algorithmic_bytes_per_update(k, elem_bytes=4):
    """SURVEY.md 8(d): read+write P_u and Q_i (4*k*s) + rating triple (12) + both biases r/w (16)."""
    return 4 * k * elem_bytes + 12 + 16


def captured_traffic(kernel, updates_per_launch):
    """DRAM bytes per launch of the dominant kernel.  NOT measured in this run (ncu replays a
    kernel ~40 times and a number taken under a profiler is never a bench value): it is the latest
    committed `ncu --set full` capture (profiles/traffic.json) rescaled to this run's updates per
    launch; the line says so in `traffic_from`.  Also returns the capture's warp instructions per
    update (for the issue-slot bound)."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(path) as f:
            t = json.load(f)[kernel]
        return (t["dram_bytes_per_launch"] * updates_per_launch / t["updates_per_launch"], t["source"],
                t.get("warp_instructions_per_update"))
    except (OSError, KeyError, ValueError):
        return None, None, None


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(object):
    """SM clocks / throttle reasons sampled DURING the timed region.

    Primary source: NVML polled every 5 ms from a thread of this process (`pynvml`: the same
    counters `nvidia-smi --query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.*` prints, without
    the few hundred ms nvidia-smi needs to produce its first row -- the timed region of a default
    run is ~80 ms).  Fallback: the nvidia-smi recipe of B200_PROFILING.md at 20 ms.  The sampler is
    started before the warm-up; c.begin() / c.end() mark the timed region and summary() uses the
    rows inside the marks (if none fell inside: the rows of the second before c.end(), i.e. warm-up
    steps of the same kernel on the same data, and it says so in "window")."""

    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"),
               (0x4, "sw_power_cap"))

    def __init__(self, device_index):
        self.device_index = device_index
        self.rows = []          # (t, sm_mhz, max_mhz, [reason names])
        self.proc = None
        self.t = None
        self.stop = threading.Event()
        self.t0 = self.t1 = None
        self.source = None

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        # CUDA_VISIBLE_DEVICES may renumber: resolve through the PCI bus id of the CUDA device
        try:
            import torch
            bus = torch.cuda.get_device_properties(self.device_index).pci_bus_id
            dom = torch.cuda.get_device_properties(self.device_index).pci_domain_id
            dev = torch.cuda.get_device_properties(self.device_index).pci_device_id
            return pynvml, pynvml.nvmlDeviceGetHandleByPciBusId(("%08x:%02x:%02x.0" % (dom, bus, dev)).encode())
        except Exception:
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.device_index)

    def __enter__(self):
        try:
            nv, h = self._nvml_handle()
            mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))

            def poll():
                while not self.stop.is_set():
                    try:
                        sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                        try:
                            mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                        except Exception:
                            mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                        self.rows.append((time.monotonic(), sm, mx, [n for b, n in self.REASONS if mask & b]))
                    except Exception:
                        pass
                    time.sleep(0.005)

            self.t = threading.Thread(target=poll, daemon=True)
            self.t.start()
            self.source = "nvml, 5 ms"
            return self
        except Exception:
            pass
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.device_index), "--query-gpu=" + q,
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            self.source = "nvidia-smi -lms 20"
            time.sleep(0.5)       # its first row takes a few hundred ms
        except OSError:
            self.proc = None
        return self

    def _read(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.proc.stdout:
            r = [x.strip() for x in line.split(",")]
            try:
                self.rows.append((time.monotonic(), float(r[0]), float(r[1]),
                                  [n for n, v in zip(names, r[2:6]) if v.lower().startswith("active")]))
            except (ValueError, IndexError):
                continue

    def begin(self):
        self.t0 = time.monotonic()

    def end(self):
        self.t1 = time.monotonic()

    def __exit__(self, *a):
        if self.t1 is None:
            self.t1 = time.monotonic()
        self.stop.set()
        if self.proc:
            time.sleep(0.1)
            self.proc.terminate()
        if self.t:
            self.t.join(timeout=2)

    def summary(self):
        t0 = self.t0 if self.t0 is not None else -1.0
        t1 = self.t1 if self.t1 is not None else float("inf")
        inside = [r for r in self.rows if t0 <= r[0] <= t1]
        window = "timed region"
        if not inside:
            inside = [r for r in self.rows if t1 - 1.0 <= r[0] <= t1 + 0.05]
            window = "last second before the end of the timed region (warm-up steps of the same load; the timed region is shorter than the sampling period)"
        sm = [r[1] for r in inside]
        mx = max([r[2] for r in inside] or [0.0])
        reasons = set()
        for r in inside:
            reasons.update(r[3])
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window, "source": self.source}


# --------------------------------------------------------------------------------------------
# synthetic data on the GPU (torch is plumbing here: RNG, sort/unique, host pinning)
# --------------------------------------------------------------------------------------------
def gpu_synth(torch, dev, nu, ni, nnz, seed, user_offset=0, item_tiles=1, item_seed=None):
    """Netflix-shaped unique (user, item, rating) triples in shuffled order (see
    mfrec_b200/synth.py for the model; this is the same recipe with torch's generator).
    item_tiles > 1: the ni items are `item_tiles` copies of one item-popularity profile (the
    multi-GPU weak-scaling workload); item_seed fixes that profile across ranks."""
    from mfrec_b200 import synth
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    ni_tile = ni // item_tiles
    wu, _ = synth.marginals(nu, ni_tile, seed)
    _, wi = synth.marginals(nu, ni_tile, seed if item_seed is None else item_seed)
    cu = torch.from_numpy(np.cumsum(wu)).to(dev)
    ci = torch.from_numpy(np.cumsum(wi)).to(dev)
    keys = None
    while keys is None or keys.numel() < nnz:
        need = nnz - (0 if keys is None else keys.numel())
        m = int(need * 1.12) + 4096
        us = torch.searchsorted(cu, torch.rand(m, device=dev, dtype=torch.float64, generator=g)).clamp_(max=nu - 1)
        it = torch.searchsorted(ci, torch.rand(m, device=dev, dtype=torch.float64, generator=g)).clamp_(max=ni_tile - 1)
        if item_tiles > 1:
            it += torch.randint(0, item_tiles, (m,), device=dev, generator=g) * ni_tile
        new = us * ni + it
        del us, it
        keys = torch.unique(new if keys is None else torch.cat([keys, new]))
        del new
    perm = torch.randperm(keys.numel(), device=dev, generator=g)[:nnz]
    keys = keys[perm]
    del perm
    users = (keys // ni).to(torch.int32)
    items = (keys % ni).to(torch.int32)
    del keys
    # planted rank-16 model.  The item side comes from its own generator: ranks of a multi-GPU run
    # that draw different users (seed) over the same catalogue (item_seed) must plant the SAME items.
    rank = 16
    gi = torch.Generator(device=dev)
    gi.manual_seed(7919 + (seed if item_seed is None else item_seed))
    bu = torch.randn(nu, device=dev, generator=g) * 0.3
    bi = torch.randn(ni, device=dev, generator=gi) * 0.3
    p = torch.randn(nu, rank, device=dev, generator=g) * 0.35
    q = torch.randn(ni, rank, device=dev, generator=gi) * 0.35
    r = torch.empty(nnz, device=dev, dtype=torch.float32)
    step = 1 << 24
    for a in range(0, nnz, step):
        ul, il = users[a:a + step].long(), items[a:a + step].long()
        val = 3.6 + bu[ul] + bi[il] + (p[ul] * q[il]).sum(1)
        val += torch.randn(val.shape[0], device=dev, generator=g) * 0.5
        r[a:a + step] = val.round_().clamp_(1.0, 5.0)
    idx = torch.stack([users + user_offset, items], dim=1).contiguous()
    return idx, r


def run_native(args):
    import torch
    import torch.distributed as dist
    from mfrec_b200 import _native, synth
    from mfrec_b200.lib import kmf_train

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit("bench.py: --gpus %d but WORLD_SIZE=%d (launch with torch.distributed.run)" % (args.gpus, world))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    nu, ni, nnz, k = synth.SHAPES[args.workload]
    if args.nnz:
        nnz = args.nnz
    if world > 1:
        from mfrec_b200 import dsgd
        return dsgd.bench_multi_gpu(args, rank, world, local, nu, ni, nnz, k, HP, gpu_synth,
                                    ClockSampler, algorithmic_bytes_per_update, measured_peaks)

    t_setup = time.time()
    G = max(1, args.emulate_slabs)
    if G > 1:
        # debug: the per-rank work of a G-GPU weak-scaling ring on ONE GPU (G item slabs processed
        # back to back, no exchange) -- not a bench line
        ni = ni * G
    idx_d, r_d = gpu_synth(torch, dev, nu, ni, nnz, seed=0, item_tiles=G)
    torch.cuda.synchronize()
    ctx = _native.default_context(local)   # the context the drop-in modules use as well: one stream, one pool
    u0, v0 = synth.init_factors(nu, ni, k, seed=2)

    # ---------------- device-resident arm: K epochs, CUDA events on the library stream ------
    R = _native.Ratings(None, None, ni, nu, ctx=ctx, device_ptrs=(idx_d.data_ptr(), r_d.data_ptr()),
                        nnz=nnz, ratings_are_f32=True, k_hint=k, row_blocks=args.row_blocks,
                        workers=args.workers, n_slabs=(G if G > 1 else 0),
                        split=_native.SPLIT_OFF if args.no_split else _native.SPLIT_AUTO)
    _vb, item_rows, n_split = R.copies()
    hot = {"items_split": n_split, "copies": item_rows - ni + n_split,
           "what": "items heavier than half a column group are trained as several copies merged after every epoch "
                   "(DESIGN.md 4.1b); --no-split restores exact sequential equivalence"}
    M = _native.Model(k, ni, nu, u0, v0, None, None, layout=R, ctx=ctx)
    layout_desc = ("stratified B=%d W=%d sub-epochs/epoch=%d max_bucket=%d widest_column_block=%d items"
                   % (R.B, R.W, R.launches_per_epoch, R.max_bucket, R.max_cb_items))
    # schedule balance: the serial chain of one epoch = sum over launches of the slowest CTA,
    # a CTA = sum over phases of its fullest bucket; ideal = nnz / (B * W)
    _, cnt = R.offsets()
    c4 = cnt.reshape(R.G, R.B, R.B, R.W, R.W).astype(np.int64)   # [g, rb, cb, w, phase]
    cta = c4.max(axis=3).sum(axis=3)                              # [g, rb, cb]
    rbs = np.arange(R.B)
    crit = sum(int(cta[g, rbs, (rbs + s) % R.B].max()) for g in range(R.G) for s in range(R.B))
    quad_types = R.quad_types()
    balance = {"critical_path_ratings": crit, "ideal": nnz / float(R.B * R.W),
               "efficiency": nnz / float(R.B * R.W) / max(crit, 1)}
    del cnt, c4, cta
    se = torch.zeros(args.steps + args.warmup, device=dev, dtype=torch.float64)
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
    launches0 = ctx.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        for e in range(args.warmup):
            M.sgd_epoch(R, _native.KERNEL_LINEAR, HP["lr"], HP["K_users"], HP["K_items"], HP["K_bias"],
                        sq_err_ptr=se.data_ptr() + 8 * e)
        ctx.sync()
        launches_warm = ctx.launch_count - launches0
        torch.cuda.synchronize()
        launches1 = ctx.launch_count
        clocks.begin()
        ev0.record(stream)
        for e in range(args.steps):
            M.sgd_epoch(R, _native.KERNEL_LINEAR, HP["lr"], HP["K_users"], HP["K_items"], HP["K_bias"],
                        sq_err_ptr=se.data_ptr() + 8 * (args.warmup + e))
        ev1.record(stream)
        ctx.sync()
        torch.cuda.synchronize()
        clocks.end()
        launches_timed = ctx.launch_count - launches1
    ms = ev0.elapsed_time(ev1)
    ms_per_step = ms / args.steps
    value = nnz * args.steps / (ms * 1e-3)
    rmse_curve = torch.sqrt(se / nnz).cpu().numpy().tolist()
    if args.dump_outputs:
        dump_model(args.dump_outputs, M, se[-1].item())

    peak, peak_src = measured_peaks()
    bpu = algorithmic_bytes_per_update(k)
    clk = clocks.summary()
    # dominant kernel = sgd_block_kernel (launches_timed - steps reduce launches); per-launch
    # figures: algorithmic bytes of one launch / its average duration
    n_sgd = launches_timed - args.steps
    achieved = value * bpu / 1e9
    upl = nnz * args.steps / max(n_sgd, 1)
    launch_s = ms * 1e-3 / max(n_sgd, 1)
    traffic, traffic_src, wipu = captured_traffic("sgd_block_kernel", upl)
    sm_hz = (clk.get("sm_mhz") or 1965.0) * 1e6
    # issue-slot bound: every warp instruction takes one of the 4 issue slots of an SM per cycle
    issue_s = (wipu * upl / (ctx_sm_count(ctx) * 4 * sm_hz)) if wipu else None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "frac_algorithmic": achieved / peak,
                "traffic": traffic, "traffic_from": ("%s (an earlier `ncu --set full` capture rescaled to this run's "
                                                     "updates per launch; NOT measured in this run)" % traffic_src) if traffic_src else None,
                "frac_dram": (traffic / launch_s / 1e9 / peak) if traffic else None,
                "issue_bound": ({"warp_instructions_per_update": wipu, "from": traffic_src,
                                 "sm_mhz": sm_hz / 1e6, "min_launch_ms": issue_s * 1e3,
                                 "frac": issue_s / launch_s}) if issue_s else None,
                "peak_source": peak_src,
                "kernel": "sgd_block_kernel", "algorithmic_bytes_per_update": bpu,
                "algorithmic_bytes_per_launch": bpu * upl,
                "updates_per_launch": upl,
                "avg_launch_us": launch_s * 1e6,
                "note": "three views of one launch: frac_algorithmic = SURVEY 8(d) bytes (every update's Q_i / P_u "
                        "read + write) / time / measured HBM peak -- it exceeds what DRAM moves because a column "
                        "block's Q rows stay in shared memory for a sub-epoch and most P-row sectors hit in the "
                        "126 MB L2; frac_dram = DRAM bytes of the ncu capture / time / peak; issue_bound.frac = "
                        "time the warp instructions alone need on 148 x 4 issue slots / time.  The kernel is bound "
                        "by the serial chain of the hottest items (config.balance), not by HBM."}

    # ---------------- secondary kernels (SURVEY 8(d)): RMSE/predict, top-N, one Funk pass ----------
    secondary = None
    if not args.no_secondary and G == 1:
        secondary = {}
        try:
            secondary["predict_rmse"] = secondary_predict(torch, dev, _native, ctx, M, idx_d, r_d, k, peak)
        except Exception as exc:   # a secondary number never takes the headline down
            secondary["predict_rmse"] = {"error": repr(exc)}
        try:
            secondary["storage_16bit"] = secondary_storage(torch, dev, _native, ctx, idx_d, r_d, nu, ni, nnz, k, u0, v0,
                                                           args, rmse_curve, ms_per_step, peak)
        except Exception as exc:
            secondary["storage_16bit"] = {"error": repr(exc)}

    # ---------------- end-to-end arm: the public drop-in call with host buffers -----------------
    e2e = None
    if not args.no_e2e and G == 1:
        del M, R
        idx_h = torch.empty((nnz, 2), dtype=torch.int32, pin_memory=True)
        r_h = torch.empty(nnz, dtype=torch.float64, pin_memory=True)
        idx_h.copy_(idx_d)
        r_h.copy_(r_d.double())
        u_h = torch.from_numpy(u0).pin_memory()
        v_h = torch.from_numpy(v0).pin_memory()
        ib_h = torch.zeros(ni, dtype=torch.float64).pin_memory()
        ub_h = torch.zeros(nu, dtype=torch.float64).pin_memory()
        pinned = (u_h.numpy(), v_h.numpy(), idx_h.numpy(), r_h.numpy(), ib_h.numpy(), ub_h.numpy())
        kmf_train.options["device"] = local

        def one_call(arrs, epochs=1):
            un, vn, idxn, rn, ibn, ubn = arrs
            kmf_train.train_linear_kernel(epochs, k, 0.1, HP["lr"], 0.0, 0.0, HP["K_users"], HP["K_items"],
                                          HP["K_bias"], 0.0, un, vn, idxn, rn, ibn, ubn)
            return kmf_train.last_rmse[-1]

        def timed_calls(arrs, n_warm, n_calls):
            for _ in range(n_warm):
                one_call(arrs)
            torch.cuda.synchronize()
            per_call, last = [], None
            for _ in range(n_calls):
                tc = time.perf_counter()
                last = one_call(arrs)
                per_call.append((time.perf_counter() - tc) * 1e3)
            return per_call, last

        # warm-up calls: the device's stream-ordered memory pool reaches its steady state after two
        # calls (445 / 76 / 70 / 70 ... ms in a fresh process, tools/e2e_probe.py).  The drop-in
        # uses the same library context as the device-resident arm above (two contexts = two
        # streams sharing one pool made single calls take 0.1 - 2.4 s at random).  The headline is
        # the MEDIAN of the timed calls; ms_per_call lists every one.
        e2e_warm = max(args.warmup, 3)
        n_calls = max(args.e2e_steps, 10)
        per_call, last = timed_calls(pinned, e2e_warm, n_calls)
        med = float(np.median(per_call))
        h2d = sum(a.nbytes for a in pinned)
        d2h = pinned[0].nbytes + pinned[1].nbytes + pinned[4].nbytes + pinned[5].nbytes + 8
        e2e = {"value": nnz / (med * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": med, "statistic": "median of calls",
               "steps": n_calls, "warmup_calls": e2e_warm, "ms_per_call": per_call,
               "host_memory": "pinned", "epochs_per_call": 1, "last_rmse": float(last)}
        # the same call the way an mfrec user makes it: plain (pageable) numpy arrays
        pageable = tuple(np.array(a, copy=True) for a in pinned)
        pc, _ = timed_calls(pageable, 1, max(args.e2e_steps // 2, 5))
        e2e["pageable"] = {"value": nnz / (float(np.median(pc)) * 1e-3), "unit": UNIT, "ms_per_step": float(np.median(pc)),
                           "ms_per_call": pc, "statistic": "median of calls",
                           "what": "identical call with pageable numpy arrays (staged through pinned bounce buffers by the library)"}
        del pageable
        # and a call of KMFRecommender's default length (kmf.py:49: nbr_epochs = 200): transfers amortised
        if args.long_call_epochs > 0:
            tc = time.perf_counter()
            one_call(pinned, args.long_call_epochs)
            dt_long = time.perf_counter() - tc
            e2e["long_call"] = {"epochs_per_call": args.long_call_epochs, "s_per_call": dt_long,
                                "value": nnz * args.long_call_epochs / dt_long, "unit": UNIT,
                                "what": "one call with nbr_epochs=%d (KMFRecommender's default is 200), pinned arrays" % args.long_call_epochs}
        del pinned, idx_h, r_h, u_h, v_h, ib_h, ub_h

    if secondary is not None:
        del idx_d, r_d
        torch.cuda.empty_cache()
        for name, fn in (("topn", secondary_topn), ("funk_pass", secondary_funk),
                         ("als_wrmf", functools.partial(secondary_als, with_cpu=not args.no_cpu))):
            try:
                secondary[name] = fn(torch, dev, _native, ctx, local)
            except Exception as exc:
                secondary[name] = {"error": repr(exc)}

    cpu_baseline = None
    if not args.no_cpu:
        cpu_baseline = time_reference(args.workload, nnz_sample=args.cpu_sample, epochs=1)

    configs_index = {"ml100k": 0, "ml20m": 1, "netflix": 2, "yahoo": 3}[args.workload]
    out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
           "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": "%s-shaped %dx%d nnz=%d k=%d (BASELINE configs[%d]%s)"
                                  % (args.workload, nu, ni, nnz, k, configs_index,
                                     "" if nnz == synth.SHAPES[args.workload][2] else ", nnz overridden"),
                      "kernel": "train_linear_kernel", "schedule": layout_desc, "balance": balance,
                      "quad_types": quad_types, "hot_item_copies": hot,
                      "l2": "inputs (%.1f GB ratings + %.0f MB factors) exceed the 126 MB L2"
                            % (nnz * 12 / 1e9, (nu + ni) * k * 4 / 1e6),
                      "hyper": HP},
           "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "secondary": secondary,
           "gpu_launches": int(launches_timed), "clocks": clk,
           "rmse_per_epoch": rmse_curve, "setup_s": time.time() - t_setup}
    return out


DUMP_BYTES = 60 << 20   # all .npy files of one --dump-outputs together (under 64 MB)


def dump_ids(n, bytes_per_id, budget):
    """Ids 0 .. n-1, or a fixed, seeded, sorted sample of them when n ids would exceed the budget."""
    cap = budget // bytes_per_id
    return np.arange(n) if n <= cap else np.sort(np.random.default_rng(0).choice(n, cap, replace=False))


def write_dump(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def dump_model(out_dir, M, sq_err_last):
    """--dump-outputs: what a caller of the timed path receives after its last step, i.e. the model
    as mfrec_model_read returns it (item / user factors [k, n] and biases) and the sum of squared
    errors of that epoch.  A side with more columns than half the budget holds is written as a
    sample of columns; <side>_ids holds the column ids written, sampled or not."""
    u, v, ib, ub = M.read()
    arrays = {"sq_err": np.array([sq_err_last])}
    for side, f, b in (("item", u, ib), ("user", v, ub)):
        ids = dump_ids(f.shape[1], (f.shape[0] + 2) * 8, DUMP_BYTES // 2)
        arrays.update({side + "_factors": f[:, ids], side + "_bias": b[ids], side + "_ids": ids})
    write_dump(out_dir, arrays)


def ctx_sm_count(ctx):
    import torch
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


# --------------------------------------------------------------------------------------------
# secondary measurements carried in the N = 1 line (SURVEY 8(d): pairs/s for RMSE, TFLOP/s for
# top-N, one Funk pass); each is timed on the device after its own warm-up
# --------------------------------------------------------------------------------------------
def secondary_predict(torch, dev, _native, ctx, M, idx_d, r_d, k, peak):
    """predict_kernel + fused RMSE reduction on the resident model over the training pairs
    themselves (device-resident pairs, 1,044 B algorithmic per pair at k = 128 fp32)."""
    n = int(min(idx_d.shape[0], 50_000_000))
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stats = None
    for _ in range(3):
        _, stats = M.predict("predict_linear", None, want_stats=True, device_ptrs=(idx_d.data_ptr(), r_d.data_ptr(), 0),
                             n=n, real_is_f32=True)
    reps = 5
    ev0.record(stream)
    for _ in range(reps):
        M.predict("predict_linear", None, want_stats=True, device_ptrs=(idx_d.data_ptr(), r_d.data_ptr(), 0),
                  n=n, real_is_f32=True)
    ev1.record(stream)
    ctx.sync()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / reps
    bpp = 2 * k * 4 + 12 + 8
    ach = n / (ms * 1e-3) * bpp / 1e9
    return {"metric": "predict_rmse_pairs_per_s", "value": n / (ms * 1e-3), "unit": "pairs/s", "pairs": n,
            "ms_per_call": ms, "rmse_of_the_pairs": float(np.sqrt(stats[0] / max(stats[2], 1.0))),
            "what": "mfrec_model_predict (predict_kernel + fused error sums) on the resident model, device-resident pairs; "
                    "each call includes its result read-back and stream sync",
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "algorithmic_bytes_per_pair": bpp, "kernel": "predict_kernel"}}


def secondary_storage(torch, dev, _native, ctx, idx_d, r_d, nu, ni, nnz, k, u0, v0, args, f32_curve, f32_ms, peak):
    """The headline workload again with the user-factor rows kept as fp16 / bf16 in HBM
    (mfrec_opts.storage; float32 arithmetic): the same warm-up + timed epochs, the running RMSE
    of the last epoch beside the float32 run's.  Beside, never instead of, the float32 line."""
    out = {"what": "same ratings, seeds, epochs and hyper-parameters as the headline; only the storage type of "
                   "the user-factor rows P (96 % of the model bytes) changes; arithmetic is float32",
           "f32": {"ms_per_epoch": f32_ms, "rmse_last_epoch": f32_curve[-1],
                   "model_bytes": (nu + ni) * (k * 4 + 4)}}
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
    for name, code in (("f16", _native.STORAGE_F16), ("bf16", _native.STORAGE_BF16)):
        R = _native.Ratings(None, None, ni, nu, ctx=ctx, device_ptrs=(idx_d.data_ptr(), r_d.data_ptr()),
                            nnz=nnz, ratings_are_f32=True, k_hint=k, row_blocks=args.row_blocks,
                            workers=args.workers, storage=code,
                            split=_native.SPLIT_OFF if args.no_split else _native.SPLIT_AUTO)
        M = _native.Model(k, ni, nu, u0, v0, None, None, layout=R, ctx=ctx)
        se = torch.zeros(args.steps + args.warmup, device=dev, dtype=torch.float64)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for e in range(args.warmup):
            M.sgd_epoch(R, _native.KERNEL_LINEAR, HP["lr"], HP["K_users"], HP["K_items"], HP["K_bias"],
                        sq_err_ptr=se.data_ptr() + 8 * e)
        ctx.sync()
        ev0.record(stream)
        for e in range(args.steps):
            M.sgd_epoch(R, _native.KERNEL_LINEAR, HP["lr"], HP["K_users"], HP["K_items"], HP["K_bias"],
                        sq_err_ptr=se.data_ptr() + 8 * (args.warmup + e))
        ev1.record(stream)
        ctx.sync()
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1) / args.steps
        curve = torch.sqrt(se / nnz).cpu().numpy().tolist()
        bpu = algorithmic_bytes_per_update(k, 4) - 2 * k * 2   # P row read + written at 2 bytes per element
        out[name] = {"dtype": name, "ms_per_epoch": ms, "value": nnz / (ms * 1e-3), "unit": "updates/s",
                     "layout": "B=%d W=%d" % (R.B, R.W),
                     "rmse_last_epoch": curve[-1], "rel_to_f32": abs(curve[-1] - f32_curve[-1]) / f32_curve[-1],
                     "model_bytes": ni * (k * 4 + 4) + nu * (k * 2 + 4),
                     "algorithmic_bytes_per_update": bpu,
                     "frac_algorithmic": nnz / (ms * 1e-3) * bpu / 1e9 / peak}
        del M, R
    return out


def secondary_topn(torch, dev, _native, ctx, local):
    class A(object):
        steps, warmup = 3, 2
    t = run_topn(A, ctx=ctx)
    keep = ("metric", "value", "unit", "ms_per_step", "roofline", "users_redone_exactly", "candidates_per_user",
            "oracle_check", "dtype")
    out = dict((k2, t[k2]) for k2 in keep if k2 in t)
    out["config"] = t["config"]["workload"]
    out["e2e_ms_per_call"] = t["e2e"]["ms_per_step"]
    return out


def secondary_funk(torch, dev, _native, ctx, local):
    """One training pass of estimator_loop_without_bias (gd_estimator.pyx:691-779) over the
    MovieLens-20M-shaped set: the difference of a 22-pass and a 2-pass call through the drop-in
    (identical transfers, packing and cache set-up), divided by 20."""
    from mfrec_b200 import synth
    from mfrec_b200.lib import gd_estimator
    nu, ni, nnz, _ = synth.SHAPES["ml20m"]
    idx_d, r_d = gpu_synth(torch, dev, nu, ni, nnz, seed=0)
    idx = idx_d.cpu().numpy()
    r = r_d.double().cpu().numpy()
    del idx_d, r_d

    def call(passes):
        u = np.zeros((1, ni)) + 0.1
        v = np.zeros((1, nu)) + 0.1
        t0 = time.perf_counter()
        gd_estimator.estimator_loop_without_bias(passes, passes, 1e9, 1, 0.1, 0.001, 0.05, u, v, idx, r, nu, ni, 0)
        return time.perf_counter() - t0, int(gd_estimator.last_feature_epochs.sum())

    call(2)
    lo = min(call(2) for _ in range(3))
    hi = min(call(22) for _ in range(3))
    per_pass = (hi[0] - lo[0]) / max(hi[1] - lo[1], 1)
    bpu = 12 + 8 + 2 * 16     # triple + cache + two float64 scalars read and written (DESIGN.md 4.3)
    peak, _src = measured_peaks()
    ach = nnz / per_pass * bpu / 1e9
    return {"metric": "funk_feature_updates_per_s", "value": nnz / per_pass, "unit": "feature-updates/s",
            "ms_per_pass": per_pass * 1e3, "passes_timed": hi[1] - lo[1],
            "config": "ml20m-shaped %dx%d nnz=%d, one feature, estimator_loop_without_bias" % (nu, ni, nnz),
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "algorithmic_bytes_per_update": bpu, "kernel": "funk_train_kernel"}}


def secondary_als(torch, dev, _native, ctx, local, with_cpu=True):
    """ALS-WRMF (SURVEY 8(f) #3, als_implicit.pyx:208-352): seconds per epoch (one user sweep + one item
    sweep) of the drop-in `als_wrmf` on ML-20M-shaped implicit feedback, k = 64, host arrays in and
    out; beside it the reference's algorithm on one host core (the oracle's C port -- this is the one
    other place bench.py runs the oracle, like cpu_baseline) on an ML-100K-shaped problem, both as
    row solves per second (a row solve = one k x k system built from the row's neighbours)."""
    from mfrec_b200 import synth
    from mfrec_b200.lib import als_implicit

    def problem(shape):
        nu, ni, nnz, _ = synth.SHAPES[shape]
        idx_d, _r = gpu_synth(torch, dev, nu, ni, nnz, seed=3)
        idx = idx_d.cpu().numpy()
        del idx_d, _r
        users, items = idx[:, 0].astype(np.int64), idx[:, 1].astype(np.int64)
        ou, oi = np.lexsort((items, users)), np.lexsort((users, items))
        ur = np.r_[0, np.bincount(users, minlength=nu)].astype(np.int32)
        ir = np.r_[0, np.bincount(items, minlength=ni)].astype(np.int32)
        return nu, ni, nnz, ur, np.ascontiguousarray(items[ou], np.int32), ir, np.ascontiguousarray(users[oi], np.int32)

    k = 64
    nu, ni, nnz, ur, uc, ir, ic = problem("ml20m")
    rng = np.random.default_rng(5)

    def call(epochs):
        u, v = rng.normal(0, 0.1, (k, ni)), rng.normal(0, 0.1, (k, nu))
        t0 = time.perf_counter()
        als_implicit.als_wrmf(epochs, k, u, v, None, None, ur, uc, ir, ic, nu, ni, c_pos=1, k=0.015)
        return time.perf_counter() - t0

    call(1)
    lo = min(call(1) for _ in range(2))
    hi = min(call(3) for _ in range(2))
    per_epoch = (hi - lo) / 2.0
    out = {"metric": "als_row_solves_per_s", "value": (nu + ni) / per_epoch, "unit": "row solves/s",
           "s_per_epoch": per_epoch, "config": "ml20m-shaped implicit feedback %dx%d nnz=%d, k=%d, float64" % (nu, ni, nnz, k),
           "kernel": "als_solve_kernel (one CTA per row: Gram in shared memory + Cholesky)"}
    if with_cpu:
        from oracle import cpu
        nu2, ni2, nnz2, ur2, uc2, ir2, ic2 = problem("ml100k")
        u, v = rng.normal(0, 0.1, (k, ni2)), rng.normal(0, 0.1, (k, nu2))
        t0 = time.perf_counter()
        cpu.als_wrmf(1, k, u, v, ur2, uc2, ir2, ic2, 1, 0.015)
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": (nu2 + ni2) / dt, "unit": "row solves/s", "cores": 1, "kind": "port",
                               "sample": "one epoch on an ml100k-shaped problem (%dx%d nnz=%d), k=%d, %.2f s" % (nu2, ni2, nnz2, k, dt)}
    return out


# --------------------------------------------------------------------------------------------
# secondary bench: BASELINE configs[4], top-N scoring of U.V^T on the tensor cores
#   python bench.py --workload topn [--steps K --warmup W]
# --------------------------------------------------------------------------------------------
def topn_float64(u, v, users, N, offset=1.0):
    """Independent float64 restatement of the reference's per-user loop for the check below
    (gradient_descent.py:769-802 with predict_rating = dot + 1.0, :621-631): score every item, skip
    the item whose id equals the user id (the reference's quirk), drop exact zeros / NaN, order by
    score descending (ties: ascending item id), keep N."""
    sc = v[:, users].T @ u + offset                       # [n_users, ni]
    sc[np.isnan(sc)] = 0.0
    ni = u.shape[1]
    for row, user in enumerate(users):
        if user < ni:
            sc[row, user] = 0.0
    order = np.lexsort((np.broadcast_to(np.arange(ni), sc.shape), -sc), axis=1)[:, :N]
    top = np.take_along_axis(sc, order, axis=1)
    return order, top


def run_topn(args, ctx=None):
    import torch
    from mfrec_b200 import _native, synth
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    nu, ni, _nnz, k = synth.SHAPES["netflix"]
    N = 100
    ctx = ctx or _native.default_context(local)   # the context the drop-in modules use as well: one stream, one pool
    u0, v0 = synth.init_factors(nu, ni, k, seed=2)
    u_h, v_h = torch.from_numpy(u0).pin_memory(), torch.from_numpy(v0).pin_memory()
    items = torch.empty((nu, N), dtype=torch.int32).pin_memory()
    scores = torch.empty((nu, N), dtype=torch.float64).pin_memory()
    counts = torch.empty(nu, dtype=torch.int32).pin_memory()
    out = (items.numpy(), scores.numpy(), counts.numpy())

    def call():
        return _native.topn_sweep("predict_rating", u_h.numpy(), v_h.numpy(), None, ni, None, None, N,
                                  ctx=ctx, out=out)[3]

    sweep_ms, finish_ms = [], []
    with ClockSampler(local) as clocks:
        for _ in range(args.warmup):
            call()
        torch.cuda.synchronize()
        clocks.begin()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            st = call()
            sweep_ms.append(st[2])
            finish_ms.append(st[7])
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        clocks.end()
    if getattr(args, "dump_outputs", None):
        # the last call's result (items -1 padded, scores, counts) for a sample of users
        ids = dump_ids(nu, (2 * N + 2) * 8, DUMP_BYTES)
        write_dump(args.dump_outputs, {"topn_items": out[0][ids], "topn_scores": out[1][ids],
                                       "topn_counts": out[2][ids], "topn_user_ids": ids})
    flops = 2.0 * nu * ni * k
    sm = float(np.mean(sweep_ms))
    peaks = {}
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            peaks = json.load(f)
    peak = float(peaks.get("bf16_tflops", 1590.0))   # the sweep kernel is timed alone: burst figure
    # check 1,024 sampled users against an independent float64 numpy restatement of the
    # reference's loop (not against this library's own exact path)
    users = np.sort(np.random.default_rng(0).permutation(nu)[:1024]).astype(np.int64)
    want_items, want_scores = topn_float64(u0, v0, users, N)
    got_items, got_scores = out[0][users], out[1][users]
    score_ok = bool(np.allclose(got_scores, want_scores, rtol=1e-5, atol=1e-6))
    same_items = float((got_items == want_items).mean())   # fp32 vs fp64 may swap near-ties
    same_sets = float(np.mean([len(set(a) & set(b)) / float(N) for a, b in zip(got_items, want_items)]))
    oracle_check = {"users": int(users.shape[0]), "scores_within_1e-5": score_ok,
                    "identical_positions": same_items, "identical_sets": same_sets,
                    "against": "float64 numpy restatement of gradient_descent.py:769-802"}
    return {"metric": "topn_user_item_scores_per_s", "value": nu * float(ni) / ((sm + float(np.mean(finish_ms))) * 1e-3),
            "unit": "scores/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": sm + float(np.mean(finish_ms)), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16 filter + f32 exact re-score", "data": "synthetic",
            "config": {"workload": "top-%d of U.V^T, netflix-shaped factors %d users x %d items, k=%d (BASELINE configs[4])" % (N, nu, ni, k),
                       "what": "value = device time of sweep (tcgen05) + finish (exact re-score, rank, certify) kernels"},
            "roofline": {"bound": "tensor", "achieved": flops / (sm * 1e-3) / 1e12, "peak": peak, "unit": "TFLOP/s",
                         "frac": flops / (sm * 1e-3) / 1e12 / peak, "traffic": None,
                         "kernel": "topn_sweep_kernel", "flops_per_launch": flops / 7.0,
                         "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst)" if peaks else "fallback",
                         "sweep_ms": sm, "finish_ms": float(np.mean(finish_ms))},
            "cpu_baseline": None,
            "e2e": {"value": nu * float(ni) * args.steps / dt, "unit": "scores/s",
                    "h2d_bytes_per_step": u0.nbytes + v0.nbytes, "d2h_bytes_per_step": sum(a.nbytes for a in out),
                    "ms_per_step": dt * 1e3 / args.steps},
            "gpu_launches": None, "users_redone_exactly": float(st[0]), "candidates_per_user": float(st[1]),
            "oracle_check": oracle_check, "clocks": clocks.summary()}


# --------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU kernel (oracle/_ref, else our C port) on host cores
# --------------------------------------------------------------------------------------------
def time_reference(workload, nnz_sample, epochs=1):
    """Times kmf_train.train_linear_kernel (the reference's own Cython build when available) on a
    bounded sample: the first `nnz_sample` ratings of the workload with FULL-SIZE factor matrices
    (so the strided access pattern is the real one).  Single thread: the reference holds the GIL
    and has no threading."""
    from mfrec_b200 import synth
    from oracle import cpu, ref
    nu, ni, nnz, k = synth.SHAPES[workload]
    n = int(min(nnz_sample, nnz))
    rng = np.random.Generator(np.random.PCG64(0))
    wu, wi = synth.marginals(nu, ni, 0)
    cu, ci = np.cumsum(wu), np.cumsum(wi)
    idx = np.empty((n, 2), dtype=np.int32)
    idx[:, 0] = np.minimum(np.searchsorted(cu, rng.random(n)), nu - 1)
    idx[:, 1] = np.minimum(np.searchsorted(ci, rng.random(n)), ni - 1)
    r = rng.integers(1, 6, n).astype(np.float64)
    u, v = synth.init_factors(nu, ni, k, seed=2)
    ib, ub = np.zeros(ni), np.zeros(nu)
    if ref.available():
        kind = "reference"
        fn = ref.kmf_train().train_linear_kernel
        t0 = time.perf_counter()
        fn(epochs, k, 0.1, HP["lr"], 0.0, 0.0, HP["K_users"], HP["K_items"], HP["K_bias"], 0.0,
           u, v, idx, r, ib, ub, 1, 1, 0)
        dt = time.perf_counter() - t0
    else:
        kind = "port"
        t0 = time.perf_counter()
        cpu.kmf_train("linear", epochs, k, HP["lr"], HP["K_users"], HP["K_items"], HP["K_bias"], u, v, idx, r, ib, ub)
        dt = time.perf_counter() - t0
    # the same arithmetic on ROW-major float32 factors (the GPU path's layout), one core: how much of
    # the gap is the reference's feature-major float64 layout (SURVEY 8(d) "fair-layout CPU figure")
    P = np.ascontiguousarray(v.T, dtype=np.float32)
    Q = np.ascontiguousarray(u.T, dtype=np.float32)
    t0 = time.perf_counter()
    cpu.kmf_epoch_rowmajor_f32(k, HP["lr"], HP["K_users"], HP["K_items"], HP["K_bias"], P, Q,
                               np.zeros(nu, dtype=np.float32), np.zeros(ni, dtype=np.float32), idx,
                               r.astype(np.float32))
    dt_fair = time.perf_counter() - t0
    # ... and on every host core (user slices per thread, item rows shared without locks: throughput only)
    cores = os.cpu_count() or 1
    P = np.ascontiguousarray(v.T, dtype=np.float32)
    Q = np.ascontiguousarray(u.T, dtype=np.float32)
    t0 = time.perf_counter()
    cpu.kmf_epoch_rowmajor_f32_mt(k, HP["lr"], HP["K_users"], HP["K_items"], HP["K_bias"], P, Q,
                                  np.zeros(nu, dtype=np.float32), np.zeros(ni, dtype=np.float32), idx,
                                  r.astype(np.float32), cores)
    dt_fair_mt = time.perf_counter() - t0
    return {"value": n * epochs / dt, "unit": UNIT, "cores": 1, "kind": kind,
            "sample": "%d-rating sample of the %s workload, full-size factor matrices (%dx%d, k=%d), %d epoch, %.1f s"
                      % (n, workload, nu, ni, k, epochs, dt),
            "host_cores_available": os.cpu_count(),
            "fair_layout": {"value": n / dt_fair, "unit": UNIT, "cores": 1,
                            "what": "same loop in C on row-major float32 factors (oracle/mfrec_oracle.c), same sample",
                            "all_cores": {"value": n / dt_fair_mt, "unit": UNIT, "cores": cores,
                                          "what": "the same loop on every host core: user slices per thread, item rows "
                                                  "updated without locks (a throughput figure, not the reference's algorithm)"}}}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    from mfrec_b200 import synth
    nu, ni, nnz, k = synth.SHAPES[args.workload]
    vals = []
    for _ in range(args.warmup):
        time_reference(args.workload, max(args.cpu_sample // 10, 1000))
    t0 = time.perf_counter()
    for _ in range(args.steps):
        vals.append(time_reference(args.workload, args.cpu_sample))
    dt = time.perf_counter() - t0
    value = float(np.mean([v["value"] for v in vals]))
    base = dict(vals[-1])
    base["value"] = value
    return {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3 / max(args.steps, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": "%s-shaped %dx%d k=%d, %d-rating sample per step" % (args.workload, nu, ni, k, args.cpu_sample),
                       "kernel": "train_linear_kernel", "hyper": HP},
            "cpu_baseline": base,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="netflix", choices=["ml100k", "ml20m", "netflix", "yahoo", "topn"])
    ap.add_argument("--nnz", type=int, default=0, help="override the number of ratings (debug)")
    ap.add_argument("--row-blocks", type=int, default=0)
    ap.add_argument("--workers", type=int, default=0)
    ap.add_argument("--e2e-steps", type=int, default=10, help="timed end-to-end calls (median reported)")
    ap.add_argument("--long-call-epochs", type=int, default=200,
                    help="epochs of the one long end-to-end call (0 = skip)")
    ap.add_argument("--no-split", action="store_true", help="pack without hot-item copies (exact sequential equivalence)")
    ap.add_argument("--no-secondary", action="store_true", help="skip the predict / top-N / Funk blocks")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N > 1: peer = persistent launches + column blocks over peer memory; nccl = slab send/recv")
    ap.add_argument("--cpu-sample", type=int, default=5_000_000)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--scaling", default="both", choices=["both", "strong", "weak"],
                    help="N > 1: strong = the named problem cut into N user slices (the line's value); "
                         "weak = one tile per GPU (secondary key); both = strong line + `weak` key")
    ap.add_argument("--emulate-slabs", type=int, default=1,
                    help="debug: run one rank's share of a G-GPU ring on one GPU (no exchange)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last step returned (the model and its squared-error "
                         "sum; top-N: items and scores) as DIR/<name>.npy (float64, < 64 MB: large outputs as a "
                         "seeded sample); --gpus 1 only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "native" or args.gpus != 1):
        ap.error("--dump-outputs needs the native path on one GPU (--gpus 1)")
    # exactly ONE line on stdout: libraries print banners there (e.g. "NCCL version ..." at the
    # first communicator), so everything but the final JSON line is sent to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if args.warmup < 3 and args.impl == "native":
        print("bench.py: warmup < 3 breaks the timing rules; using 3", file=sys.stderr)
        args.warmup = 3
    if args.workload == "topn":
        out = run_topn(args)
    else:
        out = run_reference(args) if args.impl == "reference" else run_native(args)
    if out is not None:
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(out) + "\n").encode())


if __name__ == "__main__":
    main()
