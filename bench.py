#!/usr/bin/env python
"""bench.py -- BASELINE.json metric: 256x256x3 slices/sec of the PnP-AdaNet hot path on B200, synthetic data,
random-init weights.

    python bench.py --gpus N --steps K --warmup W [--config C] [--dump-outputs DIR]     (N>1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference ...       (the CPU restatement of the reference's TF-1.4 path on the host cores --
                                                TF-1.4 itself cannot run in this image; same config, time-bounded)

--config (BASELINE.json `configs`, 1-based):
    1  segmenter forward only                      (source_segmenter.py:88-209), B slices per GPU (default 16)
    2  segmenter Adam train step                   (source_segmenter.py:484),     B = 16
    3  train_gan.py --phase pre-train: D step      (adversarial.py:852-861),      B = 32 per domain, lambda_mask = 0
    4  train_gan.py --phase train-gan joint step   (adversarial.py:840-882),      B = 8 per domain per GPU   [default, headline]
    5  config 4 on the plain-bf16 tensor-core path (one MMA term),                B = 16 per domain per GPU

Prints ONE JSON line on stdout (rank 0); everything else (per-kernel tables, NCCL's own log when NCCL_DEBUG is set) goes
to stderr.  `value` = whole-job slices/s with inputs resident in HBM; `e2e` = the same metric through the Trainer API
with pinned-host inputs copied every step and the loss read back every step.
"""
import argparse
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
import torch  # noqa: E402

# algorithmic conv/FC FLOPs (2*MAC) per unit, SURVEY 8(d) / Appendix A.5
GF_SEG_FWD_PER_SLICE = 83.004
GF_SEG_TRAIN_PER_SLICE = 248.96
GF_PRETRAIN_D_PER_PAIR = 392.87
GF_D_STEP_PER_PAIR = 394.90      # D step, lambda_mask > 0, per CT+MR pair
GF_G_STEP_PER_SLICE = 256.16     # G step, per CT slice
METRIC = "slices_per_sec_full_adversarial_step_256x256x3"
SLICE_BYTES = 256 * 256 * 3 * 4

WORKLOADS = {
    1: ("segmenter forward only (source_segmenter.py:88-209), inference-mode BN; BASELINE configs[0] shape at GPU batch", 16),
    2: ("segmenter Adam train step (source_segmenter.py:484): wCE + Dice + L2, both BN switches on; BASELINE configs[1]", 16),
    3: ("train_gan.py --phase pre-train: 1 D update (B MR + B CT, +clip), lambda_mask=0, segmenter frozen; BASELINE configs[2]", 32),
    4: ("train_gan.py --phase train-gan joint step: 1 D update (B MR + B CT, +clip) + 1 G update (B fresh CT); "
        "BASELINE configs[3] at N GPUs", 8),
    5: ("train_gan.py --phase train-gan joint step on the plain-bf16 tensor-core path (1 MMA term); BASELINE configs[4] at N GPUs", 16),
}


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"bf16_tflops": d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0)), "hbm_gbs": d.get("hbm_gbs", 6650.0),
                "source": "MEASURED_PEAKS.json (bf16_tflops_sustained: kernel timed inside a long step)"}
    return {"bf16_tflops": 1590.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """samples nvidia-smi clocks / throttle reasons during the timed region"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def bench_config(cfg, B, keep_prob, world, backend=None, graphed=None):
    """the `config` object -- identical for both arms (ours / reference) of the same --config / --batch"""
    per_step = {1: B, 2: B, 3: 2 * B, 4: 3 * B, 5: 3 * B}[cfg] * world
    c = {"workload": WORKLOADS[cfg][0], "bench_config": cfg, "batch_per_gpu_per_domain": B, "slices_per_step": per_step,
         "keep_prob": keep_prob if cfg != 1 else 1.0, "parallelism": "dp%d" % world,
         "l2": "per-step working set (activations of %d slices, GBs) exceeds the 126 MB L2; no explicit flush" % (per_step // world)}
    return c


# ------------------------------------------------------------------------------------------------------------------
# workloads (ours)
# ------------------------------------------------------------------------------------------------------------------
class Workload:
    """one `--config`: builds the model/trainer, owns the resident and the end-to-end step"""

    def __init__(self, a, dev, rank, world):
        import pnp_b200  # noqa: F401
        from pnp_b200 import runtime as rt
        from pnp_b200.data import SyntheticSource
        self.a, self.dev, self.rank, self.world, self.cfg, self.B = a, dev, rank, world, a.config, a.batch
        self.kp = a.keep_prob
        rt.set_conv_backend(a.backend)
        torch.manual_seed(0)
        rt.manual_seed(1234 + rank)
        B = self.B
        self.mr_src = SyntheticSource(B, seed=1234 + rank, pool=3)
        self.ct_src = SyntheticSource(B, seed=4321 + rank, shift=0.3, scale=0.8, pool=3)
        self.ct2_src = SyntheticSource(B, seed=8765 + rank, shift=0.3, scale=0.8, pool=3)
        self.graphed = False
        getattr(self, "_build_%d" % (4 if self.cfg == 5 else self.cfg))()

    # -- config 1 / 2: source segmenter ---------------------------------------------------------------------------------
    def _seg(self):
        from pnp_b200 import source_segmenter as seg
        ck = {"cross_flag": True, "miu_cross": 1.0, "dice_flag": True, "miu_dice": 1.0, "regularizer": 1e-4}
        self.net = seg.Full_DRN(channels=3, n_class=5, batch_size=self.B, cost_kwargs=ck, stddev=0.05)
        self.trainer = seg.Trainer(self.net, [], [], num_cls=5, batch_size=self.B, optimizer="adam", opt_kwargs={"learning_rate": 1e-3})
        self.trainer.dp.broadcast_variables(self._all_vars())
        self.x_dev = [p[0].to(self.dev) for p in self.mr_src.pool]
        self.y_dev = [self.trainer.feed(p[0], p[1])[1] for p in self.mr_src.pool]

    def _all_vars(self):
        from pnp_b200 import runtime as rt
        return rt.global_variables()

    def _build_1(self):
        self._seg()
        self.gflop_per_step = self.B * GF_SEG_FWD_PER_SLICE
        self.h2d, self.d2h = self.B * SLICE_BYTES, self.B * 256 * 256 * 8
        self._static_x = self.x_dev[0].clone()
        if self.a.graph:
            try:
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side), torch.no_grad():
                    for _ in range(2):
                        self.net.forward(self._static_x, 1.0, False, False)
                torch.cuda.current_stream().wait_stream(side)
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g), torch.no_grad():
                    self._static_logits = self.net.forward(self._static_x, 1.0, False, False)
                self._fwd_graph, self.graphed = g, True
            except Exception as e:  # noqa: BLE001
                print("bench: forward graph capture failed (%s); eager" % e, file=sys.stderr)

    def _fwd(self, x):
        if self.graphed:
            self._static_x.copy_(x, non_blocking=True)
            self._fwd_graph.replay()
            return self._static_logits
        with torch.no_grad():
            return self.net.forward(x, 1.0, False, False)

    def _build_2(self):
        self._seg()
        self.gflop_per_step = self.B * GF_SEG_TRAIN_PER_SLICE
        self.h2d, self.d2h = self.B * SLICE_BYTES + self.B * 256 * 256 * 8, 2 * 4
        if self.a.graph:
            self.graphed = self.trainer.capture_train_step(self.x_dev[0], self.y_dev[0], self.kp)

    # -- config 3 / 4 / 5: adversarial ---------------------------------------------------------------------------------------
    def _adv(self, phase):
        from pnp_b200 import adversarial as adv
        from pnp_b200.train_gan import configure
        ck, nc, tc = configure(phase)
        self.net = adv.Full_DRN(channels=3, n_class=5, batch_size=self.B, cost_kwargs=ck, network_config=nc, stddev=0.05, stddev_plain=0.05)
        tc["dis_sub_iter"] = 1           # headline: n_D = 1 discriminator update per generator update (SURVEY 8d config 4)
        self.trainer = adv.Trainer(self.net, num_cls=5, batch_size=self.B, opt_kwargs={"learning_rate": 3e-4}, train_config=tc)
        self.trainer.dp.broadcast_variables(self._all_vars())
        self.dev_pool = [(m[0].to(self.dev), c[0].to(self.dev), c2[0].to(self.dev))
                         for m, c, c2 in zip(self.mr_src.pool, self.ct_src.pool, self.ct2_src.pool)]

    def _build_3(self):
        self._adv("pre-train")
        self.gflop_per_step = self.B * GF_PRETRAIN_D_PER_PAIR
        self.h2d, self.d2h = 2 * self.B * SLICE_BYTES, 4
        if self.a.graph:
            self.graphed = self.trainer.capture_d_step(self.dev_pool[0][0], self.dev_pool[0][1], self.kp)

    def _build_4(self):
        self._adv("train-gan")
        self.gflop_per_step = self.B * (GF_D_STEP_PER_PAIR + GF_G_STEP_PER_SLICE)
        self.h2d, self.d2h = 3 * self.B * SLICE_BYTES, 3 * 4
        if self.a.graph:
            self.graphed = self.trainer.capture_joint_step(self.dev_pool[0][0], self.dev_pool[0][1], self.kp)

    # -- steps -----------------------------------------------------------------------------------------------------------
    def step_resident(self, i, eager=False):
        c = self.cfg
        if c == 1:
            x = self.x_dev[i % 3]
            if eager:
                with torch.no_grad():
                    return self.net.forward(x, 1.0, False, False)
            return self._fwd(x)
        if c == 2:
            x, y = self.x_dev[i % 3], self.y_dev[i % 3]
            return self.trainer.train_step(x, y, self.kp) if eager else self.trainer.train_step_replay(x, y, self.kp)
        mr, ct, ct2 = self.dev_pool[i % 3]
        if c == 3:
            return self.trainer.d_step(mr, ct, self.kp) if eager else self.trainer.d_step_replay(mr, ct, self.kp)
        if eager:
            return self.trainer.d_step(mr, ct, self.kp), self.trainer.g_step(ct2, self.kp)
        return self.trainer.joint_step(mr, ct, self.kp, ct_batch_g=ct2)

    def step_e2e(self, i):
        """pinned host batches -> device (inside the timed region) -> step -> loss / prediction read back to the host"""
        c, k, dev = self.cfg, i % 3, self.dev
        if c == 1:
            logits = self._fwd(self.mr_src.pool[k][0].to(dev, non_blocking=True))
            return logits.argmax(3).cpu()                    # the compact prediction (int64 [B,256,256]) is the result
        if c == 2:
            x, y = self.trainer.feed(*self.mr_src.pool[k])   # images + int64 label maps; one-hot on the device
            wce, dice = self.trainer.train_step_replay(x, y, self.kp)
            return float(wce), float(dice)
        mr_h, ct_h, ct2_h = self.mr_src.pool[k][0], self.ct_src.pool[k][0], self.ct2_src.pool[k][0]
        if c == 3:
            d = self.trainer.d_step_replay(mr_h.to(dev, non_blocking=True), ct_h.to(dev, non_blocking=True), self.kp)
            return self.trainer.loss_value(d)
        if self.graphed:
            d, g = self.trainer.joint_step(mr_h, ct_h, self.kp, ct_batch_g=ct2_h)     # pinned host -> static buffers -> replay
        else:
            d, g = self.trainer.joint_step(mr_h.to(dev, non_blocking=True), ct_h.to(dev, non_blocking=True), self.kp,
                                           ct_batch_g=ct2_h.to(dev, non_blocking=True))
        return self.trainer.loss_value(d), self.trainer.loss_value(g)

    def release(self):
        if hasattr(self.trainer, "release_graphs"):
            self.trainer.release_graphs()
        self.trainer._graph = None
        self._fwd_graph = None


# --dump-outputs: an output larger than this many elements is written as a fixed, seeded sample of them, so that the files of
# one run stay under 64 MB in all (at most two such arrays per config)
DUMP_MAX_ELEMS = 6 * 2 ** 20
DUMP_SEED = 0


def _host_sample(t):
    t = t.detach()
    if t.numel() > DUMP_MAX_ELEMS:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(t.numel(), DUMP_MAX_ELEMS, replace=False))
        t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
    return t.float().cpu().numpy()


def dump_outputs(w, out, d):
    """what the last timed step computed, as <d>/<name>.npy: config 1 the logits [B,256,256,5]; the training configs their
    losses (float64 scalars) and the parameters the step updated (float32, flat arena order)"""
    c, tr = w.cfg, w.trainer
    if c == 1:
        arrays = {"logits": out}
    elif c == 2:
        arrays = {"wce_loss": float(out[0]), "dice_loss": float(out[1]), "params": tr.arena.theta}
    elif c == 3:
        arrays = {"dis_loss": tr.loss_value(out), "dis_params": tr.d_arena.theta}
    else:
        arrays = {"dis_loss": tr.loss_value(out[0]), "gen_loss": tr.loss_value(out[1]),
                  "dis_params": tr.d_arena.theta, "gen_params": tr.g_arena.theta}
    os.makedirs(d, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(d, name + ".npy"), _host_sample(v) if torch.is_tensor(v) else np.float64(v))
    print("bench: wrote %s to %s" % (", ".join(n + ".npy" for n in arrays), d), file=sys.stderr)


def _dp_check(w, dist):
    """driver-visible data-parallel evidence (N > 1), computed after the timed loop on a fresh D-step:
      * first-step exchange error: the N-rank update (NCCL all-reduce + fused RMSProp) vs the same optimizer kernel applied to
        the explicitly gathered-and-summed per-rank gradients (what tests/test_dp_gpu.py checks against single-GPU runs);
      * the parameter arenas must be bit-identical on all ranks afterwards (checksums all-gathered)."""
    tr = w.trainer
    mr, ct, ct2 = w.dev_pool[0]
    arenas = [("d", tr.d_arena, tr.dis_optimizer)] + ([("g", tr.g_arena, tr.gen_optimizer)] if w.cfg != 3 else [])
    worst = 0.0
    for name, arena, opt in arenas:
        theta0, ms0, mom0 = arena.theta.clone(), opt.ms.clone(), opt.mom.clone()
        if name == "d":
            tr.d_step(mr, ct, 1.0, apply=False)
        else:
            tr.g_step(ct2, 1.0, apply=False)
        g_local = arena.grad.clone()
        (tr.d_apply if name == "d" else tr.g_apply)()
        theta1 = arena.theta.clone()
        gathered = [torch.empty_like(g_local) for _ in range(w.world)]
        dist.all_gather(gathered, g_local)
        arena.theta.copy_(theta0)
        opt.ms.copy_(ms0)
        opt.mom.copy_(mom0)
        acc = gathered[0].double()
        for t in gathered[1:]:
            acc += t.double()
        arena.grad.copy_(acc.float())
        opt.step(grad_scale=1.0 / w.world)
        err = float((arena.theta - theta1).abs().max() / theta1.abs().max())
        worst = max(worst, err)
        arena.theta.copy_(theta1)
        del gathered, acc
    sums = torch.stack([tr.d_arena.theta.double().sum(), tr.d_arena.theta.double().abs().sum(),
                        tr.g_arena.theta.double().sum(), tr.g_arena.theta.double().abs().sum()])
    allsums = [torch.empty_like(sums) for _ in range(w.world)]
    dist.all_gather(allsums, sums)
    same = all(bool(torch.equal(allsums[0], t)) for t in allsums[1:])
    return {"ranks": w.world, "max_rel_err": worst, "param_checksum_identical": same,
            "what": "first-step N-rank update vs optimizer applied to the gathered-and-summed per-rank gradients (D and G arenas); "
                    "fp64 checksums of both parameter arenas all-gathered after the timed loop"}


def run_ours(a):
    from pnp_b200 import parallel, _C
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # stdout carries exactly one JSON line.  NCCL_DEBUG stays as the launcher set it: NCCL logs to fd 1, so fd 1 points at
    # stderr for the whole run and the JSON line is written to the saved descriptor at the end.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    parallel.init_from_env()
    if world > 1:
        warm = torch.zeros(1, device=dev)
        dist.all_reduce(warm)
        torch.cuda.synchronize()
    from pnp_b200 import functional as F
    w = Workload(a, dev, rank, world)
    B = a.batch

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """-> (ms for `steps` calls of fn, what the last call returned)"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            last = fn(i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        barrier()
        return float(t.item()), last

    # kernel launches of one step, counted on an eager step (a graph replay issues the same kernels without host calls)
    l0 = _C.launch_count
    w.step_resident(0, eager=True)
    launches_per_step = _C.launch_count - l0
    for i in range(a.warmup):
        w.step_resident(i)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_total, last = timed(w.step_resident, a.steps)
    launches = launches_per_step * a.steps
    clocks = sampler.stop() if rank == 0 else None
    if a.dump_outputs and rank == 0:      # before anything below steps the model again
        dump_outputs(w, last, a.dump_outputs)
    del last
    ms_step = ms_total / a.steps
    cfgobj = bench_config(a.config, B, a.keep_prob, world)
    slices_per_step = cfgobj["slices_per_step"]
    value = slices_per_step / (ms_step / 1e3)

    # end-to-end through the public Trainer API with host inputs + result read-back
    for i in range(min(2, a.warmup)):
        w.step_e2e(i)
    ms_e2e = timed(w.step_e2e, a.steps)[0] / a.steps
    e2e = {"value": slices_per_step / (ms_e2e / 1e3), "unit": "slices/s", "h2d_bytes_per_step": w.h2d, "d2h_bytes_per_step": w.d2h,
           "ms_per_step": ms_e2e}

    # the reference's n_D = 20 schedule (train_gan.py:55): 20 D updates (fresh MR+CT batches) per G update
    nd20 = None
    if a.config in (4, 5) and world == 1 and not a.no_nd20:
        tr = w.trainer
        ok = True
        if a.graph:
            tr._graph = None
            ok = tr.capture_d_step(w.dev_pool[0][0], w.dev_pool[0][1], a.keep_prob, warmup=1) and \
                tr.capture_g_step(w.dev_pool[0][2], a.keep_prob, warmup=1)

        def nd20_step(i):
            for j in range(20):
                mr, ct, _ = w.dev_pool[(i + j) % 3]
                tr.d_step_replay(mr, ct, a.keep_prob)
            tr.g_step_replay(w.dev_pool[i % 3][2], a.keep_prob)
        nd20_step(0)
        ms20 = timed(nd20_step, a.steps)[0] / a.steps
        nd20 = {"n_D": 20, "slices_per_step": 41 * B, "ms_per_step": ms20, "value": 41 * B / (ms20 / 1e3), "unit": "slices/s",
                "cuda_graph": bool(ok and a.graph), "conv_tflops_algorithmic": B * (20 * GF_D_STEP_PER_PAIR + GF_G_STEP_PER_SLICE) / ms20}
        if a.graph:        # back to the joint graph for the roofline pass below (eager) -- nothing else replays after this
            tr.release_graphs()
            w.graphed = False

    # roofline of the dominant kernel (tcgen05 conv): CUDA events around every launch over a few eager steps
    roof = None
    nprof = min(a.steps, 3)
    if rank == 0:
        F.PROFILE = []
    for i in range(nprof):      # every rank steps (the steps contain the gradient all-reduce); rank 0 records events
        w.step_resident(i, eager=True)
    torch.cuda.synchronize()
    if rank == 0:
        recs_all = F.PROFILE
        F.PROFILE = None
        roof = _roofline(recs_all, nprof, ms_step, a)

    if a.profile and rank == 0 and world == 1:
        # per-kernel device time of two eager steps (CUPTI through torch.profiler: lighter than ncu, same kernel names)
        from torch.profiler import profile, ProfilerActivity
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(2):
                w.step_resident(i, eager=True)
            torch.cuda.synchronize()
        evs = prof.key_averages()
        tot = sum(e.device_time_total for e in evs)
        for e in sorted(evs, key=lambda e: -e.device_time_total)[:60]:
            print("[prof] %-110s x%4d %9.3f ms %5.1f%%" % (e.key.replace("(anonymous namespace)::", "")[:110], e.count // 2,
                                                            e.device_time_total / 1e3 / 2, 100.0 * e.device_time_total / tot), file=sys.stderr)
        print("[prof] total device time per step %.3f ms in %d launches" % (tot / 1e3 / 2, sum(e.count for e in evs) // 2), file=sys.stderr)

    dp = None
    if world > 1 and a.config in (3, 4, 5):
        dp = _dp_check(w, dist)

    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        cpu = cpu_baseline_sample(a.config, 2 if a.config != 1 else 4, 1)

    if rank == 0:
        nterms = 1 if a.backend == "tc1" else 3
        out = {
            "metric": METRIC, "value": value, "unit": "slices/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": ("bf16 (tcgen05, fp32 accumulate)" if nterms == 1 else "f32 (tcgen05 bf16 hi/lo split x3, fp32 accumulate)"),
            "data": "synthetic", "config": cfgobj,
            "detail": {"conv_backend": a.backend, "cuda_graph": bool(w.graphed or (a.graph and nd20 is not None)),
                       "gflop_per_step_algorithmic": w.gflop_per_step * world},
            "conv_tflops_algorithmic": w.gflop_per_step * world / ms_step,                     # GFLOP / ms = TFLOP/s, all GPUs
            "conv_roofline_frac_whole_step": w.gflop_per_step / ms_step / _peaks()["bf16_tflops"],   # per GPU, of the measured bf16 peak
            "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
        }
        if nd20 is not None:
            out["n_D_20"] = nd20
        if dp is not None:
            out["dp_check"] = dp
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(out) + "\n").encode())
    if world > 1:
        # teardown must never hang the launcher: drop the captured graphs (they pin NCCL work) before the last barrier, and
        # leave through a watchdog-protected hard exit
        sys.stderr.flush()
        threading.Timer(20.0, lambda: os._exit(0)).start()
        w.release()
        import gc
        gc.collect()
        torch.cuda.synchronize()
        try:
            dist.barrier()
        except Exception:
            pass
        os._exit(0)


def _latest_profile(stem):
    for r in ("r2", "r1"):
        p = os.path.join(ROOT, "profiles", "%s_%s" % (r, stem))
        if os.path.exists(p):
            return p
    return None


def _roofline(recs_all, nprof, ms_step, a):
    recs = [r_ for r_ in recs_all if not r_[3].startswith("simt:")]      # the roofline is the tcgen05 kernel's
    by_s = {}
    for s_, e_, fl_, tag_, _k in recs_all:
        if tag_.startswith("simt:"):
            c_ = by_s.setdefault((tag_, round(fl_ / 1e9, 3)), [0, 0.0])
            c_[0] += 1
            c_[1] += s_.elapsed_time(e_)
    for (tag_, gf_), (n_, ms_) in sorted(by_s.items(), key=lambda kv: -kv[1][1])[:40]:
        print("[simt] %-24s %9.3f GF x%3d  %8.3f ms  %7.1f TF/s" % (tag_, gf_, n_, ms_, gf_ * n_ / ms_), file=sys.stderr)
    by = {}
    for s_, e_, fl_, tag_, _k in recs:
        k_ = (tag_, round(fl_ / 1e9, 3))
        c_ = by.setdefault(k_, [0, 0.0])
        c_[0] += 1
        c_[1] += s_.elapsed_time(e_)
    for (tag_, gf_), (n_, ms_) in sorted(by.items(), key=lambda kv: -kv[1][1])[:64]:
        print("[tc] %-18s %9.3f GF x%3d  %8.3f ms  %7.1f TF/s" % (tag_, gf_, n_, ms_, gf_ * n_ / ms_), file=sys.stderr)
    all_ms = sum(r_[0].elapsed_time(r_[1]) for r_ in recs)
    all_fl = sum(r_[2] for r_ in recs)
    simt_ms = sum(r_[0].elapsed_time(r_[1]) for r_ in recs_all if r_[3].startswith("simt:"))
    per_k = {}
    for s_, e_, fl_, tag_, k_ in recs:
        c_ = per_k.setdefault(k_, [0, 0.0, 0.0])
        c_[0] += 1
        c_[1] += s_.elapsed_time(e_)
        c_[2] += fl_
    for k_, (n_, ms_, fl_) in sorted(per_k.items(), key=lambda kv: -kv[1][1]):
        print("[kern] %-34s x%4d %9.3f ms  %7.1f TF/s" % (k_, n_, ms_, fl_ / ms_ / 1e9), file=sys.stderr)
    print("[conv] tcgen05 %.3f ms/step, simt %.3f ms/step, step %.3f ms" % (all_ms / nprof, simt_ms / nprof, ms_step), file=sys.stderr)
    pk = _peaks()
    nterms = 1 if a.backend == "tc1" else 3
    if not recs or all_ms <= 0:
        return {"bound": "tensor", "achieved": 0.0, "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": 0.0, "traffic": None,
                "note": "no tcgen05 launches recorded (backend=%s)" % a.backend}
    # the dominant kernel = the instantiation with the largest share of the step (agrees with the committed launch list)
    dom = max(per_k.items(), key=lambda kv: kv[1][1])[0]
    dom_recs = [r_ for r_ in recs if r_[4] == dom]
    tc_ms = sum(r_[0].elapsed_time(r_[1]) for r_ in dom_recs)
    tc_fl = sum(r_[2] for r_ in dom_recs)
    traffic, traffic_note = None, "no ncu capture committed"
    tj = _latest_profile("conv_tc_ncu.json")
    if tj:
        with open(tj) as f:
            nj = json.load(f)
        # captures taken before the CTA-pair variant existed name the single-CTA kernel without its 4th template argument
        norm = lambda k_: k_.replace(", 1>", ">") if k_.count(",") == 3 else k_
        mine = [l_ for l_ in nj.get("launches", []) if norm(l_["kernel"]).endswith(norm(dom))]
        if mine:
            traffic = sum(l_["dram_bytes"] for l_ in mine) / len(mine)
            traffic_note = ("dram__bytes_read+write per launch, mean over the %d %s launches of the committed ncu --set full capture "
                            "(%s; different layers than the event-timed mean, same kernel)" % (len(mine), dom, os.path.relpath(tj, ROOT)))
    ach = tc_fl / (tc_ms * 1e-3) / 1e12
    ach_all = all_fl / (all_ms * 1e-3) / 1e12
    return {"bound": "tensor", "kernel": "%s (tcgen05.mma kind::f16 + TMA, persistent)" % dom, "achieved": ach, "peak": pk["bf16_tflops"],
            "unit": "TFLOP/s", "frac": ach / pk["bf16_tflops"], "traffic": traffic, "traffic_note": traffic_note, "peak_source": pk["source"],
            "launches_per_step": len(dom_recs) / nprof, "kernel_ms_per_step": tc_ms / nprof,
            "share_of_step": (tc_ms / nprof) / ms_step, "mma_terms": nterms, "issued_frac": nterms * ach / pk["bf16_tflops"],
            "all_tcgen05_convs": {"achieved": ach_all, "frac": ach_all / pk["bf16_tflops"], "issued_frac": nterms * ach_all / pk["bf16_tflops"],
                                  "launches_per_step": len(recs) / nprof, "kernel_ms_per_step": all_ms / nprof,
                                  "share_of_step": (all_ms / nprof) / ms_step},
            "note": "achieved = algorithmic 2*M*N*K per launch / event time (eager pass); the fp32-grade path issues mma_terms bf16 "
                    "MMAs per algorithmic MAC, so tensor-pipe occupancy ~ issued_frac"}


# ------------------------------------------------------------------------------------------------------------------
# CPU arms: the oracle port of the reference's TF-1.4 path on the host cores
# ------------------------------------------------------------------------------------------------------------------
def _host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arms use the physical cores instead (logical/2)"""
    n = max(1, (os.cpu_count() or 2) // 2)
    torch.set_num_threads(n)
    return n


def _oracle_step(cfg, B):
    """-> (callable running ONE step of --config at batch B on the CPU oracle, slices per step)"""
    from oracle.pnp_graphs import (OracleAdversarial, OracleSegmenter, init_numpy_params, synthetic_images, synthetic_labels)
    if cfg in (1, 2):
        from oracle.tf14_numpy import label_decomp
        ws, bns = OracleSegmenter.layout()
        o = OracleSegmenter(init_numpy_params(ws, bns, 0, 0.05), B)
        x = synthetic_images(B, 1234)
        y = torch.from_numpy(label_decomp(5, synthetic_labels(B, 99)))
        if cfg == 1:
            def step():
                with torch.no_grad():
                    o.forward(x, 1.0, False)
            return step, B
        return (lambda: o.train_step(x, y, 0.75)), B
    ws, bns = OracleAdversarial.layout()
    lam = 0.0 if cfg == 3 else 0.3
    o = OracleAdversarial(init_numpy_params(ws, bns, 0, 0.05), B, lambda_mask_loss=lam, dis_sub_iter=1, gen_sub_iter=1, critic_keep_prob=0.75)
    mr, ct, ct2 = synthetic_images(B, 1234), synthetic_images(B, 4321, 0.3, 0.8), synthetic_images(B, 8765, 0.3, 0.8)
    if cfg == 3:
        return (lambda: o.d_step(mr, ct, 0.75)), 2 * B

    def step():
        o.d_step(mr, ct, 0.75)
        o.g_step(ct2, 0.75)
    return step, 3 * B


def cpu_baseline_sample(cfg, B, reps):
    """bounded sample of the same workload on the host cores (oracle port; TF-1.4 semantics restated on torch-CPU)"""
    n = _host_threads()     # physical cores: os.cpu_count() logical threads oversubscribe oneDNN on the GPU host (>10x slower)
    step, slices = _oracle_step(cfg, B)
    times = []
    for _ in range(reps):
        t0 = time.time()
        step()
        times.append(time.time() - t0)
    t = sorted(times)[len(times) // 2]
    return {"value": slices / t, "unit": "slices/s", "cores": n, "kind": "port",
            "sample": "%d step(s) of --config %d at B=%d (%.1f s each); TF-1.4 semantics restated on torch-CPU, TF itself cannot run "
                      "in this image" % (reps, cfg, B, t)}


def run_reference(a):
    """--impl reference: the reference's own CPU path = the oracle port (oracle/pnp_graphs.py), rank 0 only, at the SAME
    --config and batch as our arm.  A step there takes tens of seconds, so the run is time-bounded: at least 1 warm-up and 2
    timed steps, then as many of the requested K as fit into --ref-budget seconds; `steps` reports what was timed."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = _host_threads()
    B = a.batch
    step, slices = _oracle_step(a.config, B)
    t_begin = time.time()
    t0 = time.time()
    step()                                    # warm-up (allocations, oneDNN primitive caches)
    first = time.time() - t0
    warm = 1
    while warm < a.warmup and (time.time() - t_begin) + 3 * first < a.ref_budget:
        step()
        warm += 1
    times = []
    while len(times) < a.steps and (len(times) < 2 or (time.time() - t_begin) + first < a.ref_budget):
        t0 = time.time()
        step()
        times.append(time.time() - t0)
    dt = sum(times) / len(times)
    v = slices / dt
    sample = ("%d timed step(s) (+%d warm-up) of --config %d at B=%d per domain on %d host threads, %.1f s per step; bounded by "
              "--ref-budget %ds (requested --steps %d --warmup %d)" % (len(times), warm, a.config, B, n, dt, a.ref_budget, a.steps, a.warmup))
    out = {"impl": "reference", "metric": METRIC, "value": v, "unit": "slices/s", "n_gpus": a.gpus, "steps": len(times), "warmup": warm,
           "steps_requested": a.steps, "warmup_requested": a.warmup,
           "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": bench_config(a.config, B, a.keep_prob, max(1, a.gpus)),
           "cpu_baseline": {"value": v, "unit": "slices/s", "cores": n, "kind": "port", "sample": sample},
           "e2e": {"value": v, "unit": "slices/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=4, choices=[1, 2, 3, 4, 5], help="BASELINE.json configs, 1-based (default 4: the headline)")
    ap.add_argument("--batch", type=int, default=None, help="slices per domain per GPU (default: the config's, 8 for config 4)")
    ap.add_argument("--keep-prob", type=float, default=0.75)
    ap.add_argument("--backend", default=None, choices=["auto", "simt", "tc3", "tc1"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-nd20", action="store_true", help="skip the n_D = 20 variant of configs 4/5")
    ap.add_argument("--ref-budget", type=int, default=150, help="--impl reference: wall-clock budget in seconds")
    ap.add_argument("--graph", dest="graph", action="store_true", default=True, help="replay the step as one CUDA graph (default)")
    ap.add_argument("--no-graph", dest="graph", action="store_false")
    ap.add_argument("--profile", action="store_true", help="per-kernel device-time table of two eager steps (torch.profiler) on stderr")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (same arguments, same inputs: runs of two "
                         "builds compare output for output)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if a.batch is None:
        a.batch = WORKLOADS[a.config][1]
    if a.backend is None:
        a.backend = "tc1" if a.config == 5 else "auto"
    if a.impl == "reference":
        run_reference(a)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU fallback (use --impl reference for the CPU arm)")
    run_ours(a)


if __name__ == "__main__":
    main()
