#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched Dojo step on B200 (BASELINE.json metric: forward and forward+gradient).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--mech ant|quadruped|atlas|pendulum] [--batch B] [--mode fwd|grad] [--no-sub] [--dump-outputs DIR]

One JSON line is printed by rank 0.  With --dump-outputs, rank 0 also writes what the last timed step of each record returned
(next states, status, Newton iterations and, in grad mode, the gradients; see last_step_outputs) as .npy files, so that two builds
can be compared output for output: the states and inputs are seeded, identical from run to run.

Headline (`value`, `e2e`, `roofline`, `cpu_baseline`, `parity`) = BASELINE.json configs[1]: Ant (DojoEnvironments defaults),
batch 4096 per GPU, forward-only step!.  With no --mech / --batch / --mode flags the same line also carries `sub_records`, so that one
driver invocation measures the whole metric:
    N = 1:  ant_grad (ant B=4096 step! + get_maximal_gradients), quadruped_grad (C2: B=8192 forward + IFT gradients),
            atlas_fwd (atlas B=4096 forward)
    N > 1:  c4_ant_grad (C4: ant 8192 per GPU, forward + gradients, gather of the next states), c3_atlas_fwd (C3 shape: atlas 4096 per GPU)
Every record has its own ms_per_step, value, roofline (algorithmic bytes of SURVEY.md 8d / kernel time), failed_env_steps,
mean_newton_iters and a `parity` block: a random sample of the TIMED batch stepped by the CPU oracle and compared with the GPU result
(status / iteration-count / state mismatch RATES; the oracle is the checker here, never the thing measured).

A "step" is one step! of every environment of the batch; the state advances from step to step with fresh random inputs.
Workloads (WORKLOADS below, SURVEY.md 8d): ant -- jittered poses dropped from random heights, rolled in for 20 untimed steps so that
the batch is in contact (unchanged from round 1); quadruped / atlas -- jittered stance with the lowest contact sphere ON the ground
and random joint torques, restarted from the stance every 8 steps (nothing holds these robots up without a controller: after ~0.15 s
of free fall the batch is a heap of impacts on which the reference solver itself -- the CPU oracle -- ends 15 - 25 % of its
steps :failed; round 1 timed that).

`value` = env-steps/s with inputs resident in HBM (CUDA events around the launches on the launching stream, max over ranks);
`e2e` = the same metric through the public host API with pinned HOST buffers (H2D + kernels + D2H inside the timed region; at N > 1
including the gather of the next states).  `--impl reference` times the CPU port of the reference (oracle/) on the host cores.
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
sys.path.insert(0, ROOT)
import dojo_jl_b200 as dj  # noqa: E402
from dojo_jl_b200 import capi  # noqa: E402
from dojo_jl_b200 import quat as Q  # noqa: E402

ALGO_BYTES = {  # per env-step, SURVEY.md §8(d): read z + read u + write z_next + status/iters (+ gradients)
    "fwd": lambda m: 8 * (2 * m.nz + m.nu) + 8,
    "grad": lambda m: 8 * (2 * m.nz + m.nu) + 8 + 8 * (12 * m.Nb) ** 2 + 8 * 12 * m.Nb * m.nu,
}
SCALE = {"ant": 1.0, "quadruped": 2.0, "atlas": 5.0, "pendulum": 1.0}
# base_dz: offset of the floating base height; tilt: std of the base rotation vector; jitter: +- joint coordinate jitter (inside the
# limits); ground: None, or the clearance range of the lowest contact sphere above the ground the pose is shifted to;
# rollin: untimed steps before the warm-up; episode: restart from the initial states every `episode` steps (0 = never)
WORKLOADS = {
    "ant": dict(base_dz=(-0.1, 0.25), tilt=0.15, jitter=0.3, ground=None, rollin=20, episode=0),
    "quadruped": dict(base_dz=(0.0, 0.0), tilt=0.05, jitter=0.2, ground=(0.0, 0.005), rollin=0, episode=8),
    "atlas": dict(base_dz=(0.0, 0.0), tilt=0.05, jitter=0.1, ground=(0.0, 0.005), rollin=0, episode=8),
    "pendulum": dict(base_dz=(0.0, 0.0), tilt=0.0, jitter=0.3, ground=None, rollin=0, episode=0),
}


def min_clearance(mech, z):
    """signed distance of the lowest contact sphere to its half-space (collisions/sphere_halfspace.jl:34-36)"""
    zz = z.reshape(mech.Nb, 13)
    m = np.inf
    for c in mech.contacts:
        p = zz[c.body, 0:3] + Q.qrot(np.asarray(c.origin), zz[c.body, 6:10]) - np.asarray(c.offset)
        m = min(m, float(np.dot(np.asarray(c.normal), p)) - c.radius)
    return m


def synthetic_batch(mech, B, seed, name=None):
    """Seeded synthetic states (SURVEY.md §8d): forward kinematics at jittered joint angles inside the limits, random base
    height / tilt, zero velocities (velocities and contacts develop during the untimed steps).  256 prototypes, sampled B times."""
    w = WORKLOADS.get(name or getattr(mech, "name", ""), WORKLOADS["ant"])
    rng = np.random.default_rng(seed)
    base = mech.minimal_coordinates(mech.z0)
    n_proto = min(B, 256)
    protos = np.zeros((n_proto, mech.nz))
    for e in range(n_proto):
        coords = {}
        for j in mech.joints:
            c = np.array(base[j.name], dtype=float)
            if j.nimpulses == 0:
                c[2] += rng.uniform(*w["base_dz"])
                c[3:6] += rng.normal(0.0, w["tilt"], 3) if w["tilt"] > 0 else 0.0
            elif j.input_dimension > 0:
                c = c + rng.uniform(-w["jitter"], w["jitter"], c.shape)
                if j.rot.nlimits:
                    lo, hi = j.rot.limit_lo, j.rot.limit_hi
                    c[j.tra.nfree:] = np.clip(c[j.tra.nfree:], lo + 0.05 * (hi - lo), hi - 0.05 * (hi - lo))
            coords[j.name] = c
        protos[e] = mech.forward_kinematics(coords)
        if w["ground"] is not None and mech.contacts:  # no initial penetration: the lowest contact sphere just above the ground
            protos[e].reshape(mech.Nb, 13)[:, 2] += rng.uniform(*w["ground"]) - min_clearance(mech, protos[e])
    Z = protos[rng.integers(0, n_proto, B)].copy()
    return Z, rng


DUMP_BYTES_PER_RECORD = 15_000_000  # --dump-outputs: the headline and at most three sub-records stay under 64 MB in all


def last_step_outputs(z_next, status, iters, Fz=None, Fu=None, budget=DUMP_BYTES_PER_RECORD):
    """What a caller of the timed step received from the last timed step, as float64 host arrays: next states, status and Newton
    iterations of every environment, or of a fixed seeded sample of them where that would exceed half of `budget`; the gradients
    (grad mode) of a fixed seeded sample of environments that fits in the other half."""
    import torch
    B = z_next.shape[0]

    def rows(per_env, seed):
        n = min(B, max(1, budget // 2 // per_env))
        sel = np.arange(B) if n == B else np.sort(np.random.default_rng(seed).choice(B, size=n, replace=False))
        return torch.from_numpy(sel).to(z_next.device)

    sel = rows(8 * (z_next.shape[1] + 2), 11)
    out = {"z_next": z_next[sel], "status": status[sel], "iters": iters[sel]}
    if Fz is not None:
        gsel = rows(8 * (Fz[0].numel() + Fu[0].numel()), 12)
        out.update(Fz=Fz[gsel], Fu=Fu[gsel])
    return {k: v.double().cpu().numpy() for k, v in out.items()}


def random_inputs(mech, rng, T, B, scale):
    U = rng.uniform(-scale, scale, (T, B, mech.nu))
    off = 0
    for j in mech.joints:
        if j.nimpulses == 0:
            U[:, :, off:off + j.input_dimension] = 0.0
        off += j.input_dimension
    return U


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, smax, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [x for x in sm if smax and x > 0.6 * smax]  # samples while the GPU was clocked up (the timed loops)
        return {"sm_mhz": float(np.median(busy or sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------- CPU port (oracle) timing
def host_threads():
    """Threads this process may really use: the CPU affinity mask capped by the cgroup CPU quota (os.cpu_count() reports the
    machine, not the lease: round 1 asked for 128 threads on a box that delivered 9 core-equivalents)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(p)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    if quota:
        n = max(1, min(n, int(np.ceil(quota))))
    return n, quota


def cpu_port_step(mech, Z, U, opts, threads, mode):
    """One timed pass of the CPU port over the sample.  Returns (env-steps/s, seconds, (Zn, status, iters))."""
    from oracle import oracle as orc  # test infrastructure: the timed CPU baseline and the parity checker, nothing else
    threads = max(1, min(threads, Z.shape[0]))
    t0 = time.perf_counter()
    if mode == "grad":  # step! + get_maximal_gradients with the reference's dense solmat \ datamat (gradients/state.jl:99)
        out = orc.step_grad_batch_threads(mech, Z, U, opts, threads)
    else:
        out = orc.step_batch_threads(mech, Z, U, opts, threads)
    dt = time.perf_counter() - t0
    return Z.shape[0] / dt, dt, out


def cpu_baseline_record(mech, Zs, Us, opts, threads, quota, mode, what):
    v_all, dt_all, out = cpu_port_step(mech, Zs, Us, opts, threads, mode)
    n1 = min(Zs.shape[0], 128 if mode == "fwd" else 32)
    v_one, _, _ = cpu_port_step(mech, Zs[:n1], Us[:n1], opts, 1, mode)
    rec = {"value": v_all, "unit": "env-steps/s", "cores": threads, "kind": "port",
           "sample": f"{Zs.shape[0]} environments x 1 {what} of the timed batch on {threads} threads ({dt_all:.2f} s); C++ port of the Julia reference (Julia is not "
                     f"installed); single thread: {v_one:.0f} env-steps/s on {n1} environments",
           "single_thread_value": v_one, "delivered_thread_equivalents": v_all / v_one, "cgroup_cpu_quota": quota}
    return rec, out


def parity_record(Zo, so, io, Zg, sg, ig):
    """GPU vs CPU oracle on the same environments of the timed batch: mismatch rates, not a pass / fail."""
    n = len(so)
    conv = (so == 0) & (sg == 0)
    same = conv & (ig == io)
    err = np.abs(Zg - Zo).max(axis=1)
    return {"sample": int(n), "status_mismatch": int((sg != so).sum()), "failed_gpu": int((sg != 0).sum()), "failed_oracle": int((so != 0).sum()),
            "iters_mismatch": int((conv & (ig != io)).sum()), "iters_mismatch_rate": float((conv & (ig != io)).sum() / max(1, n)),
            "max_abs_dz_same_iters": float(err[same].max(initial=0.0)), "median_abs_dz_same_iters": float(np.median(err[same])) if same.any() else None,
            "max_abs_dz_converged": float(err[conv].max(initial=0.0)), "mean_iters_gpu": float(ig.mean()), "mean_iters_oracle": float(io.mean()),
            "checker": "oracle/ (CPU port of the reference algorithm; parity unpinned against Julia, DESIGN.md section 2)"}


def peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_summary(mech_name, mode):
    p = os.path.join(ROOT, "profiles", "ncu_summary.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(f"{mech_name}_{mode}", {})
        except Exception:
            return {}
    return {}


# ---------------------------------------------------------------------------------------------------- one configuration on the GPU(s)
def run_config(name, B, mode, steps, warmup, rank, local_rank, world, dist, threads, quota, headline, e2e_steps=10, cpu_sample=2048, sample_clocks=True,
               outputs=None):
    import torch
    from dojo_jl_b200.solver import BatchedStepper
    mech = dj.get_mechanism(name)
    w = WORKLOADS[name]
    opts = capi.solver_options()
    dev = torch.device("cuda", local_rank)
    stepper = BatchedStepper(mech, B, device=local_rank)
    Z0, rng = synthetic_batch(mech, B, 0xD0D0 + 1 + 1000 * rank, name)
    rollin, episode = w["rollin"], w["episode"]
    T = warmup + steps
    U_host = random_inputs(mech, rng, rollin + T, B, SCALE.get(name, 1.0))
    Z0d = torch.from_numpy(Z0).to(dev)
    Za, Zb = Z0d.clone(), torch.empty_like(Z0d)
    U = torch.from_numpy(U_host).to(dev)
    status = torch.zeros(B, dtype=torch.int32, device=dev)
    iters = torch.zeros(B, dtype=torch.int32, device=dev)
    ng = 12 * mech.Nb
    if mode == "grad":
        Fz = torch.empty((B, ng, ng), dtype=torch.float64, device=dev)
        Fu = torch.empty((B, mech.nu, ng), dtype=torch.float64, device=dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()
    # the one exchange of the path: every rank receives the next states of the whole batch (SURVEY.md 8e)
    gather = None
    if world > 1:
        from dojo_jl_b200.shard import StateGather
        gather = StateGather(stepper, B, mech.nz, rank, world, dist, dev)

    def launch(t, zin, zout):
        kw = dict(dstatus=status.data_ptr(), diters=iters.data_ptr(), stream=stream.cuda_stream)
        if gather is not None and gather.fused:  # z_next written straight into every rank's gathered buffer by the step kernel
            if mode == "fwd":
                gather.step(zin.data_ptr(), U[t].data_ptr(), zout.data_ptr(), opts, **kw)
            else:
                gather.step_grad(zin.data_ptr(), U[t].data_ptr(), zout.data_ptr(), Fz.data_ptr(), Fu.data_ptr(), opts, **kw)
            return
        if mode == "fwd":
            stepper.step_device(zin.data_ptr(), U[t].data_ptr(), zout.data_ptr(), B, opts, **kw)
        else:
            stepper.step_grad_device(zin.data_ptr(), U[t].data_ptr(), zout.data_ptr(), Fz.data_ptr(), Fu.data_ptr(), B, opts, **kw)
        if gather is not None:
            gather.exchange(zout, stream)

    for t in range(rollin):  # untimed, forward only
        stepper.step_device(Za.data_ptr(), U[t].data_ptr(), Zb.data_ptr(), B, opts, stream=stream.cuda_stream)
        Za, Zb = Zb, Za
    torch.cuda.synchronize()
    k_global = 0

    def maybe_restart():
        nonlocal Za
        if episode and k_global % episode == 0:
            Za.copy_(Z0d)

    for t in range(warmup):
        maybe_restart()
        launch(rollin + t, Za, Zb)
        Za, Zb = Zb, Za
        k_global += 1
    torch.cuda.synchronize()

    sampler = ClockSampler(local_rank) if (rank == 0 and sample_clocks) else None
    if sampler:
        sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches0 = stepper.launch_count
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    it_sum, fails = 0.0, 0
    timed_inputs = []  # (state, input index) of the timed steps: replayed by the end-to-end loop and the parity sample
    for k in range(steps):
        maybe_restart()
        if k < 1 + e2e_steps:
            timed_inputs.append((Za.clone(), rollin + warmup + k))
        flush.fill_(k & 0xFF)  # L2 flush, outside the event pair
        ev[k][0].record(stream)
        launch(rollin + warmup + k, Za, Zb)
        ev[k][1].record(stream)
        Za, Zb = Zb, Za
        it_sum += float(iters.float().mean().item())
        fails += int((status != 0).sum().item())
        k_global += 1
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    launches = stepper.launch_count - launches0
    clocks = sampler.stop() if sampler else None
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = float(sum(step_ms))
    if world > 1:
        tmax = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        total_ms = float(tmax.item())
    ms_per_step = total_ms / steps
    value = world * B / (ms_per_step * 1e-3)
    Z_final_stepwise = Za.clone()
    if outputs is not None:  # --dump-outputs
        outputs.update(last_step_outputs(Za, status, iters, *((Fz, Fu) if mode == "grad" else ())))

    what = "forward-only step!" if mode == "fwd" else "step! + get_maximal_gradients"
    rec = {"workload": f"{name} (DojoEnvironments defaults, h={mech.timestep}) batch={B}/GPU {what}", "mechanism": name, "batch_per_gpu": B, "global_batch": B * world,
           "mode": mode, "value": value, "unit": "env-steps/s", "ms_per_step": ms_per_step, "steps": steps, "warmup": warmup,
           "mean_newton_iters": it_sum / steps, "failed_env_steps": fails, "failed_rate": fails / (steps * B), "gpu_launches": int(launches),
           "states": {k: (list(v) if isinstance(v, tuple) else v) for k, v in w.items()},
           "step_ms_min_max": [float(min(step_ms)), float(max(step_ms))]}
    if gather is not None:
        rec["gather"] = gather.describe()

    # ---- fused rollout (dojo_rollout_async): the same steps of the same batch in ONE launch (no per-step launch / tail)
    if headline and mode == "fwd" and world == 1 and not episode:
        Zs0, i0 = timed_inputs[0]
        Zr, Zf = Zs0.clone(), torch.empty_like(Zs0)
        Ur = U[i0: i0 + steps].contiguous()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stepper.rollout_device(Zr.data_ptr(), Ur.data_ptr(), Zf.data_ptr(), B, steps, opts, stream=stream.cuda_stream)  # warm
        torch.cuda.synchronize()
        flush.fill_(1)
        r0.record(stream)
        stepper.rollout_device(Zr.data_ptr(), Ur.data_ptr(), Zf.data_ptr(), B, steps, opts, stream=stream.cuda_stream)
        r1.record(stream)
        torch.cuda.synchronize()
        rms = r0.elapsed_time(r1) / steps
        rec["rollout"] = {"value": B / (rms * 1e-3), "unit": "env-steps/s", "ms_per_step": rms, "steps_fused": steps, "launches": 1,
                          "final_state_matches_stepwise": bool(torch.equal(Zf, Z_final_stepwise))}

    # ---- minimal-coordinate path (SURVEY 8 f1): the maps either side of step! and step_minimal_coordinates! = map + step + map
    if headline and mode == "fwd" and world == 1 and mech.nu > 0:
        Zs0 = timed_inputs[0][0]
        Xd = torch.empty((B, 2 * mech.nu), dtype=torch.float64, device=dev)
        Zd = torch.empty_like(Zs0)
        m0, m1, m2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        stepper.maximal_to_minimal_device(Zs0.data_ptr(), Xd.data_ptr(), B, stream=stream.cuda_stream)  # warm
        stepper.minimal_to_maximal_device(Xd.data_ptr(), Zd.data_ptr(), B, stream=stream.cuda_stream)
        torch.cuda.synchronize()
        flush.fill_(2)
        m0.record(stream)
        stepper.maximal_to_minimal_device(Zs0.data_ptr(), Xd.data_ptr(), B, stream=stream.cuda_stream)
        m1.record(stream)
        stepper.minimal_to_maximal_device(Xd.data_ptr(), Zd.data_ptr(), B, stream=stream.cuda_stream)
        m2.record(stream)
        torch.cuda.synchronize()
        bytes_map = 8 * B * (2 * mech.nu + mech.nz)
        t_mm, t_mM = m0.elapsed_time(m1), m1.elapsed_time(m2)
        rec["minimal_coordinates"] = {"maximal_to_minimal_us": 1e3 * t_mm, "minimal_to_maximal_us": 1e3 * t_mM,
                                      "maximal_to_minimal_GBps": bytes_map / (t_mm * 1e-3) / 1e9, "minimal_to_maximal_GBps": bytes_map / (t_mM * 1e-3) / 1e9,
                                      "round_trip_max_abs_err": float((Zd - Zs0).abs().max().item()),
                                      "step_minimal_ms": ms_per_step + t_mm + t_mM, "step_minimal_value": B / ((ms_per_step + t_mm + t_mM) * 1e-3), "unit": "env-steps/s"}

    # ---- end to end through the public host API: pinned host buffers, H2D + kernel(s) + D2H (+ the gather at N > 1) inside the timed
    #      region; the SAME states and inputs as the first device-timed steps (the kernels are deterministic), same L2 flush before
    def pinned(shape, dtype):
        return torch.empty(shape, dtype=dtype, pin_memory=True).numpy()
    ne2e = min(e2e_steps, len(timed_inputs) - 1)
    Zh, Zh2 = pinned((B, mech.nz), torch.float64), pinned((B, mech.nz), torch.float64)
    Uh = pinned((B, mech.nu), torch.float64)
    sth, ith = pinned((B,), torch.int32), pinned((B,), torch.int32)
    if mode == "grad":
        Fzh, Fuh = pinned((B, ng, ng), torch.float64), pinned((B, mech.nu, ng), torch.float64)
    Zallh = pinned((world * B, mech.nz), torch.float64) if world > 1 else None

    def host_call():
        if mode == "fwd":
            stepper.step(Zh, Uh, opts, out=(Zh2, sth, ith))
            loss = float(Zh2[0, 2])  # the result is on the host
        else:
            stepper.step_grad(Zh, Uh, opts, out=(Zh2, Fzh, Fuh, sth, ith))
            loss = float(Fzh[0, 0, 0])
        if gather is not None:  # every rank ends with the next states of the whole batch on its host
            gather.exchange_host(Zh2, Zallh)
            loss += float(Zallh[-1, 2])
        return loss

    # Step k is timed right after an untimed host call of step k - 1: the library orders the work queue by the iteration counts of the
    # previous call (longest first), so the timed call has the information the device-timed step k had -- the previous TIME STEP of the
    # same batch.  (Round 1 warmed up with the very step it then timed: a perfect longest-first order, hence an end-to-end figure
    # 5 % above the device-timed one.)
    e2e_t = []
    for k in range(1, ne2e + 1):
        Zh[:] = timed_inputs[k - 1][0].cpu().numpy()
        Uh[:] = U_host[timed_inputs[k - 1][1]]
        host_call()
        Zh[:] = timed_inputs[k][0].cpu().numpy()
        Uh[:] = U_host[timed_inputs[k][1]]
        if world > 1:
            dist.barrier()
        flush.fill_(k & 0xFF)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        host_call()
        e2e_t.append(time.perf_counter() - t0)
    e2e_ms = 1e3 * float(np.mean(e2e_t))
    if world > 1:
        tmax = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        e2e_ms = float(tmax.item())
    h2d = 8 * B * (mech.nz + mech.nu)
    d2h = 8 * B * mech.nz + 8 * B + (8 * B * (ng * ng + ng * mech.nu) if mode == "grad" else 0) + (8 * world * B * mech.nz if world > 1 else 0)
    rec["e2e"] = {"value": world * B / (e2e_ms * 1e-3), "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms,
                  "calls_timed": len(e2e_t), "what": "stepper.step / step_grad with page-locked host buffers (the call a user makes), wall clock after a device synchronize; "
                  "replays device-timed steps 1.. (identical states, inputs and work-queue order: each timed call follows an untimed call of the step before it)"}
    # the device-timed number for exactly the replayed steps, so that the two clocks can be compared like for like
    rec["e2e"]["device_ms_same_steps"] = float(np.mean([step_ms[k] for k in range(1, ne2e + 1)]))

    if rank == 0:
        # ---- roofline of the dominant kernel(s) of this configuration
        peak, peak_src = peak_hbm()
        algo = ALGO_BYTES[mode](mech) * B
        kernel_ms = float(np.mean(step_ms))
        achieved = algo / (kernel_ms * 1e-3) / 1e9
        nc = ncu_summary(name, mode)
        rec["roofline"] = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": nc.get("dram_bytes_per_launch"),
                           "peak_source": peak_src, "algorithmic_bytes_per_launch": algo, "kernel_ms": kernel_ms,
                           "issue_active_pct": nc.get("issue_active_pct"), "fp64_pipe_pct": nc.get("fp64_pipe_pct"),
                           "note": "the KKT system lives in shared memory: latency bound (dependent fp64 block algebra, 8 warps/SM), not HBM bound (DESIGN.md section 5)"}
        # ---- CPU port on a bounded sample of the FIRST timed step + parity of the GPU result on the same environments
        try:
            Zs0, i0 = timed_inputs[0]
            n = min(B, cpu_sample if mode == "fwd" else max(64, cpu_sample // 8))
            sel = np.sort(np.random.default_rng(7).choice(B, size=n, replace=False))
            Zs, Us = Zs0.cpu().numpy()[sel], U_host[i0][sel]
            cpu, out = cpu_baseline_record(mech, Zs, Us, opts, threads, quota, mode, "step!" if mode == "fwd" else "step! + get_maximal_gradients")
            Zg, sg, ig = stepper.step(Zs, Us, opts)
            rec["cpu_baseline"] = cpu
            rec["parity"] = parity_record(out[0], out[1], out[2], Zg, sg, ig)
        except Exception as ex:  # the oracle is test infrastructure; its absence must not break the product bench
            rec["cpu_baseline"] = {"value": None, "unit": "env-steps/s", "cores": 0, "kind": "port", "sample": f"unavailable: {ex}"}
        rec["clocks"] = clocks
        rec["shared_bytes_per_env"] = stepper.shared_bytes_per_env
    if gather is not None:
        gather.close()
    stepper.close()
    del stepper
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mech", default=None)
    ap.add_argument("--batch", type=int, default=None, help="environments per GPU")
    ap.add_argument("--mode", default=None, choices=["fwd", "grad"])
    ap.add_argument("--no-sub", action="store_true", help="headline record only")
    ap.add_argument("--cpu-threads", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of every record returned to DIR/<record>.<array>.npy (float64, < 64 MB in all)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    args.warmup = max(args.warmup, 3)
    custom = args.mech is not None or args.batch is not None or args.mode is not None
    name, B, mode = args.mech or "ant", args.batch or 4096, args.mode or "fwd"

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    mech = dj.get_mechanism(name)
    opts = capi.solver_options()
    metric = "env-steps/sec (forward step!)" if mode == "fwd" else "env-steps/sec (forward + IFT gradients)"
    threads, quota = host_threads()
    if args.cpu_threads:
        threads = args.cpu_threads
    what = "forward-only step!" if mode == "fwd" else "step! + get_maximal_gradients"
    config = {"workload": f"{name} (DojoEnvironments defaults, h={mech.timestep}) batch={B}/GPU {what}",
              "mechanism": name, "batch_per_gpu": B, "global_batch": B * world, "mode": mode,
              "solver": "rtol=1e-6 btol=1e-4 max_iter=50 max_ls=10 (reference defaults)",
              "l2": "L2 flushed (256 MiB write) before every timed step", "sharding": f"env batch split over {world} GPU(s), one gather of the next states per step"}

    # ------------------------------------------------------------------ reference arm: CPU port of the reference on the host cores
    if args.impl == "reference":
        if rank != 0:
            return
        w = WORKLOADS[name]
        bound = min(B, 1024 if mode == "fwd" else 128)  # bounded sample per step: the whole run ends within a few minutes
        Z0, rng = synthetic_batch(mech, B, 0xD0D0 + 1, name)
        T = args.warmup + args.steps
        U = random_inputs(mech, rng, w["rollin"] + T, B, SCALE.get(name, 1.0))
        Z0, U = Z0[:bound], U[:, :bound]
        Z = Z0.copy()
        for t in range(w["rollin"]):  # same roll-in as the GPU arm: the state advances with U[t]
            _, _, out = cpu_port_step(mech, Z, U[t], opts, threads, "fwd")
            Z = out[0]
        times, its, fails = [], [], 0
        for k in range(T):
            if w["episode"] and k % w["episode"] == 0:
                Z = Z0.copy()
            v, dt, out = cpu_port_step(mech, Z, U[w["rollin"] + k], opts, threads, mode)
            Z = out[0]
            if k >= args.warmup:
                times.append(dt)
                its.append(float(out[2].mean()))
                fails += int((out[1] != 0).sum())
        v_one, _, _ = cpu_port_step(mech, Z[:min(bound, 64 if mode == "fwd" else 16)], U[w["rollin"]][:min(bound, 64 if mode == "fwd" else 16)], opts, 1, mode)
        sec = float(np.mean(times))
        value = bound / sec
        ms = 1e3 * sec * (B / bound)
        line = {"impl": "reference", "metric": metric, "value": value, "unit": "env-steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config,
                "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": threads, "kind": "port",
                                 "sample": f"{bound} environments x 1 {what} per timed step on {threads} host threads (affinity / cgroup quota {quota}); C++ port of the "
                                           f"Julia reference (Julia is not installed); single thread {v_one:.0f} env-steps/s",
                                 "single_thread_value": v_one, "delivered_thread_equivalents": value / v_one},
                "mean_newton_iters": float(np.mean(its)), "failed_env_steps": fails, "failed_rate": fails / (args.steps * bound),
                "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ our arm
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback (use --impl reference for the CPU port)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    dumps = {} if args.dump_outputs else None
    head = run_config(name, B, mode, args.steps, args.warmup, rank, local_rank, world, dist, threads, quota, headline=True,
                      outputs=None if dumps is None else dumps.setdefault("headline", {}))
    subs = {}
    if not custom and not args.no_sub:
        ksub, wsub = min(args.steps, 10), 3
        if world == 1:
            plan = [("ant_grad", "ant", 4096, "grad"), ("quadruped_grad", "quadruped", 8192, "grad"), ("atlas_fwd", "atlas", 4096, "fwd")]
        else:
            plan = [("c4_ant_grad", "ant", 8192, "grad"), ("c3_atlas_fwd", "atlas", 4096, "fwd")]
        for key, n2, b2, m2 in plan:
            try:
                r = run_config(n2, b2, m2, ksub, wsub, rank, local_rank, world, dist, threads, quota, headline=False, e2e_steps=2,
                               cpu_sample=512 if n2 != "atlas" else 128, sample_clocks=False,
                               outputs=None if dumps is None else dumps.setdefault(key, {}))
                subs[key] = r
            except Exception as ex:  # a sub-record must never take the headline down
                subs[key] = {"error": f"{type(ex).__name__}: {ex}"}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    line = {"metric": metric, "value": head["value"], "unit": "env-steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
            "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "clocks": head.get("clocks"), "roofline": head.get("roofline"), "cpu_baseline": head.get("cpu_baseline"),
            "parity": head.get("parity"), "rollout": head.get("rollout"), "minimal_coordinates": head.get("minimal_coordinates"),
            "mean_newton_iters": head["mean_newton_iters"], "failed_env_steps": head["failed_env_steps"], "failed_rate": head["failed_rate"],
            "shared_bytes_per_env": head.get("shared_bytes_per_env"), "gather": head.get("gather"), "step_ms_min_max": head["step_ms_min_max"],
            "sub_records": subs}
    if dumps is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for rec_name, arrays in dumps.items():
            for arr_name, a in arrays.items():
                np.save(os.path.join(args.dump_outputs, f"{rec_name}.{arr_name}.npy"), a)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
