#!/usr/bin/env python
"""bench.py - env-steps/s of the vid2player3d rollout hot path on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--envs 8192] [--impl b200|reference] [--legs all|none|amass,dual,ppo,tables]
  torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...        (one rank per GPU, NCCL)

PRIMARY WORKLOAD (value / ms_per_step / roofline / e2e): BASELINE config 3, "vid2player federer single-player": 8192 envs per GPU,
SMPL humanoid + welded racket + tennis ball per env, sim dt 1/60 x controlFrequencyInv 2 x substeps 6 (12 articulated substeps per
env step), ball launcher pool + racket / ground contact, reward return_w_estimate with estimator tables on the device, episode
length 300.  One "step" = one high-level `PhysicsMVAEController.step(actions)`:
    motion generator (resident kinematic target stream + the MVAE mixture-of-experts decoder forward, random weights of the
    reference's shapes) -> SMPL FK targets -> 734-d imitation obs -> low-level policy MLP 734-1024-1024-512-75 (random weights,
    tcgen05 layers) -> PD targets + articulated step + ball (one physics launch) -> state views -> high-level obs / reward /
    reset FSM,
followed by `reset(done ids)` like the rl_games loop does every step.  The whole step is ONE CUDA-graph replay, the reset a
second one.  Random high-level policy: actions ~ clamp(N(0,1), -5, 5), [N, 35].

Timing: every timed step sits between two CUDA events on the launching stream; a 256 MiB memset flushes the L2 between timed
steps (outside the event pairs).  value = envs x K / sum(step times), max over ranks.  Clocks are sampled in-process through NVML
every 2 ms during the timed region.

SECONDARY LEGS (flat top-level keys, every N): config 2 (embodied_pose amass_im at 8192 envs), config 5 (dual 2 x 8192 paired envs
over the box, sharded 16384 / N per GPU), config 4 (djokovic_im PPO: horizon-32 rollouts + minibatch updates with the gradient
all-reduce inside the timed region).

--impl reference: the CPU restatement of the SAME primary workload (oracle/, "kind": "port": Isaac Gym cannot be installed) on the
host cores, all 8192 envs, honouring --steps / --warmup.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "env-steps/sec"
ALGO_BYTES_CFG3 = 10900   # SURVEY.md 8(d): config 3 / 5, bytes per env step (derivation in DESIGN.md 5)
ALGO_BYTES_CFG2 = 9792    # SURVEY.md 8(d): configs 2 / 4
PHYS_BYTES_CFG3 = (164 + 69 + 6 + 164 + 338 + 78) * 4   # the physics launch's share: state + PD targets + wrench in, state / rigid-body / contact rows out
HORIZON = 32
WORKLOAD = ("vid2player federer single-player (BASELINE config 3): 8192 envs/GPU, SMPL humanoid + racket + ball, dt 1/60 x 2 x substeps 6, "
            "return_w_estimate, episode 300, MVAE decoder + low-level policy MLP (reference shapes, random weights) inside the step")


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=200)
    p.add_argument("--warmup", type=int, default=20)
    p.add_argument("--envs", type=int, default=8192, help="envs per GPU (primary workload)")
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--legs", default="all", help="secondary legs: all | none | comma list of amass,dual,ppo,tables")
    p.add_argument("--cpu-sample-envs", type=int, default=1024, help="envs of the in-line cpu_baseline sample (N=1 b200 arm)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned to its caller (primary workload, "
                   "rank 0) as DIR/<name>.npy, at most 64 MB (a seeded sample of envs above that): the same arguments give the same "
                   "inputs, so two builds can be compared output for output")
    return p.parse_args()


PHYS_KERNEL_NAME = {"tmem": "step_kernel_tmem (56 envs per SM, lane-private body fields in tensor memory: one round for 8192 envs)",
                    "packed": "step_kernel_packed<split> (28 envs per SM, two rounds)", "packed3": "step_kernel_packed3", "lane": "step_kernel"}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            d = json.load(f)
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock / throttle reasons sampled in-process through NVML every `period` s while the timed region runs."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index, period=0.002):
        self.idx, self.period, self.rows, self.stop_flag, self.th, self.err = gpu_index, period, [], False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[gpu_index]) if vis and vis.split(",")[gpu_index].strip().isdigit() else gpu_index
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as ex:
            self.nv, self.err = None, repr(ex)[:120]

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                self.rows.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM), nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                                  if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)))
            except Exception as ex:
                self.err = repr(ex)[:120]
                return
            time.sleep(self.period)

    def sample_now(self):
        """one sample from the calling thread (the timed loop calls it between two launches: the GPU is busy with the previous step,
        the host thread is not - the background thread alone can be starved of the GIL by the launch loop)"""
        if self.nv is None:
            return
        try:
            nv = self.nv
            self.rows.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM), nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                              if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)))
        except Exception as ex:
            self.err = repr(ex)[:120]

    def start(self):
        if self.nv is not None:
            self.th = threading.Thread(target=self._loop, daemon=True)
            self.th.start()

    def stop(self):
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + str(self.err)], "samples": 0}
        self.stop_flag = True
        self.th.join(timeout=1.0)
        sm = sorted(r[0] for r in self.rows)
        bits = 0
        for r in self.rows:
            bits |= int(r[1])
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "samples": len(sm),
                "reasons": sorted(n for b, n in self.REASONS.items() if bits & b), "source": "NVML in-process: one sample per timed step from the launch loop + a %.0f ms background thread" % (self.period * 1e3)}


# ================================================================================================ workloads
def federer_env(envs, device_index, seed=10, policy="b200nn", player="stream+decoder", **v2p_over):
    import torch
    from vid2player3d_b200.configs import SIM_PARAMS, v2p_cfg
    from vid2player3d_b200.tasks import PhysicsMVAEController
    torch.manual_seed(seed)
    cfg = v2p_cfg(envs, **v2p_over)
    cfg["seed"] = seed
    cfg["env"]["motion_player"] = player
    cfg["env"]["low_level_policy"] = policy
    env = PhysicsMVAEController(cfg, SIM_PARAMS, 1, "cuda", device_index, True)
    env.reset()
    return env


def amass_task(envs, device_index, seed, asset="smpl_mesh_humanoid_amass_v1"):
    import torch
    from vid2player3d_b200 import model_compiler, motion_lib
    from vid2player3d_b200.configs import SIM_PARAMS, im_cfg
    from vid2player3d_b200.tasks import HumanoidSMPLIM
    model = model_compiler.load_compiled(asset)
    flat = motion_lib.synthetic(model_compiler.load_compiled("smpl_mesh_humanoid_amass_v1"), num_motions=64, num_frames=300, seed=7, sigma=0.05)
    torch.manual_seed(seed)
    task = HumanoidSMPLIM(im_cfg(envs, flat, episodeLength=300, asset=f"mjcf/{asset}.xml"), SIM_PARAMS, 1, "cuda", device_index, True)
    return model, flat, task


def timed_steps(step_fn, K, flush, sampler=None):
    """K calls of step_fn(i), each between two CUDA events, L2 flushed before each (outside the pair) -> list of ms"""
    import torch
    evs = []
    for i in range(K):
        if sampler is not None and i > 0:
            sampler.sample_now()           # while step i-1 runs on the GPU
        if flush is not None:
            flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step_fn(i)
        e1.record()
        evs.append((e0, e1))
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in evs]


def amass_leg(envs, device_index, rank, K, W, flush):
    """BASELINE config 2 at the metric's 8192 envs: embodied_pose amass_im, random policy, reset(all) every 32 steps (in the timed
    region) like ImitatorAgent.play_steps (agents/im_agent.py:305-409)."""
    import torch
    _, _, task = amass_task(envs, device_index, 7 + rank)
    g = torch.Generator(device=task.device).manual_seed(100 + rank)
    pool = [torch.rand(envs, task.num_actions, device=task.device, generator=g) * 2 - 1 for _ in range(8)]
    task.reset()

    def step(i):
        if i % HORIZON == 0:
            task.reset()
        task.step(pool[i % 8])
    for i in range(max(W, 3)):
        step(i)
    torch.cuda.synchronize()
    task._env.set_kernel_timing(True)
    ms = timed_steps(step, K, flush)
    phys_ms, _ = task._env.kernel_ms()
    task._env.set_kernel_timing(False)
    resets = int(task._terminate_buf.sum())
    # standing / tracking workload next to the random policy: the action of embodied_pose IS the PD target (clamp(action, q +- lim),
    # humanoid_smpl_im.py:391-396), so feeding the current MoCap target pose makes the humanoid track its reference motion
    track = torch.zeros(envs, task.num_actions, device=task.device)
    task.reset()

    def track_step(i):
        track[:, :task.num_dof].copy_(task._target_dof_pos)
        task.step(track)
    for i in range(4):
        track_step(i)
    ms_track = timed_steps(track_step, min(K, 24), flush)   # within the 32 frames that follow the sampled start times
    fallen_track = int(task._terminate_buf.sum())
    total = sum(ms)
    return {"amass_im_env_steps_per_s": envs * K / (total * 1e-3), "amass_im_ms_per_step": total / K, "amass_im_physics_kernel_ms": phys_ms,
            "amass_im_roofline_frac_hbm": ALGO_BYTES_CFG2 * envs / (total / K * 1e-3) / 1e9 / peaks()[0],
            "amass_im_envs_terminated_at_end": resets,
            "amass_im_tracking_env_steps_per_s": envs * len(ms_track) / (sum(ms_track) * 1e-3),
            "amass_im_tracking_envs_terminated": fallen_track,
            "amass_im_workload": f"embodied_pose amass_im: {envs} envs/GPU, 24 bodies / 69 dof, synthetic MoCap 64x300 frames, dt 1/60 x 2 x substeps 2, "
                                 f"random policy U(-1,1) with reset(all) every {HORIZON} steps; `tracking` = PD targets at the MoCap target pose (standing / tracking humanoids)"}


def dual_leg(envs, device_index, rank, K, W, flush):
    """BASELINE config 5: federer vs djokovic, paired envs (2k, 2k+1), full rally FSM; `envs` = this rank's share of the box's
    2 x 8192 paired envs (pairs never straddle GPUs, dist.shard_envs(pair=True))."""
    import torch
    from vid2player3d_b200.configs import SIM_PARAMS, v2p_dual_cfg
    from vid2player3d_b200.tasks import PhysicsMVAEControllerDual
    torch.manual_seed(10 + rank)
    cfg = v2p_dual_cfg(envs)
    cfg["env"]["motion_player"] = "stream"
    cfg["env"]["low_level_policy"] = "b200nn"
    env = PhysicsMVAEControllerDual(cfg, SIM_PARAMS, 1, "cuda", device_index, True)
    env.reset()
    acts = [torch.clamp(torch.randn(envs, env.num_actions, device=env.device), -5, 5) for _ in range(8)]
    stats = {"resets": 0}

    def step(i):
        env.step(acts[i % 8])
        done = env.reset_buf.nonzero(as_tuple=False).flatten()
        stats["resets"] += len(done)
        env.reset(done)
    for i in range(4):
        step(i)
    env.enable_cuda_graph()
    for i in range(max(W, 3)):
        step(i)
    torch.cuda.synchronize()
    stats["resets"] = 0
    ms = timed_steps(step, K, flush)
    total = sum(ms)
    return {"dual_env_steps_per_s": envs * K / (total * 1e-3), "dual_ms_per_step": total / K, "dual_envs_this_gpu": envs,
            "dual_pair_resets_per_step": stats["resets"] / 2 / K,
            "dual_workload": "vid2player federer_djokovic dual (BASELINE config 5): 2 x 8192 paired envs over the box, sharded "
                             f"{envs} envs / GPU, two assets (two physics launches per step), dual reset FSM, ball hand-over through the "
                             "incoming-ball table, low-level policy MLP in the step, step + reset as CUDA graphs"}


def ppo_leg(envs, device_index, rank, world, iters=2):
    """BASELINE config 4: embodied_pose djokovic_im PPO training step.  Horizon-32 rollout of `envs` envs per GPU (actor + critic
    forward each step, reset of finished envs), GAE, then mini_epochs 6 x 16 minibatches of 512 actors x 32 steps (cfg/djokovic_im.yaml:
    horizon_length 32, minibatch_size 512, mini_epochs 6, e_clip 0.2, critic_coef 5, grad_norm 50, lr 1e-5) with ONE flat gradient
    all-reduce per minibatch (dist.GradAllReducer = the Horovod optimizer.synchronize of common_agent.py:388-395) inside the timed
    region.  Networks: the reference's MLP sizes (actor 734-1024-1024-512-75 with fixed sigma, critic 734-1024-1024-512-1; 4.69 M
    parameters = 18.8 MB of fp32 gradients), plain PyTorch fp32 like the reference (mixed_precision False).  The context encoder of
    the reference network is not part of this leg."""
    import torch
    import torch.distributed as dist
    from vid2player3d_b200 import dist as D
    _, _, task = amass_task(envs, device_index, 7 + rank, asset="smpl_mesh_humanoid_djokovic")
    dev = task.device
    torch.manual_seed(0)                       # same initial weights on every rank (then broadcast like hvd.broadcast_parameters)

    def mlp(out):
        return torch.nn.Sequential(torch.nn.Linear(734, 1024), torch.nn.ReLU(), torch.nn.Linear(1024, 1024), torch.nn.ReLU(),
                                   torch.nn.Linear(1024, 512), torch.nn.ReLU(), torch.nn.Linear(512, out))
    A = task.num_actions
    net = torch.nn.ModuleDict(dict(actor=mlp(A), critic=mlp(1))).to(dev)
    D.broadcast_parameters(net)
    params = list(net.parameters())
    opt = torch.optim.Adam(params, lr=1e-5, eps=1e-8)
    red = D.GradAllReducer(params)
    sigma = torch.full((A,), -1.756, device=dev).exp()
    H, MB_ENVS, EPOCHS = HORIZON, 512, 6
    n_mb = envs // MB_ENVS
    obs_b = torch.zeros(H, envs, 734, device=dev)
    act_b, mu_b = torch.zeros(H, envs, A, device=dev), torch.zeros(H, envs, A, device=dev)
    val_b, rew_b, done_b, logp_b = (torch.zeros(H, envs, device=dev) for _ in range(4))
    nb = task._num_lib_bodies
    c = lambda x: x.contiguous()  # noqa: E731

    def policy_obs():   # compute_humanoid_observations_imitation on the live state (what the reference network does inside forward)
        rbs = task._rigid_body_state.view(envs, -1, 13)[:, :nb]
        return task.compute_imitation_obs(c(rbs[..., 0:3]), c(rbs[..., 3:7]), task._target_rb_pos, task._target_rb_rot, c(task._dof_pos),
                                          c(task._dof_vel), task._target_dof_pos, c(rbs[..., 7:10]), c(rbs[..., 10:13]),
                                          task._reset_ref_motion_bodies, True, True)

    def neglogp(a, mu):
        return (0.5 * (((a - mu) / sigma) ** 2).sum(-1) + 0.5 * A * 1.8378770664093453 + sigma.log().sum())

    ar_ev, tm = [], {}

    def iteration():
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        with torch.no_grad():
            for t in range(H):
                o = policy_obs()
                mu, v = net["actor"](o), net["critic"](o).squeeze(-1)
                a = mu + sigma * torch.randn_like(mu)
                obs_b[t], act_b[t], mu_b[t], val_b[t], logp_b[t] = o, a, mu, v, neglogp(a, mu)
                task.step(torch.clamp(a, -1.0, 1.0))
                rew_b[t], done_b[t] = task.rew_buf, task.reset_buf.float()
                ids = task.reset_buf.nonzero(as_tuple=False).flatten()      # env_reset(done_indices), im_agent.py:375-378
                if len(ids):
                    task.reset(ids)
            last_v = net["critic"](policy_obs()).squeeze(-1)
            adv, gae = torch.zeros_like(val_b), torch.zeros(envs, device=dev)
            for t in reversed(range(H)):                                     # discount_values, gamma 0.99 tau 0.95
                nv = last_v if t == H - 1 else val_b[t + 1]
                nd = 1.0 - done_b[t]
                gae = rew_b[t] + 0.99 * nv * nd - val_b[t] + 0.99 * 0.95 * nd * gae
                adv[t] = gae
            ret = adv + val_b
            adv = (adv - adv.mean()) / (adv.std() + 1e-8)                    # per-rank normalisation like the reference (im_agent.py:469-471)
        e[1].record()
        for _ in range(EPOCHS):
            perm = torch.randperm(envs, device=dev)
            for m in range(n_mb):
                idx = perm[m * MB_ENVS:(m + 1) * MB_ENVS]
                o, a = obs_b[:, idx].reshape(-1, 734), act_b[:, idx].reshape(-1, A)
                mu, v = net["actor"](o), net["critic"](o).squeeze(-1)
                nl = neglogp(a, mu)
                ratio = torch.exp(logp_b[:, idx].reshape(-1) - nl)
                ad = adv[:, idx].reshape(-1)
                a_loss = torch.max(-ad * ratio, -ad * torch.clamp(ratio, 0.8, 1.2)).mean()
                c_loss = ((v - ret[:, idx].reshape(-1)) ** 2).mean()
                b_loss = (torch.clamp_min(mu - 1.0, 0) ** 2 + torch.clamp_max(mu + 1.0, 0) ** 2).sum(-1).mean()
                loss = a_loss + 5.0 * c_loss + 10.0 * b_loss
                red.zero_grad()
                loss.backward()
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record()
                red.synchronize()                                            # the one collective of the path
                a1.record()
                ar_ev.append((a0, a1))
                torch.nn.utils.clip_grad_norm_(params, 50.0)
                opt.step()
        e[2].record()
        return e
    task.reset()
    iteration()                      # warm-up (cuBLAS heuristics, NCCL channels, allocator)
    ar_ev.clear()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    evs = [iteration() for _ in range(iters)]
    torch.cuda.synchronize()
    roll = sum(e[0].elapsed_time(e[1]) for e in evs)
    upd = sum(e[1].elapsed_time(e[2]) for e in evs)
    ar = sum(a.elapsed_time(b) for a, b in ar_ev)
    t = torch.tensor([roll, upd, ar], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    roll, upd, ar = t.tolist()
    n_ar = max(len(ar_ev), 1)
    frames = envs * H * iters * world
    busbw = (2.0 * (world - 1) / world) * red.nbytes / (ar / n_ar * 1e-3) / 1e9 if world > 1 and ar > 0 else None
    return {"ppo_rollout_env_steps_per_s": frames / (roll * 1e-3), "ppo_total_fps": frames / ((roll + upd) * 1e-3),
            "ppo_rollout_ms_per_iter": roll / iters, "ppo_update_ms_per_iter": upd / iters, "ppo_allreduce_ms": ar / n_ar,
            "ppo_allreduce_ms_per_iter": ar / iters, "ppo_allreduce_bytes": red.nbytes, "ppo_allreduce_calls_per_iter": n_ar // iters,
            "ppo_allreduce_busbw_gbps": busbw, "ppo_iters": iters,
            "ppo_workload": f"embodied_pose djokovic_im PPO (BASELINE config 4): {envs} envs/GPU, horizon {H}, {EPOCHS} mini-epochs x {n_mb} "
                            f"minibatches of {MB_ENVS} actors, actor + critic MLPs of the reference's sizes (4.69 M parameters), fp32 PyTorch, "
                            "one flat NCCL all-reduce of the gradient per minibatch inside the timed region"}


def ball_tables_leg(reps=3):
    """SURVEY.md 8f-2: the reference's offline ball data products at their full sizes, one launch each"""
    import torch
    from vid2player3d_b200 import ball_gen as G
    dev = "cuda:%d" % torch.cuda.current_device()

    def best_ms(fn):
        fn()
        torch.cuda.synchronize()
        ms = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        return min(ms)
    vh, vv, vs = G._mesh(G.traj_out_params.VEL_X_RANGE, G.traj_out_params.VEL_Y_RANGE, G.traj_out_params.VSPIN_RANGE, device=dev)
    n = int(vh.shape[0])
    ms_out = best_ms(lambda: G.simulate_without_bounce(vh, vv, vs, device=dev))
    del vh, vv, vs
    hh, vx, vz, sp = G._mesh(G.traj_in_params.HEIGHT_RANGE, G.traj_in_params.VEL_X_RANGE, G.traj_in_params.VEL_Y_RANGE,
                             G.traj_in_params.VSPIN_RANGE, device=dev)
    m = int(hh.shape[0])
    pos = torch.stack([torch.zeros_like(hh), torch.zeros_like(hh), hh], 1)
    vel = torch.stack([torch.zeros_like(hh), vx, vz], 1)
    ms_in = best_ms(lambda: G.simulate(pos, vel, sp, num_frames=50, first_comp=1, device=dev))
    return {"ball_out_tables_rows": n, "ball_out_tables_ms": ms_out, "ball_out_tables_gbps": n * (120 * 4 + 12) / 1e9 / (ms_out * 1e-3),
            "ball_in_table_rows": m, "ball_in_table_ms": ms_in}


# ================================================================================================ CPU arm (oracle/, test infrastructure)
def _cpu_worker(conn, n, seed, threads):
    """One process = one slice of `n` envs of the primary workload stepped by the CPU restatement: numpy FK targets
    (oracle/ref_port_v2p.smpl_to_sim) -> numpy 734-d obs (oracle/ref_port) -> fp32 policy MLP (torch CPU, 1 thread) -> float64
    articulated step + ball, 12 substeps (oracle/physics_ref.c) -> numpy state views + high-level obs + reward."""
    import numpy as np
    import torch
    torch.set_num_threads(threads)
    os.environ["OMP_NUM_THREADS"] = str(threads)
    from oracle import physics_ref, ref_port as R, ref_port_v2p as V
    from vid2player3d_b200 import abi, model_compiler
    from vid2player3d_b200.tasks.humanoid_smpl_im_mvae import SMPL_NAMES, SMPL_PARENTS
    physics_ref.set_threads(threads)
    rng = np.random.default_rng(seed)
    model = model_compiler.canonical_racket_last(model_compiler.load_compiled("smpl_mesh_humanoid_federer"))
    ms, verts = abi.pack_model(model, float(model["mass"].sum()) / 90.0)
    cfg = abi.make_cfg(model, substeps=6, task_mode=1, pd_mode=1, contact_bodies=(), key_bodies=(), enable_early_termination=False,
                       ball=dict(spin_scale=5.0, ball_e_racket=0.9, ball_e_ground=0.7, ball_mu_racket=0.5, ball_mu_ground=0.6, ball_body_contact=1,
                                 ball_e_body=0.45, ball_mu_body=0.6))
    physics_ref.set_hull_faces(*abi.pack_faces(model, verts))              # exact ball / hull contact, as the GPU arm's task installs
    names = [str(x) for x in model["body_names"]][:24]
    s2m = np.array([SMPL_NAMES.index(q) for q in names])
    rest = np.zeros((24, 3))
    for i in range(24):
        rest[i] = model["offset"][i] + (rest[model["parent"][i]] if model["parent"][i] >= 0 else 0)
    rest = np.stack([rest[names.index(q)] for q in SMPL_NAMES]).astype(np.float32)
    rest_n = np.broadcast_to(rest, (n, 24, 3)).copy()
    g = torch.Generator().manual_seed(seed)
    dims = [734, 1024, 1024, 512, 75]
    W = [((torch.rand(dims[i + 1], dims[i], generator=g) * 2 - 1) / dims[i] ** 0.5 * (0.1 if i == 3 else 1.0)) for i in range(4)]
    Bv = [torch.zeros(dims[i + 1]) for i in range(4)]
    # state: standing humanoids at the FK pose of a smooth random-walk target stream, a ball in flight per env
    aa = 0.05 * rng.normal(size=(n, 24, 3))
    rootp = np.stack([rng.uniform(-4, 4, n), rng.uniform(-15, -11, n), np.full(n, 0.95)], -1).astype(np.float32)
    root = np.zeros((n, 13))
    root[:, :3], root[:, 3:7] = rootp, [0.5, 0.5, 0.5, 0.5]
    q, qd = np.zeros((n, 69)), np.zeros((n, 69))
    ball = np.zeros((n, 13))
    ball[:, :3] = np.stack([rng.uniform(-4, 4, n), rng.uniform(10, 12, n), rng.uniform(1, 1.5, n)], -1)
    ball[:, 6], ball[:, 7:10] = 1.0, np.stack([rng.normal(0, 1, n), -rng.uniform(20, 28, n), rng.uniform(2, 5, n)], -1)
    hits = np.zeros(n, np.int32)
    mb = np.zeros((n, 11), np.float32)
    prev = {"root": rootp.copy(), "rot": None}
    traj = rng.normal(size=(n, 100, 3)).astype(np.float32)
    tgt = np.tile(np.array([0.0, 10.0, 0.0], np.float32), (n, 1))
    rb = np.zeros((n, 25, 13), np.float32)
    rb[..., 6] = 1.0
    dt = np.float32(1 / 30)

    def one_step():
        nonlocal aa, rb
        aa = 0.97 * aa + 0.02 * rng.normal(size=aa.shape)
        Rm = V.angle_axis_to_rotation_matrix(aa.reshape(-1, 3).astype(np.float32)).reshape(n, 24, 3, 3)
        out = V.smpl_to_sim(rootp, Rm, rest_n, np.array(SMPL_PARENTS), s2m, dt, prev["root"] if prev["rot"] is not None else None, prev["rot"])
        t_dof, t_pos, t_rot = out[2], out[6], out[7]
        prev["rot"] = t_rot
        obs = R.compute_humanoid_observations_imitation(rb[:, :24, 0:3], rb[:, :24, 3:7], t_pos, t_rot, q.astype(np.float32), qd.astype(np.float32),
                                                        t_dof, rb[:, :24, 7:10], rb[:, :24, 10:13], mb, True, True)
        with torch.no_grad():
            x = torch.from_numpy(np.clip(obs, -5, 5).astype(np.float32))
            for i in range(4):
                x = x @ W[i].T + Bv[i]
                if i < 3:
                    x = torch.relu(x)
            act = np.clip(x.numpy(), -1, 1)
        pd = np.clip(t_dof + act[:, :69], q - 0.5 * np.pi, q + 0.5 * np.pi).astype(np.float64)
        wrench = np.zeros((n, 6))
        rbo, _ = physics_ref.control_step(ms, verts, cfg, root, q, qd, pd, wrench, ball=ball, hits=hits)
        rb = rbo.astype(np.float32)
        contact = hits > 0
        st = V.update_state_from_sim(np.concatenate([rb, np.zeros((n, 1, 13), np.float32)], 1), root.astype(np.float32), ball.astype(np.float32),
                                     ball[:, 7:10].astype(np.float32), contact, "eastern")
        V.controller_obs(rb, st["root_pos"], st["root_vel"], st["racket_normal"], traj, tgt, 10, True)
        back = ball[:, 1] < -20                                      # relaunch balls that left the court behind the player
        if back.any():
            k = int(back.sum())
            ball[back, :3] = np.stack([rng.uniform(-4, 4, k), rng.uniform(10, 12, k), rng.uniform(1, 1.5, k)], -1)
            ball[back, 7:10] = np.stack([rng.normal(0, 1, k), -rng.uniform(20, 28, k), rng.uniform(2, 5, k)], -1)
    try:
        one_step()
        conn.send("ready")
        while True:
            cmd = conn.recv()
            if cmd[0] == "stop":
                return
            t0 = time.perf_counter()
            for _ in range(cmd[1]):
                one_step()
            conn.send(time.perf_counter() - t0)
    except Exception as ex:   # noqa: BLE001
        import traceback
        conn.send("error: " + repr(ex)[:300] + traceback.format_exc()[-600:])


def cpu_arm(envs, steps, warmup, procs=None):
    """the primary workload on the host cores: `procs` worker processes, each stepping envs / procs envs (physics + task logic +
    policy) on one core; no per-step barrier between workers (favours the CPU).  Returns (env-steps/s, ms per step, procs)."""
    import multiprocessing as mp
    from oracle import physics_ref
    physics_ref.build()
    cores = os.cpu_count() or 1
    procs = procs or max(1, min(cores // 2 if cores > 8 else cores, 64))   # one worker per physical core (SMT siblings hurt, round 1)
    procs = min(procs, envs)
    per = [envs // procs + (1 if i < envs % procs else 0) for i in range(procs)]
    ctx = mp.get_context("spawn")
    conns, ps = [], []
    for i in range(procs):
        a, b = ctx.Pipe()
        p = ctx.Process(target=_cpu_worker, args=(b, per[i], 100 + i, 1), daemon=True)
        p.start()
        conns.append(a)
        ps.append(p)
    for c in conns:
        r = c.recv()
        if r != "ready":
            raise RuntimeError("cpu worker failed: " + str(r))

    def run(k):
        t0 = time.perf_counter()
        for c in conns:
            c.send(("step", k))
        for c in conns:
            r = c.recv()
            if isinstance(r, str):
                raise RuntimeError("cpu worker failed: " + r)
        return time.perf_counter() - t0
    if warmup > 0:
        run(warmup)
    dt = run(steps)
    for c in conns:
        c.send(("stop",))
    for p in ps:
        p.join(timeout=5)
    return envs * steps / dt, dt / steps * 1e3, procs


DUMP_CAP_BYTES = 64 * 10 ** 6


def dump_outputs(path, outputs, n):
    """outputs: per-env float32 arrays [n, ...] -> path/<name>.npy.  Above DUMP_CAP_BYTES in all, the same fixed, seeded sample of
    env rows is written for every array, and its env ids as path/env_ids.npy."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    row_bytes = sum(v.nbytes // n for v in outputs.values())
    rows = min(n, (DUMP_CAP_BYTES - 4096 - 8 * n) // row_bytes)            # 4096: the .npy headers; 8 n: env_ids
    if rows < n:
        ids = np.sort(np.random.default_rng(0).choice(n, rows, replace=False))
        outputs = {k: v[ids] for k, v in outputs.items()}
        outputs["env_ids"] = ids.astype(np.float64)
    for k, v in outputs.items():
        np.save(os.path.join(path, k + ".npy"), v)


# ================================================================================================ main
def main():
    args = parse()
    # stdout carries exactly ONE line, the JSON: anything a library prints there meanwhile goes to stderr instead
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(obj) + "\n").encode())

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores = os.cpu_count() or 1
    N, K, W = args.envs, args.steps, max(args.warmup, 3)
    config = {"workload": WORKLOAD, "envs_per_gpu": N, "sim": "dt 1/60 x controlFreqInv 2 x substeps 6", "high_level_obs": 257, "low_level_obs": 734,
              "l2": "flushed (256 MiB memset) between timed steps; per-step CUDA events summed"}

    if args.impl == "reference":
        if rank != 0:
            return
        v, ms_step, procs = cpu_arm(N, K, args.warmup)
        emit({"impl": "reference", "metric": METRIC, "value": v, "unit": "env-steps/s", "n_gpus": args.gpus, "steps": K, "warmup": args.warmup,
              "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64 physics / f32 task logic + policy",
              "data": "synthetic", "config": config,
              "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": procs, "kind": "port", "host_logical_cpus": cores,
                               "sample": f"all {N} envs x {K} steps; {procs} worker processes x 1 thread, each steps its env slice: numpy FK targets + 734-d obs, "
                                         "fp32 policy MLP, float64 articulated step + ball (12 substeps), numpy state views / high-level obs",
                               "note": "CPU restatement (oracle/) of the same step; the reference's Isaac Gym CPU pipeline cannot be installed (closed "
                                       "binary, py3.8) - stand-in, labelled as such"},
              "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        return

    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    legs = {"amass", "dual", "ppo", "tables"} if args.legs == "all" else (set() if args.legs == "none" else set(args.legs.split(",")))
    if world > 1:
        legs.discard("tables")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    env = federer_env(N, local_rank, seed=10 + rank)
    dev = env.device
    task = env._physics_player.task
    gen = torch.Generator(device=dev).manual_seed(100 + rank)
    pool = [torch.clamp(torch.randn(N, env.num_actions, device=dev, generator=gen), -5, 5) for _ in range(16)]
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    stats = {"resets": 0}

    def step_ids(i):
        env.step(pool[i % len(pool)])
        done = env.reset_buf.nonzero(as_tuple=False).flatten()     # the rl_games loop resets finished envs every step (id list = host sync)
        stats["resets"] += len(done)
        env.reset(done)

    def step(i, snap=None):
        env.step(pool[i % len(pool)])                              # one graph replay
        if snap is not None:                                       # --dump-outputs: the step's outputs before the reset rewrites them
            for k, src in step_outputs().items():
                snap[k].copy_(src)
        env.reset_done()                                           # reset(finished envs) from the device flags: mask + one graph replay
        # (step + reset captured as ONE graph measured 1.4 % slower than the two replays, profiles/r2z_notes.md: not kept)

    def step_outputs():
        return {"obs": env.obs_buf, "rew": env.rew_buf, "reset": env.reset_buf, "terminate": env.extras["terminate"],
                "sub_rewards": env.extras["sub_rewards"]}
    for i in range(4):
        step_ids(i)
    env.enable_cuda_graph(count_nodes=True)
    for i in range(W):
        step_ids(i)
    barrier()
    stats["resets"] = 0
    for i in range(8):
        step_ids(i)
    resets_per_step = stats["resets"] / 8
    for i in range(W):
        step(i)
    barrier()
    # ---------------- device-resident arm (`value`)
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = task._env.launch_count
    t_wall = time.perf_counter()
    prof = os.environ.get("B200_BENCH_PROFILE") == "1"      # tools/federer_launches.sh: ncu --profile-from-start off sees the timed loop only
    if prof:
        torch.cuda.cudart().cudaProfilerStart()
    dump = args.dump_outputs and rank == 0
    snap = {k: torch.empty_like(v) for k, v in step_outputs().items()} if dump else None
    timed_step = (lambda i: step(i, snap if i == K - 1 else None)) if dump else step
    step_ms = timed_steps(timed_step, K, flush, sampler)
    barrier()
    if prof:
        torch.cuda.cudart().cudaProfilerStop()
    wall = time.perf_counter() - t_wall
    clocks = sampler.stop()
    total_ms = sum(step_ms)
    # what the caller of the timed path receives from its last step: the step's outputs (taken before reset_done clears the flags of
    # the finished envs) and the observation after the reset, the one the policy sees next
    outputs = None
    if dump:
        snap["obs_after_reset"] = env.obs_buf
        outputs = {k: v.detach().float().cpu().numpy() for k, v in snap.items()}
    # the physics launch alone (dominant kernel): the SAME rollout continued for 10 steps with the step run eagerly (an event pair
    # inside b200env_step cannot live in a graph), L2 flushed before every step as in the timed loop
    g_saved, env._graph = env._graph, None
    task._env.set_kernel_timing(True)
    for i in range(10):
        flush.zero_()
        step(i)
    phys_ms, phys_n = task._env.kernel_ms()
    task._env.set_kernel_timing(False)
    env._graph = g_saved
    # back-to-back (hot L2), single event pair: informational
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        step(i)
    e1.record()
    barrier()
    hot_ms = e0.elapsed_time(e1)

    # ---------------- end-to-end arm: PhysicsMVAEController.step / reset with HOST buffers
    host_act = [p.cpu().pin_memory() for p in pool[:4]]
    host_rew = torch.empty(N, dtype=torch.float32).pin_memory()
    host_reset = torch.empty(N, dtype=torch.long).pin_memory()
    dev_act = [torch.empty(N, env.num_actions, device=dev) for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)

    def e2e_strict(k):
        for i in range(k):
            dev_act[0].copy_(host_act[i % 4], non_blocking=True)
            env.step(dev_act[0])
            host_rew.copy_(env.rew_buf, non_blocking=True)
            host_reset.copy_(env.reset_buf, non_blocking=True)
            torch.cuda.current_stream().synchronize()                 # the caller consumes reward / reset on the host every step
            done = host_reset.nonzero(as_tuple=False).flatten()       # ... and resets the finished envs from the HOST flags
            env.reset(done.to(dev, non_blocking=True) if len(done) else done.to(dev))

    def e2e_pipelined(k):
        """same API and bytes; the upload of step t+1's actions rides a side stream under step t, reward / reset flags of step t are
        read on the host while step t+1 runs (one step of latency on the host's view, what an async actor loop does)"""
        main = torch.cuda.current_stream()
        ev_up = [torch.cuda.Event(), torch.cuda.Event()]
        ev_free = [torch.cuda.Event(), torch.cuda.Event()]
        ev_out = torch.cuda.Event()
        with torch.cuda.stream(copy_stream):
            dev_act[0].copy_(host_act[0], non_blocking=True)
            ev_up[0].record(copy_stream)
        for i in range(k):
            b = i & 1
            main.wait_event(ev_up[b])
            env.step(dev_act[b])
            ev_free[b].record(main)
            env.reset_done()                                          # reset of the finished envs from the DEVICE flags: no host round trip
            with torch.cuda.stream(copy_stream):                      # next actions up while this step runs
                if i >= 1:
                    copy_stream.wait_event(ev_free[b ^ 1])
                dev_act[b ^ 1].copy_(host_act[(i + 1) % 4], non_blocking=True)
                ev_up[b ^ 1].record(copy_stream)
            if i > 0:
                ev_out.synchronize()                                  # reward / reset of step i-1 are on the host now
            host_rew.copy_(env.rew_buf, non_blocking=True)
            host_reset.copy_(env.reset_buf, non_blocking=True)
            ev_out.record(main)
        ev_out.synchronize()

    def timed(fn, k):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        a.record()
        fn(k)
        b.record()
        barrier()
        return max(a.elapsed_time(b), (time.perf_counter() - t0) * 1e3 * 0.0)   # device time between the first and the last op
    e2e_strict(W)
    e2e_ms = timed(e2e_strict, K)
    e2e_pipelined(W)
    e2e_pipe_ms = timed(e2e_pipelined, K)

    t = torch.tensor([total_ms, hot_ms, e2e_ms, e2e_pipe_ms, phys_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, hot_ms, e2e_ms, e2e_pipe_ms, phys_ms = t.tolist()

    # ---------------- secondary legs (every rank takes part; rank 0 reports max-over-ranks times)
    extra = {}
    free = lambda: (torch.cuda.synchronize(), torch.cuda.empty_cache())   # noqa: E731
    step_launches = task._env.launch_count - launches0
    graph_nodes = getattr(env, "graph_kernel_nodes", None)
    reset_nodes = getattr(env, "reset_graph_kernel_nodes", None)
    kform = task._env.kernel_form
    del env, task
    free()

    def run_leg(name, fn):
        if name not in legs:
            return
        try:
            barrier()
            r = fn()
            keys = [k for k, v in r.items() if isinstance(v, float) and ("_ms" in k)]
            if world > 1 and keys:
                tt = torch.tensor([r[k] for k in keys], device=dev, dtype=torch.float64)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                mx = dict(zip(keys, tt.tolist()))
                for k in keys:                      # throughput keys follow the slowest rank
                    rate = k.replace("_ms_per_step", "_env_steps_per_s")
                    if rate in r and r[k] > 0:
                        r[rate] = r[rate] * r[k] / mx[k]
                    r[k] = mx[k]
            extra.update(r)
        except Exception as ex:   # a secondary measurement must never break the contract line
            import traceback
            extra[name + "_error"] = repr(ex)[:200] + " | " + traceback.format_exc()[-300:]
        free()
    Ks = min(K, 200)
    run_leg("amass", lambda: amass_leg(N, local_rank, rank, Ks, W, flush))
    dual_total = 2 * 8192
    if dual_total % world == 0 and (dual_total // world) % 2 == 0:
        run_leg("dual", lambda: dual_leg(dual_total // world, local_rank, rank, min(Ks, 96), W, flush))
    run_leg("ppo", lambda: ppo_leg(N, local_rank, rank, world))
    if world == 1:
        run_leg("tables", ball_tables_leg)
    for k in ("amass_im_env_steps_per_s", "amass_im_tracking_env_steps_per_s"):
        if k in extra and world > 1:
            extra[k] *= world          # whole-job aggregate (weak scaling: every rank runs its own 8192 envs)
    if "dual_env_steps_per_s" in extra and world > 1:
        extra["dual_env_steps_per_s"] *= world   # 16384 paired envs in total, each rank steps its share
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    total_envs = N * world
    value = total_envs * K / (total_ms * 1e-3)
    peak, peak_src = peaks()
    ms_step = total_ms / K
    achieved = ALGO_BYTES_CFG3 * N / (ms_step * 1e-3) / 1e9
    out = {
        "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (physics, task logic); bf16 operands / f32 accumulate (policy, MVAE decoder)",
        "data": "synthetic", "config": config, "clocks": clocks,
        "e2e": {"value": total_envs * K / (e2e_ms * 1e-3), "unit": "env-steps/s", "h2d_bytes_per_step": N * 35 * 4 + 8 * 64, "d2h_bytes_per_step": N * 4 + N * 8,
                "api": "PhysicsMVAEController.step(actions) / reset(done ids): pinned host actions up, reward + reset flags down, host sync and reset ids "
                       "taken from the HOST flags every step (strict)", "ms_per_step": e2e_ms / K,
                "value_pipelined": total_envs * K / (e2e_pipe_ms * 1e-3),
                "pipelined": "same calls and bytes, action upload of step t+1 on a side stream under step t, flags of step t read while step t+1 runs"},
        "gpu_launches": int((graph_nodes + (reset_nodes or 0) + 1) * K) if graph_nodes else int(step_launches),
        "gpu_launches_note": "kernel nodes of the step graph + the reset graph (+ the mask kernel) x timed steps, counted from the graphs' DOT dumps; "
                             "our own kernels among them per step: 22 (step graph) + 7 (reset graph)",
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": {"tmem": 17394176, "packed": 8026112}.get(kform),
                     "traffic_note": "from_profile: dram__bytes_read.sum + dram__bytes_write.sum of ONE physics launch (the dominant kernel) in the "
                                     "ncu --set full captures profiles/r2i_step_kernel_ncu.md (step_kernel_packed) / profiles/r2t_tmem.md "
                                     "(step_kernel_tmem, capture r2ac_c3: 17.4 MB); not measured by this run",
                     "kernel": "one env step = one CUDA graph (motion targets, FK, 734-d obs, decoder + policy GEMMs, physics, post step); dominant launch "
                               + PHYS_KERNEL_NAME[kform], "kernel_ms": ms_step, "algorithmic_bytes_per_env_step": ALGO_BYTES_CFG3,
                     "dominant_kernel": {"name": PHYS_KERNEL_NAME[kform] + " (12 substeps + ball)", "ms": phys_ms, "launches_timed": 10,
                                         "share_of_step": phys_ms / ms_step if ms_step > 0 else None, "algorithmic_bytes_per_env": PHYS_BYTES_CFG3,
                                         "GBps": PHYS_BYTES_CFG3 * N / (phys_ms * 1e-3) / 1e9 if phys_ms > 0 else None},
                     "peak_source": peak_src,
                     "note": "latency / issue bound along the kinematic chain x 12 substeps, not HBM bound (DESIGN.md 5); the GEMMs of the step are "
                             "tensor-core work reported in DESIGN.md against the bf16 peak"},
        "value_hot_l2_back_to_back": total_envs * K / (hot_ms * 1e-3), "wall_s_timed_loop": wall, "resets_per_step": resets_per_step,
        "target_env_steps_per_s_1gpu": 4.0e6, "cuda_graph_kernel_nodes_per_step": graph_nodes, "cuda_graph_kernel_nodes_per_reset": reset_nodes,
    }
    out.update(extra)
    if not args.no_cpu_baseline and world == 1:   # contract: the CPU baseline is timed at N = 1 only, on a bounded sample
        try:
            v, _, procs = cpu_arm(args.cpu_sample_envs, 6, 1)
            out["cpu_baseline"] = {"value": v, "unit": "env-steps/s", "cores": procs, "kind": "port", "host_logical_cpus": cores,
                                   "sample": f"{args.cpu_sample_envs} of {N} envs x 6 steps of the primary workload ({procs} worker processes x 1 thread: numpy task "
                                             "logic + fp32 policy MLP + float64 articulated step with ball); `--impl reference` runs all envs"}
        except Exception as ex:
            out["cpu_baseline"] = {"value": None, "unit": "env-steps/s", "cores": None, "kind": "port", "sample": "failed: " + repr(ex)[:200]}
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs, N)
    emit(out)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
