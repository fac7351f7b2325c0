#!/usr/bin/env python
"""bench.py -- the hot path's headline measurement (DESIGN.md section 5).

Workload (BASELINE.json configs[2], the configuration the metric is quoted
on): Rainbow's replay path -- PrioritizedReplayBuffer(10**6, alpha=.5,
beta0=.4, num_steps=3, normalize_by_max="memory") holding synthetic Atari
transitions (84x84 uint8 frames, stack 4, frame-shared), minibatch 512.
One replay PASS = one pass of the hot path over one minibatch:

    priority write-back of the previous minibatch's TD errors -> prioritized
    sample(512) -> IS weights -> gather state/next_state as f32 (/255) +
    reward / discount / terminal / action            (ONE launch: k_replay_step)

One bench STEP = `--passes` (default 128) passes, so that the driver's
`--steps 20` times >= 2 500 passes (>= 1 s) and one host hiccup cannot move
the number.

metric   replay_samples_per_sec (whole job, all ranks), EXACT sampler
         (bit-identical indices to the reference)
value    device-resident: uniforms and TD errors already in HBM, C-ABI calls
e2e      public API with HOST buffers: buf.sample() -> batch_experiences() ->
         D2H of weights/reward/indices -> buf.update_errors(host float list)
roofline the PATH: SURVEY 8(d) algorithmic bytes per sample x samples per
         pass / pass time, vs MEASURED_PEAKS.json hbm_gbs; per-kernel
         sub-records from the stand-alone kernels
throughput_mode  the same pass with the PARALLEL sampler (all descents
         concurrent on the frozen tree, with replacement), its own roofline
secondary  BASELINE configs[1] (DQN B=32), [3] (PPO), [4] (SAC) lines
cpu_baseline / --impl reference: the reference's OWN classes on the host
         (oracle/_ref archive of pfnet/pfrl, kind "reference"; the pure-Python
         port oracle/pyport.py only if the archive is absent), bounded sample.

Launch: python bench.py [--gpus N --steps K --warmup W]; for N > 1 under
torch.distributed.run (one rank per GPU, NCCL only for the timing barrier and
max-reduction: the replay shards never exchange data -> "scaling": "weak").
--dump-outputs DIR writes the minibatch the last timed exact pass returned
(rank 0) as DIR/<name>.npy; the inputs are seeded, so two builds run with the
same arguments can be compared array for array.
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

FRAME = (84, 84)
STACK = 4
N_STEP = 3
GAMMA = 0.99
ALPHA = 0.5
BETA0 = 0.4
FRAME_BYTES = 84 * 84
# Algorithmic bytes per sampled experience, f32 outputs (SURVEY.md 8(d), C3):
# 7 distinct input frames (3-step, stack 4) + state and next_state as f32
# + scalars (action 8, reward 4, terminal 4, discount 4, weight 4, index 8)
ALGO_BYTES_GATHER = 7 * FRAME_BYTES + 2 * STACK * FRAME_BYTES * 4 + 32
# ... + tree traffic of the draw and of the write-back (~1.7 KB, SURVEY 8(d)) = 276.9 KB
ALGO_BYTES_TREE = 1684
ALGO_BYTES_PATH = ALGO_BYTES_GATHER + ALGO_BYTES_TREE
# uint8 batches out (x/255 folded into conv1): 7 frames read + 2 x 4 frames written = 107.6 KB
ALGO_BYTES_PATH_U8 = 7 * FRAME_BYTES + 2 * STACK * FRAME_BYTES + 32 + ALGO_BYTES_TREE
# --dump-outputs: rows of state / next_state written (2 x 64 x 113 KB = 14.5 MB)
DUMP_ROWS = 64


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--passes", type=int, default=128, help="replay passes per bench step")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--capacity", type=int, default=10 ** 6)
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--cpu-seconds", type=float, default=12.0,
                    help="CPU baseline budget (timed part)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-rainbow", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--no-rainbow-graph", action="store_true",
                    help="run the Rainbow learn step eagerly instead of as one CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the headline pass returned in its last timed step to "
                         "DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return args


# ---------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(np.max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------
# CPU arms (reference itself when oracle/_ref travelled, else the port)
# ---------------------------------------------------------------------------
def cpu_port_replay(capacity, batch, steps, warmup, seconds=None, pool=65536, seed=0):
    """Fallback: pure-Python port of the reference path (oracle/pyport.py)."""
    import torch
    from oracle.pyport import PyPrioritizedReplayBuffer, py_batch_experiences
    from pfrl_b200.utils.lazy_frames import LazyFrames

    torch.set_num_threads(min(16, os.cpu_count() or 1))
    rng = np.random.RandomState(seed)
    pool = min(pool, capacity + STACK + N_STEP)
    frames = rng.randint(0, 256, size=(pool, 1) + FRAME, dtype=np.uint8)
    flist = [frames[i] for i in range(pool)]
    buf = PyPrioritizedReplayBuffer(capacity, alpha=ALPHA, beta0=BETA0, betasteps=None,
                                    num_steps=N_STEP, normalize_by_max="memory")
    T = capacity + N_STEP - 1
    obs = [LazyFrames([flist[(t + j) % pool] for j in range(STACK)], stack_axis=0)
           for t in range(T + 1)]
    acts = rng.randint(0, 18, size=T)
    rews = rng.randint(-1, 2, size=T).astype(np.float64)
    trans = [dict(state=obs[t], action=int(acts[t]), reward=float(rews[t]),
                  next_state=obs[t + 1], next_action=None, is_state_terminal=False)
             for t in range(T)]
    buf.memory.bulk_load([trans[s:s + N_STEP] for s in range(capacity)],
                         rng.rand(capacity) + 0.05)
    phi = lambda x: np.asarray(x, dtype=np.float32) / 255  # noqa: E731
    dev = torch.device("cpu")
    np.random.seed(seed)

    def one():
        exps = buf.sample(batch)
        py_batch_experiences(exps, dev, phi, GAMMA)
        buf.update_errors([float(x) for x in np.abs(rng.randn(batch))])

    for _ in range(warmup):
        one()
    done = 0
    t0 = time.perf_counter()
    while done < steps:
        one()
        done += 1
        if seconds is not None and time.perf_counter() - t0 > seconds:
            break
    dt = time.perf_counter() - t0
    return {"samples_per_sec": done * batch / dt, "steps": done, "seconds": dt,
            "ms_per_step": 1e3 * dt / done, "kind": "port", "cores": 1}


def cpu_arm(capacity, batch, steps, warmup, seconds, rainbow_seconds):
    """(replay result, rainbow result or None) from the reference itself when it is
    importable (oracle/_ref archive or /root/reference), else from the port."""
    from oracle import ref_bench

    if ref_bench.kind() == "reference":
        r = ref_bench.replay_run(capacity, batch, steps, warmup, seconds=seconds, n_step=N_STEP,
                                 alpha=ALPHA, beta0=BETA0, normalize_by_max="memory", gamma=GAMMA)
        rb = None
        if rainbow_seconds:
            rb = ref_bench.rainbow_run(r["buffer"], r["frames"], batch, rainbow_seconds,
                                       num_envs=RAINBOW_ENVS,
                                       update_interval=RAINBOW_UPDATE_INTERVAL, gamma=GAMMA)
        r.pop("buffer", None)
        r.pop("frames", None)
        return r, rb
    r = cpu_port_replay(capacity, batch, steps, warmup, seconds=seconds)
    rb = None
    if rainbow_seconds:
        rb = cpu_port_rainbow(capacity, batch, rainbow_seconds)
    return r, rb


def cpu_sample_text(r, batch):
    what = ("the reference's own PrioritizedReplayBuffer.sample + batch_experiences + "
            "update_errors (pfnet/pfrl, oracle/_ref)" if r["kind"] == "reference" else
            "pure-Python port of the reference (oracle/pyport.py)")
    return ("%d passes (%.1f s) of sample(%d)+batch_experiences+update_errors, 1M-leaf tree, "
            "LazyFrames over a pool of 65536 frames; %s" % (r["steps"], r["seconds"], batch, what))


# ---------------------------------------------------------------------------
# Rainbow end-to-end training loop (train_agent_batch's inner loop, untimed
# bookkeeping stripped): act -> env.step -> observe (append / sample / update)
# ---------------------------------------------------------------------------
RAINBOW_ENVS = 16
RAINBOW_UPDATE_INTERVAL = 4


def make_rainbow_agent(buf, dev_index, batch, grad_sync=None, cuda_graph=False):
    import torch
    from pfrl_b200 import agents, explorers, nn as pnn, parallel, q_functions
    from pfrl_b200.utils.phi import RawU8

    torch.manual_seed(0)
    q = q_functions.DistributionalDuelingDQN(18, 51, -10, 10)
    pnn.to_factorized_noisy(q, sigma_scale=0.5)
    q.to(torch.device('cuda', dev_index))
    opt = torch.optim.Adam(q.parameters(), 6.25e-5, eps=1.5e-4, fused=True)
    agent = agents.CategoricalDoubleDQN(
        q, opt, buf, gpu=dev_index, gamma=GAMMA, explorer=explorers.Greedy(),
        minibatch_size=batch, replay_start_size=batch, target_update_interval=32000,
        update_interval=RAINBOW_UPDATE_INTERVAL, batch_accumulator="mean", phi=RawU8(),
        grad_sync=grad_sync, cuda_graph=cuda_graph)
    parallel.broadcast_parameters(agent.model)
    parallel.broadcast_parameters(agent.target_model)
    return agent


def rainbow_loop(agent, env, vec_steps):
    obss = env.reset()
    for _ in range(vec_steps):
        actions = agent.batch_act(obss)
        obss, rs, dones, infos = env.step(actions)
        resets = np.zeros(env.num_envs, dtype=bool)
        agent.batch_observe(obss, rs, dones, resets)
        obss = env.reset(np.logical_not(dones))


def k10_record():
    """The tensor-core path (csrc/gemm.cu, tcgen05 3xTF32, fp32 results) on the Rainbow layers
    at B = 512 against the fp32 library calls the reference configuration makes (TF32 off):
    median of 20 event-timed calls each, L2 flushed in between."""
    import torch
    import torch.nn.functional as F

    from pfrl_b200.ops.conv import geometry
    from pfrl_b200.ops.linear import gemm

    flush = torch.zeros(64 << 20, dtype=torch.float32, device="cuda")

    def t_us(fn, reps=20):
        for _ in range(3):
            fn()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
               for _ in range(reps)]
        for a, b in evs:
            flush.add_(1)
            a.record()
            fn()
            b.record()
        torch.cuda.synchronize()
        ts = sorted(a.elapsed_time(b) for a, b in evs)
        return round(ts[len(ts) // 2] * 1e3, 1)

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    x = torch.randn(512, 3136, device="cuda")
    w = torch.randn(1024, 3136, device="cuda")
    gy = torch.randn(512, 1024, device="cuda")
    out = {"arithmetic": "fp32 in / fp32 out, 3 x TF32 split on tcgen05.mma.kind::tf32",
           "main_stream_fwd_512x1024x3136_us": {"tcgen05": t_us(lambda: gemm(x, w)),
                                                "cublas_fp32": t_us(lambda: x @ w.t())},
           "main_stream_dX_us": {"tcgen05": t_us(lambda: gemm(gy, w, b_mn_major=True)),
                                 "cublas_fp32": t_us(lambda: gy @ w)},
           "main_stream_dW_us": {"tcgen05": t_us(lambda: gemm(gy, x, a_mn_major=True, b_mn_major=True)),
                                 "cublas_fp32": t_us(lambda: gy.t() @ x)}}
    xc = torch.rand(512, 32, 20, 20, device="cuda")
    wc = torch.randn(64, 32, 4, 4, device="cuda") * 0.05
    geo = geometry(512, 32, 20, 20, 64, 4, 4, 2, "cuda:0")
    out["conv2_fwd_512x32x20x20_us"] = {"tcgen05": t_us(lambda: geo.forward(xc, wc)),
                                         "cudnn_fp32": t_us(lambda: F.conv2d(xc, wc, stride=2))}
    x3 = torch.rand(512, 64, 9, 9, device="cuda")
    w3 = torch.randn(64, 64, 3, 3, device="cuda") * 0.05
    g3 = torch.randn(512, 64, 7, 7, device="cuda")
    geo3 = geometry(512, 64, 9, 9, 64, 3, 3, 1, "cuda:0")
    out["conv3_dgrad_us"] = {
        "tcgen05": t_us(lambda: geo3.dgrad(g3, w3)),
        "cudnn_fp32": t_us(lambda: torch.ops.aten.convolution_backward(
            g3, x3, w3, None, [1, 1], [0, 0], [1, 1], False, [0, 0], 1, [True, False, False]))}
    return out


def best_torch_threads():
    import torch
    from oracle.pyport_rainbow import RainbowNet

    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    cands = sorted({c for c in (4, 8, 16, 32, 64, avail) if c <= avail})
    net = RainbowNet()
    x = torch.rand(32, 4, 84, 84)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        for rep in range(2):
            t0 = time.perf_counter()
            net(x).sum().backward()
            dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def cpu_port_rainbow(capacity, batch, seconds, num_envs=RAINBOW_ENVS, pool=65536, seed=0):
    """Fallback CPU port of the Rainbow loop: pyport replay + plain-torch update."""
    import torch
    from oracle.pyport import PyPrioritizedReplayBuffer
    from oracle.pyport_rainbow import PyRainbow
    from pfrl_b200.utils.lazy_frames import LazyFrames

    best_torch_threads()
    rng = np.random.RandomState(seed)
    frames = rng.randint(0, 256, size=(pool, 1) + FRAME, dtype=np.uint8)
    flist = [frames[i] for i in range(pool)]
    buf = PyPrioritizedReplayBuffer(capacity, alpha=ALPHA, beta0=BETA0, betasteps=None,
                                    num_steps=N_STEP, normalize_by_max="memory")
    T = capacity + N_STEP - 1
    obs = [LazyFrames([flist[(t + j) % pool] for j in range(STACK)], stack_axis=0)
           for t in range(T + 1)]
    trans = [dict(state=obs[t], action=int(t % 18), reward=float((t % 3) - 1),
                  next_state=obs[t + 1], next_action=None, is_state_terminal=False)
             for t in range(T)]
    buf.memory.bulk_load([trans[s:s + N_STEP] for s in range(capacity)], rng.rand(capacity) + 0.05)
    agent = PyRainbow(buf, GAMMA, batch)
    np.random.seed(seed)
    cur = [LazyFrames([flist[rng.randint(pool)]] * STACK, stack_axis=0) for _ in range(num_envs)]
    t = 0
    env_steps = 0
    updates = 0

    def vec_step():
        nonlocal t, env_steps, updates
        acts = agent.act(cur)
        for i in range(num_envs):
            nf = flist[rng.randint(pool)]
            nxt = LazyFrames(cur[i]._frames[1:] + [nf], stack_axis=0)
            t += 1
            buf.append(cur[i], int(acts[i]), float(rng.randint(-1, 2)), nxt, None, False, env_id=i)
            cur[i] = nxt
            if t % RAINBOW_UPDATE_INTERVAL == 0:
                agent.update()
                updates += 1
        env_steps += num_envs

    vec_step()  # warm-up
    env_steps = updates = 0
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        vec_step()
    dt = time.perf_counter() - t0
    return {"env_steps_per_sec": env_steps / dt, "updates_per_sec": updates / dt,
            "ms_per_update": 1e3 * dt / max(updates, 1), "seconds": dt, "num_envs": num_envs,
            "threads": torch.get_num_threads(), "kind": "port"}


# ---------------------------------------------------------------------------
def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank != 0:
            return
        # each step = a bounded sample of the same workload: ONE pass (0.1-0.2 s of host
        # work), not `--passes` of them, so that K steps end within minutes
        r, rb = cpu_arm(args.capacity, args.batch, args.steps, args.warmup, None,
                        None if args.no_rainbow else 20.0)
        line = {
            "impl": "reference", "metric": "replay_samples_per_sec", "value": r["samples_per_sec"],
            "unit": "samples/s", "n_gpus": args.gpus, "steps": r["steps"], "warmup": args.warmup,
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64 priorities / u8->f32 frames", "data": "synthetic",
            "config": workload_config(args, 1, passes=1),
            "cpu_baseline": {"value": r["samples_per_sec"], "unit": "samples/s",
                             "cores": r["cores"], "kind": r["kind"],
                             "sample": cpu_sample_text(r, args.batch)},
            "e2e": {"value": r["samples_per_sec"], "unit": "samples/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0},
        }
        if rb is not None:
            line["rainbow"] = {"env_steps_per_sec": rb["env_steps_per_sec"],
                               "e2e_env_steps_per_sec": rb["env_steps_per_sec"],
                               "updates_per_sec": rb["updates_per_sec"],
                               "ms_per_update": rb["ms_per_update"], "num_envs": rb["num_envs"],
                               "torch_threads": rb["threads"], "kind": rb["kind"],
                               "sample": "%.0f s of act/append/sample(%d)/update on the host"
                                         % (rb["seconds"], args.batch)}
        print(json.dumps(line))
        return

    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)  # fail before the run, not after it
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    import ctypes

    from pfrl_b200 import _lib
    from pfrl_b200.replay_buffer import batch_experiences
    from pfrl_b200.replay_buffers import PrioritizedReplayBuffer
    from pfrl_b200.utils.phi import ScaleU8

    B, cap = args.batch, args.capacity
    K, W, R = args.steps, args.warmup, args.passes
    # ---- build and prefill the shard (untimed) ---------------------------------
    buf = PrioritizedReplayBuffer(cap, alpha=ALPHA, beta0=BETA0, betasteps=None,
                                  normalize_by_max="memory", num_steps=N_STEP, device=local_rank,
                                  max_batch=max(B, 512), part_capacity=cap + 4096,
                                  sample_mode="exact")
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + rank)
    rng = np.random.RandomState(100 + rank)
    T = cap + N_STEP - 1
    chunk = 1 << 17
    t_fill = time.perf_counter()
    done = 0
    while done < T:
        m = min(chunk, T - done)
        # each chunk is its own trajectory segment (stack extra frames up front)
        frames = torch.randint(0, 256, (m + STACK,) + FRAME, dtype=torch.uint8, device=dev,
                               generator=g)
        acts = rng.randint(0, 18, size=m).astype(np.int64)
        rews = rng.randint(-1, 2, size=m).astype(np.float64)
        term = rng.rand(m) < 1e-3
        term[-1] = True  # close the segment so that its tail is emitted
        buf.append_trajectory(frames, acts, rews, term)
        done += m
    # non-uniform priorities so that the tree descent is not degenerate
    for _ in range(64):
        np.random.seed(rng.randint(1 << 30))
        buf.sample(B)
        buf.update_errors(torch.rand(B, device=dev, dtype=torch.float32, generator=g) * 2)
    buf.store.flush()
    torch.cuda.synchronize()
    fill_s = time.perf_counter() - t_fill
    assert len(buf) == cap, (len(buf), cap)

    store = buf.store
    phi = ScaleU8()
    gp = buf._gamma_pow(GAMMA)
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident loops through the C ABI ---------------------------------
    # Argument objects are built ONCE (static output tensors, cached pointers); a
    # pass is two ctypes calls: b2rl_per_defer_errors (no launch) and
    # b2rl_replay_step (the one launch).
    L = _lib.load()
    cvp = ctypes.c_void_p
    stream = cvp(torch.cuda.current_stream().cuda_stream)
    obs_elems = STACK * FRAME_BYTES
    o_index = torch.empty(B, dtype=torch.int64, device=dev)
    o_weight = torch.empty(B, dtype=torch.float32, device=dev)
    o_state = torch.empty((B, obs_elems), dtype=torch.float32, device=dev)
    o_next = torch.empty((B, obs_elems), dtype=torch.float32, device=dev)
    o_action = torch.empty(B, dtype=torch.int64, device=dev)
    o_reward = torch.empty(B, dtype=torch.float32, device=dev)
    o_term = torch.empty(B, dtype=torch.float32, device=dev)
    o_disc = torch.empty(B, dtype=torch.float32, device=dev)
    batch_out = _lib.BatchOut(
        state=o_state.data_ptr(), next_state=o_next.data_ptr(), action=o_action.data_ptr(),
        reward=o_reward.data_ptr(), terminal=o_term.data_ptr(), discount=o_disc.data_ptr(),
        step_rewards=None, len=None)
    gp_arr = np.ascontiguousarray(gp, dtype=np.float64)
    n_pass = (K + W) * R
    # uniforms of all passes, resident in HBM before the timed region (drawn on the host
    # from the legacy MT stream, like np.random.uniform in collections/prioritized.py:302)
    u_dev = torch.from_numpy(rng.random_sample((min(n_pass, 4096), B))).to(dev)
    err_dev = torch.rand((16, B), device=dev, dtype=torch.float32, generator=g).abs() * 1.5
    err_ptrs = [cvp(err_dev[j].data_ptr()) for j in range(16)]
    h = store.h
    beta, scale = float(buf.beta), float(phi.b2rl_obs_scale)

    def fused_loop(mode, obs_mode=_lib.OBS_U8_TO_F32, K=K, W=W):
        sa = _lib.StepArgs(
            n=B, mode=mode, u=u_dev.data_ptr(), u_on_device=1, norm=_lib.NORM_MEMORY, beta=beta,
            gamma_pow_host=gp_arr.ctypes.data, obs_mode=obs_mode, obs_scale=scale,
            index_dev=o_index.data_ptr(), priority_dev=None, weight_dev=o_weight.data_ptr(),
            prob_dev=None, out=batch_out)
        sa_ref = ctypes.byref(sa)
        u_base, u_stride, u_rows = u_dev.data_ptr(), B * 8, u_dev.shape[0]
        state = {"i": 0}

        def one_pass():
            i = state["i"]
            state["i"] = i + 1
            sa.u = u_base + (i % u_rows) * u_stride
            _lib.check(L.b2rl_replay_step(h, sa_ref, stream))
            # the TD errors of this minibatch (inputs of the replay micro-benchmark):
            # registered now, written back at the head of the next launch
            _lib.check(L.b2rl_per_defer_errors(h, err_ptrs[i % 16], 0, B, ALPHA, 0.01, 0.0, 1.0))

        for _ in range(W * R):
            one_pass()
        barrier()
        t0, t1 = ev(), ev()
        t0.record()
        for _ in range(K * R):
            one_pass()
        t1.record()
        barrier()
        ph = (ctypes.c_uint64 * 36)()
        _lib.check(L.b2rl_step_times(h, ph, stream))  # %globaltimer stamps of the last launch
        _lib.check(L.b2rl_per_flush(h, stream))
        return t0.elapsed_time(t1), {"write_back_us": ph[0] / 1e3, "sampling_us": ph[1] / 1e3,
                                     "gather_after_last_draw_us": ph[2] / 1e3,
                                     "launch_us": ph[3] / 1e3,
                                     "write_back_phases_us_since_entry": {
                                         "cta0_entries_collected": ph[31] / 1e3,
                                         "cta0_subtree_stored": ph[32] / 1e3,
                                         "cta0_arrival_ticket": ph[33] / 1e3,
                                         "last_cta_roots_loaded": ph[34] / 1e3,
                                         "last_cta_flag_released": ph[35] / 1e3,
                                         **({"fine_cta0_unique_done": ph[28] / 1e3,
                                             "fine_cta0_siblings_in": ph[29] / 1e3,
                                             "fine_cta0_levels_done": ph[30] / 1e3}
                                            if os.environ.get("B2RL_WB_FINE") else {})},
                                     **({"sampler_cycles_per_draw": {
                                         "main_wait_scout": ph[4] / B, "main_decide": ph[5] / B,
                                         "main_wait_queue": ph[6] / B, "main_loads": ph[7] / B,
                                         "main_stores": ph[8] / B,
                                         "scout0_wait": ph[12] / (B / 4), "scout0_predict_issue": ph[13] / (B / 4),
                                         "scout0_arrive_sums_store": ph[14] / (B / 4),
                                         "ascent_wait": ph[20] / B, "ascent_work": ph[21] / B}}
                                        if ph[5] else {})}

    def last_step_outputs():
        """The minibatch the last exact pass handed its caller, as float32 / float64 arrays
        (indices and actions exactly); state / next_state as DUMP_ROWS rows drawn with a
        fixed seed (state_rows), which keeps the dump far below 64 MB."""
        rows = np.sort(np.random.RandomState(0).choice(B, min(B, DUMP_ROWS), replace=False))
        sel = torch.from_numpy(rows).to(dev)
        out = {"index": o_index.double(), "weight": o_weight, "action": o_action.double(),
               "reward": o_reward, "terminal": o_term, "discount": o_disc,
               "state": o_state[sel].view(-1, STACK, *FRAME),
               "next_state": o_next[sel].view(-1, STACK, *FRAME)}
        out = {k: v.cpu().numpy() for k, v in out.items()}
        out["state_rows"] = rows.astype(np.float64)
        return out

    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()  # samples SM clock / throttle reasons through all timed regions
    ms_value, phases_exact = fused_loop(_lib.SAMPLE_EXACT)
    # taken now: the loops below reuse the output tensors
    dumped = last_step_outputs() if args.dump_outputs and rank == 0 else None
    scout = store.info()["scout_hits"]
    ms_par, phases_par = fused_loop(_lib.SAMPLE_PARALLEL)
    # the same pass emitting uint8 batches (x/255 folded into the first conv layer): the
    # f32 output tensors are simply reused as byte buffers
    K8 = max(2, K // 4)
    ms_par_u8, phases_par_u8 = fused_loop(_lib.SAMPLE_PARALLEL, _lib.OBS_RAW, K=K8, W=1)

    # ---- stand-alone kernels (sub-records of the roofline): event pairs around each
    kern = {"sample_exact": [], "sample_parallel": [], "weights": [], "gather": [], "update": []}
    batch_out_ref = ctypes.byref(batch_out)
    u_host = rng.random_sample((24, B))
    for i in range(24):
        mode = _lib.SAMPLE_EXACT if i % 2 == 0 else _lib.SAMPLE_PARALLEL
        e = [ev() for _ in range(8)]
        e[0].record()
        _lib.check(L.b2rl_per_sample(h, cvp(u_host[i].ctypes.data), B, mode,
                                     cvp(o_index.data_ptr()), None, stream))
        e[1].record()
        e[2].record()
        _lib.check(L.b2rl_per_weights(h, beta, _lib.NORM_MEMORY, cvp(o_weight.data_ptr()), None,
                                      stream))
        e[3].record()
        e[4].record()
        _lib.check(L.b2rl_replay_gather(h, None, B, cvp(gp_arr.ctypes.data), _lib.OBS_U8_TO_F32,
                                        scale, batch_out_ref, stream))
        e[5].record()
        e[6].record()
        _lib.check(L.b2rl_per_update_errors(h, err_ptrs[i % 16], 0, B, ALPHA, 0.01, 0.0, 1.0,
                                            stream))
        e[7].record()
        if i >= 4:
            kern["sample_exact" if i % 2 == 0 else "sample_parallel"].append((e[0], e[1]))
            kern["weights"].append((e[2], e[3]))
            kern["gather"].append((e[4], e[5]))
            kern["update"].append((e[6], e[7]))
    torch.cuda.synchronize()
    kern_ms = {k: float(np.mean([a.elapsed_time(b) for a, b in v])) for k, v in kern.items()}

    # ---- e2e: public API with host buffers --------------------------------------
    np.random.seed(7 + rank)
    err_host = [[float(x) for x in np.abs(rng.randn(B))] for _ in range(8)]
    pinned = torch.empty((3, B), dtype=torch.float64).pin_memory()
    R_e2e = max(1, R // 2)

    def pass_e2e(i):
        exps = buf.sample(B)                      # host-drawn uniforms -> H2D, fused launch
        b = batch_experiences(exps, dev, phi, GAMMA)
        pinned[0].copy_(b["weights"], non_blocking=True)
        pinned[1].copy_(b["reward"], non_blocking=True)
        pinned[2].copy_(exps.index, non_blocking=True)
        torch.cuda.current_stream().synchronize()  # the D2H read of the step's result
        buf.update_errors(err_host[i % 8])         # host float list -> priorities -> H2D
        return b

    for i in range(W * 4):
        pass_e2e(i)
    barrier()
    t2, t3 = ev(), ev()
    t2.record()
    for i in range(K * R_e2e):
        pass_e2e(i)
    t3.record()
    barrier()
    ms_e2e = t2.elapsed_time(t3)

    # ---- Rainbow training loop on the same shard ----------------------------------
    rb = None
    if not args.no_rainbow:
        from pfrl_b200 import parallel
        from pfrl_b200.envs import SyntheticAtariVectorEnv

        torch.backends.cudnn.allow_tf32 = False  # fp32 parity configuration
        torch.backends.cuda.matmul.allow_tf32 = False
        graph = not args.no_rainbow_graph  # N > 1: two graphs around the eager all-reduce
        agent = make_rainbow_agent(buf, local_rank, B,
                                   grad_sync=parallel.GradSync() if world > 1 else None,
                                   cuda_graph=graph)
        vec_steps = max(8, min(4 * K, 80))
        res = {}
        for tag, env_dev in (("value", dev), ("e2e", "cpu")):
            env = SyntheticAtariVectorEnv(RAINBOW_ENVS, device=env_dev, seed=11 + rank)
            rainbow_loop(agent, env, 8)  # warm-up: cuDNN autotune, allocator, graph captures (first 4), then steady state
            barrier()
            a, b = ev(), ev()
            n0 = agent.optim_t
            a.record()
            rainbow_loop(agent, env, vec_steps)
            b.record()
            barrier()
            res[tag] = (a.elapsed_time(b), agent.optim_t - n0)
        rb = (res, vec_steps, graph)

    # ---- secondary workloads: BASELINE configs[1], [3], [4] -------------------------
    secondary = None
    if not args.no_secondary and world == 1:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import bench_secondary

            secondary = bench_secondary.run_all(graph=True)
        except Exception as exc:  # secondary lines never take the headline down
            secondary = {"error": repr(exc)}
        try:
            secondary["k10_tensor_cores"] = k10_record()
        except Exception as exc:
            secondary["k10_tensor_cores"] = {"error": repr(exc)}

    clk = clocks.stop() if rank == 0 else None

    # ---- max over ranks ---------------------------------------------------------
    tm = torch.tensor([ms_value, ms_e2e, ms_par] +
                      ([rb[0]["value"][0], rb[0]["e2e"][0]] if rb else []),
                      device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    tml = [float(x) for x in tm.tolist()]
    ms_value, ms_e2e, ms_par = tml[0], tml[1], tml[2]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    value = world * B * K * R / (ms_value / 1e3)
    e2e = world * B * K * R_e2e / (ms_e2e / 1e3)
    value_par = world * B * K * R / (ms_par / 1e3)
    ms_pass = ms_value / (K * R)
    ms_pass_par = ms_par / (K * R)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak = json.load(open(peaks_path))["hbm_gbs"]
        peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (of fallback)"

    def roof(bytes_per_launch, ms, kernel, traffic=None, **extra):
        ach = bytes_per_launch / (ms * 1e-3) / 1e9
        d = {"bound": "hbm", "kernel": kernel, "achieved": ach, "peak": peak, "unit": "GB/s",
             "frac": ach / peak, "traffic": traffic, "algorithmic_bytes_per_launch": bytes_per_launch,
             "kernel_ms": ms, "peak_source": peak_src}
        d.update(extra)
        return d

    full = B == 512 and args.capacity == 10 ** 6
    sub = {
        "k_sample_exact_deep": {"ms": kern_ms["sample_exact"],
                                "ns_per_draw": 1e6 * kern_ms["sample_exact"] / B,
                                "bound": "latency of the dependent draw chain",
                                "achieved_GBps": ALGO_BYTES_TREE * B / kern_ms["sample_exact"] / 1e6},
        "k_sample_parallel": {"ms": kern_ms["sample_parallel"]},
        "k_weights": {"ms": kern_ms["weights"]},
        "k_gather": roof(ALGO_BYTES_GATHER * B, kern_ms["gather"], "k_gather",
                         traffic=ncu_traffic("gather") if full else None),
        "k_update_paths": {"ms": kern_ms["update"]},
    }
    line = {
        "metric": "replay_samples_per_sec", "value": value, "unit": "samples/s", "n_gpus": world,
        "steps": K, "warmup": W, "ms_per_step": ms_value / K, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64 priorities / u8->f32 frames",
        "data": "synthetic", "config": workload_config(args, world, passes=R),
        "e2e": {"value": e2e, "unit": "samples/s", "ms_per_pass": ms_e2e / (K * R_e2e),
                "passes_per_step": R_e2e,
                "h2d_bytes_per_step": R_e2e * (8 * B + 8 * B),
                "d2h_bytes_per_step": R_e2e * (4 * B + 4 * B + 8 * B)},
        "gpu_launches": K * R,
        "ms_per_pass": ms_pass,
        # the PATH: SURVEY 8(d) bytes per sample x samples per launch / launch time
        "roofline": roof(ALGO_BYTES_PATH * B, ms_pass, "k_replay_step<exact> (whole pass: "
                         "write-back + sample + weights + gather in one launch)",
                         traffic=ncu_traffic("step_exact") if full else None,
                         dominant_phase="exact sampler (dependent chain of %d draws)" % B,
                         traffic_source="profiles/r*_ncu_full_summary.csv (ncu --set full, per launch)",
                         algorithmic_bytes_per_sample=ALGO_BYTES_PATH,
                         phases_of_one_launch=phases_exact, kernels=sub),
        "sampler": {"mode": "exact", "ns_per_draw_fused_pass": 1e6 * ms_pass / B,
                    "ns_per_draw_sampling_phase": 1e3 * phases_exact["sampling_us"] / B,
                    "ns_per_draw_kernel": 1e6 * kern_ms["sample_exact"] / B,
                    "fast_draws": scout & 0xffff, "slow_draws": scout >> 16},
        "throughput_mode": {
            "sampler": "parallel (all descents concurrent on the frozen tree, with replacement; "
                       "not index-identical to the reference)",
            "value": value_par, "unit": "samples/s", "ms_per_pass": ms_pass_par,
            "gpu_launches": K * R,
            "roofline": roof(ALGO_BYTES_PATH * B, ms_pass_par, "k_replay_step<parallel>",
                             traffic=ncu_traffic("step_parallel") if full else None,
                             phases_of_one_launch=phases_par),
            "u8_out": {
                "note": "same pass, uint8 state / next_state out (SURVEY 8(d): 107.6 KB/sample); "
                        "rank 0 only, not part of `value`",
                "ms_per_pass": ms_par_u8 / (K8 * R),
                "samples_per_sec_per_gpu": B * K8 * R / (ms_par_u8 / 1e3),
                "roofline": roof(ALGO_BYTES_PATH_U8 * B, ms_par_u8 / (K8 * R),
                                 "k_replay_step<parallel, u8 out>",
                                 phases_of_one_launch=phases_par_u8)}},
        "separate_launches_ms": kern_ms,
        "clocks": clk, "prefill_s": fill_s,
        "hbm_bytes_per_rank": store.device_bytes,
    }
    if rb is not None:
        res, vec_steps, graph = rb
        steps_total = world * RAINBOW_ENVS * vec_steps
        line["rainbow"] = {
            "env_steps_per_sec": steps_total / (tml[3] / 1e3),
            "e2e_env_steps_per_sec": steps_total / (tml[4] / 1e3),
            "num_envs_per_rank": RAINBOW_ENVS, "vector_steps": vec_steps,
            "updates": res["value"][1], "update_interval": RAINBOW_UPDATE_INTERVAL,
            "ms_per_update_incl_acting": tml[3] / max(res["value"][1], 1),
            "minibatch_per_rank": B, "dtype": "fp32 (TF32 off)", "cuda_graph": graph,
            "observations": "uint8 minibatches out of the replay gather; x / 255 applied inside "
                            "conv1 (b2rl_conv_nature1_fwd_u8), same numbers as f32 batches",
            "model": "DistributionalDuelingDQN(18, 51) + factorized noisy, Adam(6.25e-5)",
            "dense_layers": "tcgen05 3xTF32 (k_gemm_tf32x3) for main_stream fwd/dX/dW, conv2 forward, "
                            "conv3 input gradient; cuDNN / cuBLAS fp32 where they measured faster; "
                            "conv1 forward own FFMA kernel",
            "note": "value: GPU-resident synthetic env; e2e: host numpy env (frames H2D, "
                    "actions D2H); gradient all-reduce (NCCL) when n_gpus > 1"}
    if secondary is not None:
        line["secondary"] = secondary
    if not args.no_cpu_baseline and world == 1:  # reported baseline: rank 0 at N = 1 only
        r, rc = cpu_arm(cap, B, 10 ** 9, 2, args.cpu_seconds, 10.0 if rb is not None else None)
        if rc is not None:
            line["rainbow"]["cpu_baseline"] = {
                "value": rc["env_steps_per_sec"], "unit": "env-steps/s", "kind": rc["kind"],
                "cores": rc["threads"], "ms_per_update": rc["ms_per_update"],
                "sample": "%.0f s of the same loop on the host" % rc["seconds"]}
        line["cpu_baseline"] = {
            "value": r["samples_per_sec"], "unit": "samples/s", "cores": r["cores"],
            "kind": r["kind"], "host_cores_available": os.cpu_count(),
            "sample": cpu_sample_text(r, B)}
    if dumped is not None:
        for name, arr in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def ncu_traffic(kernel):
    """dram__bytes_read + dram__bytes_write of `kernel` per launch, from the
    newest committed ncu --set full summary under profiles/ (bytes)."""
    import csv
    import glob

    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_full_summary.csv")))
    mult = {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    for f in reversed(files):
        total = 0.0
        for row in csv.reader(open(f)):
            if len(row) == 4 and row[0] == kernel and row[1] in ("dram__bytes_read.sum",
                                                               "dram__bytes_write.sum"):
                total += float(row[2]) * mult.get(row[3], 1)
        if total:
            return total
    return None


def workload_config(args, world, passes):
    return {"workload": "Rainbow replay path (BASELINE configs[2]): PER 1M cap, 3-step, "
                        "84x84x4 u8 frames, minibatch %d per rank" % args.batch,
            "capacity_per_rank": args.capacity, "batch_per_rank": args.batch,
            "global_batch": args.batch * world, "n_step": N_STEP, "alpha": ALPHA,
            "passes_per_step": passes,
            "pass": "priority write-back of the previous minibatch + sample + IS weights + gather",
            "sampler": "exact", "obs_out": "f32 (x/255)", "l2": "inputs_larger_than_l2",
            "parallelism": "replay shard per rank, no data-path collective"}


if __name__ == "__main__":
    main()
