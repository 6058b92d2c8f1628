"""Time crl_c51_run on one GPU, next to crl_dqn_run, and print one JSON line.

Workload: bench.py's DQN shape — 4,096 CartPole envs, a 1,048,576-transition ring, a learning step every 10 iterations
after 10,000 global steps — with C51's own batch of 128 and target copy every 500 iterations; DQN runs the same shape at
bench.py's DQN settings (batch 120, target every 100). Then the same with num_envs 1 (CleanRL's ratio of one env step per
iteration). Reported:
  * env-steps/s and learner steps/s over whole run calls (device synchronised around the timed window, after a warm-up
    past learning_starts);
  * us per acting launch and per learning step (the three learning kernels), from torch.profiler's CUDA activity in a
    separate profiled run;
  * C51's learning step written in PyTorch eager (CleanRL's c51.py) at B = 128 on the same GPU;
  * the card's name, power limit and max SM clock, read in the same call.
Usage: python tools/c51_bench.py [--iters 3000] [--out path.json] [--trace-dir dir]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def make(num_envs, algo):
    from cleanrl_jl_b200 import _abi
    kw = dict(num_envs=num_envs, buffer_size=1 << 20, seed=1, max_episode_steps=500)
    if algo == "c51":
        from cleanrl_jl_b200.c51_algo import C51Handle, init_c51_params
        h = C51Handle(_abi.make_c51_config(learning_starts=10_000, batch_size=128, train_frequency=10,
                                           target_network_frequency=500, epsilon_duration=250_000.0, **kw))
        h.set_params(init_c51_params(1))
    else:
        from cleanrl_jl_b200.dqn_algo import DQNHandle, init_q_params
        h = DQNHandle(_abi.make_dqn_config(min_buff_size=10_000, batch_size=120, train_freq=10, target_net_freq=100,
                                           epsilon_duration=250_000.0, **kw))
        h.set_params(init_q_params(1))
    h.reset()
    return h


def timed(torch, num_envs, iters, algo):
    h = make(num_envs, algo)
    h.run(10_000 // num_envs + 20)            # warm-up: past learning_starts, every kernel launched
    torch.cuda.synchronize()
    st0 = h.run(0)
    t0 = time.perf_counter()
    st = h.run(iters)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    h.close()
    return {"num_envs": num_envs, "iterations": iters, "seconds": dt, "env_steps_per_s": iters * num_envs / dt,
            "learner_steps_per_s": (st.learn_steps - st0.learn_steps) / dt}


def profiled(torch, iters, out_dir, algo):
    """per-kernel device time from torch.profiler (CUDA activities) in a run of its own"""
    from torch.profiler import ProfilerActivity, profile
    h = make(4096, algo)
    h.run(10_000 // 4096 + 20)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        st0 = h.run(0)
        st = h.run(iters)
        torch.cuda.synchronize()
    learn = st.learn_steps - st0.learn_steps
    acting = st.kernel_launches - st0.kernel_launches - (3 if algo == "c51" else 2) * learn
    h.close()
    per = {}
    for e in prof.key_averages():
        if algo + "_" in e.key:
            k = e.key.replace("void ", "").replace("(anonymous namespace)::", "").split("(")[0]
            per[k] = per.get(k, 0.0) + e.device_time_total
    act = sum(v for k, v in per.items() if "act_kernel" in k)
    lrn = sum(v for k, v in per.items() if "act_kernel" not in k)
    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
        prof.export_chrome_trace(os.path.join(out_dir, "%s_trace.json" % algo))
    return {"us_per_acting_launch": act / max(acting, 1), "us_per_learning_step": lrn / max(learn, 1),
            "kernel_us_per_learning_step": {k: round(v / max(learn, 1), 2) for k, v in per.items() if "act_kernel" not in k}}


def eager(torch, reps=200):
    """c51.py's learning step in PyTorch eager at B = 128 (sampling from a 2^20 ring, target pmfs with the index_add_
    loop, the clamp-log loss, Adam with eps 0.01 / B)"""
    import copy
    nn = torch.nn
    dev, B, C, n_atoms = "cuda", 128, 1 << 20, 101
    net = nn.Sequential(nn.Linear(4, 120), nn.ReLU(), nn.Linear(120, 84), nn.ReLU(), nn.Linear(84, 2 * n_atoms)).to(dev)
    tgt = copy.deepcopy(net)
    opt = torch.optim.Adam(net.parameters(), lr=2.5e-4, eps=0.01 / B)
    atoms = torch.linspace(-100, 100, n_atoms, device=dev)
    obs, nobs = torch.randn(C, 4, device=dev), torch.randn(C, 4, device=dev)
    act, rew, term = torch.randint(0, 2, (C,), device=dev), torch.ones(C, 1, device=dev), torch.zeros(C, 1, device=dev)

    def get_action(n, x, action=None):
        pmfs = torch.softmax(n(x).view(len(x), 2, n_atoms), dim=2)
        q_values = (pmfs * atoms).sum(2)
        if action is None:
            action = torch.argmax(q_values, 1)
        return action, pmfs[torch.arange(len(x)), action]

    def step():
        idx = torch.randint(0, C, (B,), device=dev)
        with torch.no_grad():
            _, next_pmfs = get_action(tgt, nobs[idx])
            next_atoms = rew[idx] + 0.99 * atoms * (1 - term[idx])
            delta_z = atoms[1] - atoms[0]
            tz = next_atoms.clamp(-100, 100)
            b = (tz + 100) / delta_z
            l = b.floor().clamp(0, n_atoms - 1)
            u = b.ceil().clamp(0, n_atoms - 1)
            d_m_l = (u + (l == u).float() - b) * next_pmfs
            d_m_u = (b - l) * next_pmfs
            target_pmfs = torch.zeros_like(next_pmfs)
            for i in range(target_pmfs.size(0)):
                target_pmfs[i].index_add_(0, l[i].long(), d_m_l[i])
                target_pmfs[i].index_add_(0, u[i].long(), d_m_u[i])
        _, old_pmfs = get_action(net, obs[idx], act[idx])
        loss = (-(target_pmfs * old_pmfs.clamp(min=1e-5, max=1 - 1e-5).log()).sum(-1)).mean()
        opt.zero_grad(); loss.backward(); opt.step()

    for _ in range(10):
        step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        step()
    torch.cuda.synchronize()
    return {"eager_us_per_learning_step": (time.perf_counter() - t0) / reps * 1e6}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=3000)
    ap.add_argument("--out", default=None)
    ap.add_argument("--trace-dir", default=None, help="write the profiled runs' Chrome traces here")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("c51_bench needs a GPU")
    res = {**card()}
    for algo in ("c51", "dqn"):
        res[algo] = {"n4096": timed(torch, 4096, args.iters, algo), "n1": timed(torch, 1, args.iters * 5, algo),
                     "profile_n4096": profiled(torch, 500, args.trace_dir, algo)}
    res["c51"].update(eager(torch))
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
