"""Time crl_ddpg_run (or, with --algo td3 / sac, crl_td3_run / crl_sac_run) on one GPU and print one JSON line.

Workload: 4,096 Pendulum envs, a 1,048,576-transition ring, batch 256, a learning step every iteration,
policy_frequency 2, learning_starts 10,000; and the same with num_envs 1 (one learning step per env step, CleanRL's
update-to-data ratio). Reported:
  * env-steps/s and learner steps/s over a timed window of whole crl_ddpg_run calls (device synchronised around it,
    after a warm-up that fills past learning_starts);
  * us per acting launch and per learning step (critic pair; actor pair + Polyak on every second step), from CUDA events
    of torch.profiler in a separate profiled run;
  * the same learning step written in PyTorch eager on the same GPU at B = 256, for comparison;
  * the card's name, power limit and max SM clock, read in the same call.
TD3 runs the same workload with CleanRL's smoothing noise (0.2, clip 0.5); its learning step is the twin-critic pair
every step and the actor pair + two Polyak launches on every second step. The kernel filter counts the reused ddpg_*
kernels as well as the td3_* ones.
SAC runs the same workload with CleanRL's SAC settings (policy_lr 3e-4, q_lr 1e-3, autotune): its learning step is the
twin-critic pair every step, and on every second step two actor iterations (actor pair + temperature pair each), with
one Polyak launch for both critics every step. The kernel filter counts ddpg_*, td3_* and sac_* kernels.
Usage: python tools/ddpg_bench.py [--algo {ddpg,td3,sac}] [--iters 2000] [--out path.json]"""
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


def make(num_envs, algo="ddpg"):
    from cleanrl_jl_b200 import _abi
    kw = dict(num_envs=num_envs, buffer_size=1 << 20, learning_starts=10_000, batch_size=256, train_freq=1, policy_frequency=2, seed=1)
    if algo == "sac":
        from cleanrl_jl_b200.sac_algo import SACHandle, init_sac_params
        kw.update(policy_lr=3e-4, q_lr=1e-3, target_network_frequency=1, autotune=1)
        h = SACHandle(_abi.make_sac_config(**kw))
        h.set_params(*init_sac_params(1))
    elif algo == "td3":
        from cleanrl_jl_b200.td3_algo import TD3Handle, init_td3_params
        h = TD3Handle(_abi.make_td3_config(**kw))
        h.set_params(*init_td3_params(1))
    else:
        from cleanrl_jl_b200.ddpg_algo import DDPGHandle, init_ddpg_params
        h = DDPGHandle(_abi.make_ddpg_config(**kw))
        h.set_params(*init_ddpg_params(1))
    h.reset()
    return h


def timed(torch, num_envs, iters, algo="ddpg"):
    h = make(num_envs, algo)
    h.run(10_000 // num_envs + 64)            # warm-up: past learning_starts, every kernel launched
    torch.cuda.synchronize()
    st0 = h.run(0)
    t0 = time.perf_counter()
    st = h.run(iters)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    h.close()
    return {"num_envs": num_envs, "iterations": iters, "seconds": dt, "env_steps_per_s": iters * num_envs / dt,
            "learner_steps_per_s": (st.learn_steps - st0.learn_steps) / dt}


def profiled(torch, iters, out_dir, algo="ddpg"):
    """per-kernel device time from torch.profiler (CUDA activities) in a run of its own"""
    from torch.profiler import ProfilerActivity, profile
    h = make(4096, algo)
    h.run(10_000 // 4096 + 8)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        st0 = h.run(0)
        st = h.run(iters)
        torch.cuda.synchronize()
    learn = st.learn_steps - st0.learn_steps
    h.close()
    per = {}
    for e in prof.key_averages():
        if any(k in e.key for k in ("ddpg", "td3", "sac")):
            k = e.key.replace("void ", "").replace("(anonymous namespace)::", "").split("(")[0]
            per[k] = per.get(k, 0.0) + e.device_time_total
    act = sum(v for k, v in per.items() if "act_kernel" in k)
    lrn = sum(v for k, v in per.items() if "act_kernel" not in k)
    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
        prof.export_chrome_trace(os.path.join(out_dir, "%s_trace.json" % algo))
    return {"us_per_acting_launch": act / iters, "us_per_learning_step": lrn / max(learn, 1),
            "kernel_us_total": {k: round(v, 1) for k, v in per.items()}}


def eager_sac_step(torch, dev):
    """CleanRL's sac_continuous_action.py learning step in PyTorch eager (two actor and temperature iterations on every
    second step); returns step(i)"""
    import copy
    nn = torch.nn
    mlp = lambda i, o: nn.Sequential(nn.Linear(i, 64), nn.ReLU(), nn.Linear(64, 64), nn.ReLU(), nn.Linear(64, o)).to(dev)
    actor, qf1, qf2 = mlp(3, 2), mlp(4, 1), mlp(4, 1)
    qt1, qt2 = copy.deepcopy(qf1), copy.deepcopy(qf2)
    log_alpha = torch.zeros(1, requires_grad=True, device=dev)
    oq = torch.optim.Adam(list(qf1.parameters()) + list(qf2.parameters()), lr=1e-3)
    oa, oal = torch.optim.Adam(actor.parameters(), lr=3e-4), torch.optim.Adam([log_alpha], lr=1e-3)
    C, B = 1 << 20, 256
    obs, nobs = torch.randn(C, 3, device=dev), torch.randn(C, 3, device=dev)
    act, rew, term = torch.rand(C, 1, device=dev) * 4 - 2, torch.randn(C, 1, device=dev), torch.zeros(C, 1, device=dev)

    def get_action(x):
        mean, log_std = actor(x).chunk(2, dim=1)
        log_std = -5 + 3.5 * (torch.tanh(log_std) + 1)
        std = log_std.exp()
        x_t = mean + std * torch.randn_like(mean)
        y_t = torch.tanh(x_t)
        lp = torch.distributions.Normal(mean, std).log_prob(x_t) - torch.log(2 * (1 - y_t.pow(2)) + 1e-6)
        return 2 * y_t, lp

    def step(i):
        idx = torch.randperm(C, device=dev)[:B]
        o, a, r, n, d = obs[idx], act[idx], rew[idx], nobs[idx], term[idx]
        alpha = log_alpha.exp().item()
        with torch.no_grad():
            na, nlp = get_action(n)
            xn = torch.cat([n, na], 1)
            y = r + 0.99 * (1 - d) * (torch.min(qt1(xn), qt2(xn)) - alpha * nlp)
        x = torch.cat([o, a], 1)
        loss = ((qf1(x) - y) ** 2).mean() + ((qf2(x) - y) ** 2).mean()
        oq.zero_grad(); loss.backward(); oq.step()
        if i % 2 == 1:
            for _ in range(2):
                pi, lp = get_action(o)
                xp = torch.cat([o, pi], 1)
                al = (alpha * lp - torch.min(qf1(xp), qf2(xp))).mean()
                oa.zero_grad(); al.backward(); oa.step()
                with torch.no_grad():
                    _, lp = get_action(o)
                tl = (-log_alpha.exp() * (lp - 1.0)).mean()
                oal.zero_grad(); tl.backward(); oal.step()
                alpha = log_alpha.exp().item()
        with torch.no_grad():
            for net, tgt in ((qf1, qt1), (qf2, qt2)):
                for p, tp in zip(net.parameters(), tgt.parameters()):
                    tp.mul_(0.995).add_(0.005 * p)
    return step


def eager(torch, reps=200, algo="ddpg"):
    """the same learning step (critic step every time, actor step + Polyak every second) in PyTorch eager, B = 256; TD3:
    two critics with one Adam over both, the smoothed target action and the minimum of the two target critics"""
    import copy
    nn = torch.nn
    dev = "cuda"
    mlp = lambda i: nn.Sequential(nn.Linear(i, 64), nn.ReLU(), nn.Linear(64, 64), nn.ReLU(), nn.Linear(64, 1)).to(dev)
    actor, critic = mlp(3), mlp(4)
    at, ct = copy.deepcopy(actor), copy.deepcopy(critic)
    critic_params = list(critic.parameters())
    if algo == "td3":
        critic2 = mlp(4)
        ct2 = copy.deepcopy(critic2)
        critic_params += list(critic2.parameters())
    oa, oc = torch.optim.Adam(actor.parameters(), lr=3e-4), torch.optim.Adam(critic_params, lr=3e-4)
    C, B = 1 << 20, 256
    obs, nobs = torch.randn(C, 3, device=dev), torch.randn(C, 3, device=dev)
    act, rew, term = torch.rand(C, 1, device=dev) * 4 - 2, torch.randn(C, 1, device=dev), torch.zeros(C, 1, device=dev)

    def step(i):
        idx = torch.randperm(C, device=dev)[:B]
        o, a, r, n, d = obs[idx], act[idx], rew[idx], nobs[idx], term[idx]
        with torch.no_grad():
            if algo == "td3":
                na = (2 * torch.tanh(at(n)) + (torch.randn_like(a) * 0.2).clamp(-0.5, 0.5) * 2).clamp(-2, 2)
                y = r + 0.99 * (1 - d) * torch.min(ct(torch.cat([n, na], 1)), ct2(torch.cat([n, na], 1)))
            else:
                y = r + 0.99 * (1 - d) * ct(torch.cat([n, 2 * torch.tanh(at(n))], 1))
        loss = ((critic(torch.cat([o, a], 1)) - y) ** 2).mean()
        if algo == "td3":
            loss = loss + ((critic2(torch.cat([o, a], 1)) - y) ** 2).mean()
        oc.zero_grad(); loss.backward(); oc.step()
        if i % 2 == 1:
            al = -critic(torch.cat([o, 2 * torch.tanh(actor(o))], 1)).mean()
            oa.zero_grad(); al.backward(); oa.step()
            with torch.no_grad():
                for net, tgt in ((actor, at), (critic, ct)) + (((critic2, ct2),) if algo == "td3" else ()):
                    for p, tp in zip(net.parameters(), tgt.parameters()):
                        tp.mul_(0.995).add_(0.005 * p)

    if algo == "sac":
        step = eager_sac_step(torch, dev)
    for i in range(20):
        step(i)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(reps):
        step(i)
    torch.cuda.synchronize()
    return {"eager_us_per_learning_step": (time.perf_counter() - t0) / reps * 1e6}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--algo", choices=("ddpg", "td3", "sac"), default="ddpg")
    ap.add_argument("--iters", type=int, default=2000)
    ap.add_argument("--out", default=None)
    ap.add_argument("--trace-dir", default=None, help="write the profiled run's Chrome trace here")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("ddpg_bench needs a GPU")
    res = {**card()}
    if args.algo != "ddpg":
        res["algo"] = args.algo
    res["n4096"] = timed(torch, 4096, args.iters, args.algo)
    res["n1"] = timed(torch, 1, args.iters * 5, args.algo)
    res["profile_n4096"] = profiled(torch, 200, args.trace_dir, args.algo)
    res.update(eager(torch, algo=args.algo))
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
