"""Runner: `python -m cleanrl_jl_b200 {ppo,a2c,dqn,ddpg,td3,sac,c51} [--field value ...]`.

The reference leaves this wiring as a TODO ("Make individual file runners e.g experiments/run_ppo.(jl/sh)", README.md:24):
`ConfigParser.argparse_struct` exists (config_parser.jl:18-40) but nothing calls it. Here every field of the algorithm's
config struct is a command-line option, typed and defaulted from the struct (argparse_struct), and the parsed struct goes
to the algorithm entry point:   argparse_struct(PPOConfig()) |> ppo.

Multi-GPU: launch under torchrun (`python -m torch.distributed.run --nproc-per-node N -m cleanrl_jl_b200 ppo ...`); the
env vector is sharded over the ranks (SURVEY 8e) and rank 0 logs."""
import json
import os
import sys


def _configs():
    from .a2c_algo import A2CConfig
    from .config import PPOConfig
    from .dqn_algo import DQNConfig
    return {"ppo": PPOConfig, "a2c": A2CConfig, "dqn": DQNConfig}


def _single_gpu_configs():
    """algorithms with no multi-GPU path (DDPG on Pendulum: one GPU, include/cleanrl_ddpg.h)"""
    from .ddpg_algo import DDPGConfig
    return {"ddpg": DDPGConfig}


def _extension_configs():
    """one-GPU algorithms the reference does not have (TD3 on Pendulum: include/cleanrl_td3.h)"""
    from .td3_algo import TD3Config
    return {"td3": TD3Config}


def _sac_configs():
    """SAC on Pendulum (include/cleanrl_sac.h): one GPU, not in the reference, on a usage line of its own"""
    from .sac_algo import SACConfig
    return {"sac": SACConfig}


def _c51_configs():
    """C51 on CartPole (include/cleanrl_c51.h): one GPU, not in the reference, on a usage line of its own"""
    from .c51_algo import C51Config
    return {"c51": C51Config}


def main(argv=None):
    argv = list(sys.argv[1:] if argv is None else argv)
    algos = _configs()
    single = _single_gpu_configs()
    ext = _extension_configs()
    sac_ = _sac_configs()
    c51_ = _c51_configs()
    if not argv or argv[0] in ("-h", "--help") or argv[0] not in {**algos, **single, **ext, **sac_, **c51_}:
        sys.stderr.write("usage: python -m cleanrl_jl_b200 {%s} [--<config field> <value> ...]\n"
                         "       python -m cleanrl_jl_b200 {%s} [--<config field> <value> ...]   (one GPU)\n"
                         "       python -m cleanrl_jl_b200 {%s} [--<config field> <value> ...]   (one GPU, not in the reference)\n"
                         "       python -m cleanrl_jl_b200 {%s} [--<config field> <value> ...]   (one GPU, not in the reference)\n"
                         "       python -m cleanrl_jl_b200 {%s} [--<config field> <value> ...]   (one GPU, not in the reference)\n"
                         "       (every field of the algorithm's config struct is an option; --help after the algorithm lists them)\n"
                         % (",".join(sorted(algos)), ",".join(sorted(single)), ",".join(sorted(ext)), ",".join(sorted(sac_)),
                            ",".join(sorted(c51_))))
        return 2
    algos = {**algos, **single, **ext, **sac_, **c51_}
    from .config import argparse_struct
    algo = argv[0]
    config = argparse_struct(algos[algo](), argv[1:])
    world = int(os.environ.get("WORLD_SIZE", 1))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        local_rank = int(os.environ.get("LOCAL_RANK", 0))
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        from . import a2c, c51, ddpg, dqn, ppo, sac, td3
        res = {"ppo": ppo, "a2c": a2c, "dqn": dqn, "ddpg": ddpg, "td3": td3, "sac": sac, "c51": c51}[algo](config)
    finally:
        if dist is not None:
            dist.destroy_process_group()
    if int(os.environ.get("RANK", 0)) == 0:
        keep = {k: v for k, v in res.items() if isinstance(v, (int, float, str)) or v is None}
        print(json.dumps({"algorithm": algo, **keep}))
    return 0


if __name__ == "__main__":
    sys.exit(main())
