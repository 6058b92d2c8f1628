#!/bin/sh
# vectorised SAC on Pendulum with command-line hyper-parameters: experiments/run_sac.sh --num_envs 4096 --buffer_size 1048576
cd "$(dirname "$0")/.." || exit 1
exec python -m cleanrl_jl_b200 sac "$@"
