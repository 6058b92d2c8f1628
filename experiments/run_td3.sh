#!/bin/sh
# vectorised TD3 on Pendulum with command-line hyper-parameters: experiments/run_td3.sh --num_envs 4096 --buffer_size 1048576
cd "$(dirname "$0")/.." || exit 1
exec python -m cleanrl_jl_b200 td3 "$@"
