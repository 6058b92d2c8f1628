#!/bin/sh
# vectorised C51 on CartPole with command-line hyper-parameters: experiments/run_c51.sh --num_envs 64 --buffer_size 100000
cd "$(dirname "$0")/.." || exit 1
exec python -m cleanrl_jl_b200 c51 "$@"
