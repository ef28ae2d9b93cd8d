"""`three-mlagents` command line — same sub-commands, flags and JSON outputs as
backend/mlagents/cli.py:13-95 (`list [--trainable-only]`, `inspect <task>`,
`train <task> [-a ALGO] [-t N] [--seed] [--n-envs] [--eval-episodes] [--eval-freq] [--run-name] [--quiet]`,
`evaluate <task> <model> [--episodes] [--seed] [--stochastic]`), running on the CUDA backend.

    python -m three_mlagents_b200.cli train basic -a ppo -t 25000 --seed 1
"""
from __future__ import annotations

import argparse
import json
from dataclasses import asdict

from .registry import list_task_cards, make_env


def build_parser() -> argparse.ArgumentParser:
    parser = argparse.ArgumentParser(prog="three-mlagents")
    sub = parser.add_subparsers(dest="command", required=True)
    p = sub.add_parser("list", help="List registered tasks")
    p.add_argument("--trainable-only", action="store_true")
    p = sub.add_parser("inspect", help="Print one environment's spaces")
    p.add_argument("task")
    p = sub.add_parser("train", help="Train one task (PPO or A2C on the CUDA backend)")
    p.add_argument("task")
    p.add_argument("--algorithm", "-a")
    p.add_argument("--timesteps", "-t", type=int)
    p.add_argument("--seed", type=int, default=1)
    p.add_argument("--n-envs", type=int)
    p.add_argument("--eval-episodes", type=int)
    p.add_argument("--eval-freq", type=int, default=10_000)
    p.add_argument("--run-name")
    p.add_argument("--quiet", action="store_true")
    p = sub.add_parser("evaluate", help="Evaluate a saved policy zip")
    p.add_argument("task")
    p.add_argument("model")
    p.add_argument("--episodes", type=int)
    p.add_argument("--seed", type=int, default=10_001)
    p.add_argument("--stochastic", action="store_true")
    return parser


def main(argv: list[str] | None = None) -> None:
    args = build_parser().parse_args(argv)
    if args.command == "list":
        print(json.dumps(list_task_cards(include_roadmap=not args.trainable_only), indent=2))
    elif args.command == "inspect":
        env = make_env(args.task)
        try:
            print(json.dumps({"task": args.task, "observation_space": repr(env.observation_space),
                              "action_space": repr(env.action_space)}, indent=2))
        finally:
            env.close()
    elif args.command == "train":
        from .training import TrainConfig, train_task

        result = train_task(TrainConfig(task_id=args.task, total_timesteps=args.timesteps, algorithm=args.algorithm,
                                        seed=args.seed, n_envs=args.n_envs, eval_episodes=args.eval_episodes,
                                        eval_freq=args.eval_freq, run_name=args.run_name, verbose=0 if args.quiet else 1))
        print(json.dumps(asdict(result), indent=2))
    elif args.command == "evaluate":
        from .training import evaluate_model

        print(json.dumps(evaluate_model(args.task, args.model, episodes=args.episodes, deterministic=not args.stochastic,
                                        seed=args.seed), indent=2))


if __name__ == "__main__":
    main()
