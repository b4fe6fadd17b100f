"""Command-line front-end of the sweep (reference: ``main.py:90-245``), re-hosted on the GPU path.

    python -m highway_rope_ppo_b200.main --get-total-experiments
    python -m highway_rope_ppo_b200.main --run-single-experiment <name or unique prefix>
    python -m highway_rope_ppo_b200.main --array-task-id 3 --slurm-num-tasks 68 [--n-jobs 16] [--gym-id highway-fast-v0]
    torchrun --nproc-per-node 8 -m highway_rope_ppo_b200.main --n-jobs 32        # the whole grid, 8 GPUs x 32 runs at a time

The experiment grid, names, selection rules and the end-of-run summary are the reference's
(``experiments/sweep.py``).  What differs is how the selected experiments are executed: the reference fans them out
over ``--n-jobs`` joblib workers that time-share the GPUs through ``DevicePool``; here every process owns one GPU
(``LOCAL_RANK``), takes the experiments ``rank, rank + world, ...`` of the selection, and runs ``--n-jobs`` of them AT
A TIME on shared env handles (``experiments/multiplex.py``; 1 = one after the other).  SLURM script generation
(``--generate-slurm``) is the reference's control plane and is not rebuilt.
"""
from __future__ import annotations

import argparse
import logging
import os
import sys
from typing import List, Optional


def parse(argv: Optional[List[str]] = None) -> argparse.Namespace:
    p = argparse.ArgumentParser(description="Run Highway PPO Experiments (B200 path)")
    p.add_argument("--generate-slurm", action="store_true", help="(reference control plane: not rebuilt here)")
    p.add_argument("--run-single-experiment", type=str, default=None, help="Experiment name (or unique prefix) to run.")
    p.add_argument("--n-jobs", type=int, default=-1,
                   help="Experiments multiplexed at a time on this process's GPU (-1: 16; 1: sequential)")
    p.add_argument("--num-seeds", type=int, default=3, help="Num seeds per condition")
    p.add_argument("--slurm-num-tasks", type=int, default=None, help="Number of array tasks (batches)")
    p.add_argument("--array-task-id", type=int, default=None, help="ID of the current array task (batch)")
    p.add_argument("--get-total-experiments", action="store_true", help="Print total number of experiments and exit")
    p.add_argument("--artifacts-dir", type=str, default=None)
    p.add_argument("--max-episodes", type=int, default=None, help="override Experiment.max_episodes (smoke runs)")
    p.add_argument("--gym-id", type=str, default=None, choices=("highway-v0", "highway-fast-v0"),
                   help="env id of every experiment (the config key gym_id; default: the base config's, highway-v0)")
    return p.parse_args(argv)


def main(argv: Optional[List[str]] = None) -> int:
    args = parse(argv)
    from .experiments.sweep import define_experiments, run_experiments, select_experiments, shard_for_rank, summarize
    from .utils.reproducibility import SEED

    experiments = define_experiments(SEED, args.num_seeds)
    if args.get_total_experiments:
        print(len(experiments))
        return 0
    if args.generate_slurm:
        print("--generate-slurm: SLURM script generation is the reference's control plane and is not part of this "
              "package; use the reference's own generator with python_script pointing at this module", file=sys.stderr)
        return 2
    log = logging.getLogger("master")
    try:
        selected = select_experiments(experiments, args.array_task_id, args.slurm_num_tasks, args.run_single_experiment)
    except ValueError as err:
        log.error(str(err))
        return 1
    if args.max_episodes is not None:
        for e in selected:
            e.max_episodes = args.max_episodes
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    mine = shard_for_rank(selected, rank, world)
    jobs = 16 if args.n_jobs < 0 else max(1, args.n_jobs)
    log.info(f"rank {rank}/{world}: launching {len(mine)} of {len(selected)} experiments, {jobs} at a time")
    from .config.base_config import HIGHWAY_CONFIG

    base = HIGHWAY_CONFIG if args.gym_id is None else dict(HIGHWAY_CONFIG, gym_id=args.gym_id)
    results = run_experiments(mine, base, artifacts_dir=args.artifacts_dir, multiplex=jobs)
    succ = sum(1 for r in results if r.get("status") == "COMPLETED")
    log.info(f"Summary: {succ} succeeded, {len(results) - succ} failed.")
    for cond, (score, name) in summarize(results).items():
        print(f"{cond:20s} best avg_reward={score:.2f}  ({name})")
    return 0 if succ == len(results) else 3


if __name__ == "__main__":
    sys.exit(main())
