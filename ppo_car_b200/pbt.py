"""Population-based training (Jaderberg et al. 2017, "Population Based Training of Neural Networks") of a population.

Every ``--pbt-every K`` epochs ``train_population`` scores every member (``evaluate_population``, one launch), ranks
them, and the bottom fraction each take the full training state of a member of the top fraction (*exploit*:
weights, Adam moments and step count, the current learning rate and every other per-member hyperparameter) and then
scale some of the copied hyperparameters by 0.8 or 1.2 (*explore*).  A slot keeps its seed, Philox stream,
environments, minibatch generator and checkpoint directory.

The decisions depend only on the fitness of all members and one CPU generator seeded ``--pbt-seed``; a member's bits
depend neither on P nor on how the members are split over ranks, so a PBT run gives the same bits at any world size.

    python -m ppo_car_b200.population --track big_track --n-envs 24 --seeds 0-7 \\
        --learning-rate 1e-4,3e-4,1e-3,3e-3 --pbt-every 10 --pbt-explore learning_rate,ent_coef
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from .population import HPARAMS

FACTORS = (0.8, 1.2)


def parse_explore(spec: str) -> list[str]:
    """``--pbt-explore``: comma-separated names of :data:`HPARAMS` (empty: exploit only), returned in HPARAMS order."""
    names = {s.strip() for s in str(spec).split(",") if s.strip()}
    unknown = names - set(HPARAMS)
    if unknown:
        raise ValueError(f"--pbt-explore: unknown hyperparameters {sorted(unknown)}; choose from {', '.join(HPARAMS)}")
    return [k for k in HPARAMS if k in names]


def pbt_decisions(fitness, fraction: float, explore, generator: torch.Generator) -> list[tuple[int, int, dict]]:
    """One round's ``[(dst, src, {name: factor})]``, ascending in ``dst``.

    Members are ranked by fitness, descending, ties to the lower index; with ``m = floor(P * fraction)`` each of the
    bottom m members copies a member drawn uniformly from the top m (best first), and each name of ``explore`` gets a
    factor of 0.8 or 1.2.  The draws come from ``generator`` in a fixed order — destinations ascending, for each its
    source, then its factors in HPARAMS order — so every rank holding the same fitness makes the same decisions."""
    fitness = [float(f) for f in fitness]
    P = len(fitness)
    if not 0.0 < fraction <= 0.5:
        raise ValueError("fraction must be in (0, 0.5]")
    names = [k for k in HPARAMS if k in set(explore)]
    order = sorted(range(P), key=lambda i: (-fitness[i], i))
    m = int(P * fraction)
    top, bottom = order[:m], sorted(order[P - m:])
    draw = lambda n: int(torch.randint(0, n, (1,), generator=generator))
    out = []
    for dst in bottom:
        src = top[draw(m)]
        out.append((dst, src, {k: FACTORS[draw(2)] for k in names}))
    return out


def _gather_padded(local: torch.Tensor, counts: list[int]) -> torch.Tensor:
    """Rows of every rank in member order: each rank pads its ``[counts[rank], ...]`` rows to ``max(counts)`` for one
    ``all_gather_into_tensor``."""
    mx = max(counts)
    buf = local.new_zeros((mx, *local.shape[1:]))
    buf[:local.shape[0]] = local
    out = local.new_empty((len(counts) * mx, *local.shape[1:]))
    dist.all_gather_into_tensor(out, buf)
    return torch.cat([out[r * mx:r * mx + c] for r, c in enumerate(counts)])


def gather_fitness(local: list[float], counts: list[int], device) -> list[float]:
    """Every member's fitness (float64, exact) on every rank, from each rank's own members."""
    return _gather_padded(torch.tensor(local, dtype=torch.float64, device=device), counts).tolist()


def gather_states(pop, counts: list[int]) -> tuple[torch.Tensor, torch.Tensor]:
    """Every member's packed training state on every rank: ``(float32 [P, S], int32 [P])`` in member order, from one
    all-gather of each rank's ``Population.state_rows`` (plus one of the step counts)."""
    rows, steps = pop.state_rows(range(pop.P))
    return _gather_padded(rows, counts), _gather_padded(steps, counts)


def pbt_round(pop, env, args, r: int, epoch: int, lo: int, counts: list[int], generator: torch.Generator,
              explore: list[str]) -> tuple[list[float], list[dict]]:
    """Round ``r`` after epoch ``epoch`` for the members ``lo .. lo + pop.P - 1`` of this rank (``counts``: members
    per rank).  Fitness is each member's mean return over episodes ``r * eval_episodes ..`` of one
    ``evaluate_population`` call, every member with the seed ``--pbt-seed``.  Returns every member's fitness and one
    lineage record per replaced member of this rank."""
    from .evaluate import evaluate_population

    n_ep = args.eval_episodes
    with torch.no_grad():
        res = evaluate_population(env, pop.params[:4], n_ep, greedy=args.eval_greedy, seeds=args.pbt_seed,
                                  episode0=r * n_ep)
        sums = torch.stack([x.sums() for x in res]).cpu()
    fitness = [x.summary(s)["mean_return"] for x, s in zip(res, sums)]
    if len(counts) > 1:
        fitness = gather_fitness(fitness, counts, pop.device)
    mine = [(d, s, f) for d, s, f in pbt_decisions(fitness, args.pbt_fraction, explore, generator)
            if lo <= d < lo + pop.P]
    before = pop.current_hparams()
    if len(counts) > 1:
        rows, steps = gather_states(pop, counts)
        src = torch.tensor([s for _, s, _ in mine], dtype=torch.int64).to(pop.device)
        pop.set_rows([d - lo for d, _, _ in mine], rows[src], steps[src], [f for _, _, f in mine])
    else:
        pop.copy_members([d for d, _, _ in mine], [s for _, s, _ in mine], [f for _, _, f in mine])
    after = pop.current_hparams()
    return fitness, [{"pbt_round": r, "epoch": epoch, "member": d, "parent": s,
                      "fitness": {"member": fitness[d], "parent": fitness[s]},
                      "hparams_before": before[d - lo], "hparams_after": after[d - lo]} for d, s, _ in mine]
