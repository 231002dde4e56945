"""The IMPALA learners written out by hand (test helper): per family, the forward of a set of time columns under
the current module, then impala.vtrace, the loss written from its formula, torch's clip_grad_norm_ (or its per-agent
counterpart as a loop over the agents) and the optimizer step, on the same generator draws as the learners.  The
recurrent forwards run one max_seq_len chunk at a time over all columns, not the learners' single batched call."""
import torch

from dl_reference_models_b200 import impala
from dl_reference_models_b200.cte_rollout import joint_logp_entropy
from dl_reference_models_b200.recurrent import features_from_channels
from dl_reference_models_b200.rollout import draw_permutation, per_agent_minibatches


def forward(kind, policy, batch, idx, L=32):
    """(target logp, entropy, value), each [T, M], of batch columns idx."""
    T = batch.rewards.shape[0]
    Cat = torch.distributions.Categorical
    if kind in ("mlp", "lstm"):
        N = batch.actions.shape[2]
        b, n = idx // N, idx % N
        acts = batch.actions[:, b, n]
    else:
        acts = batch.actions[:, idx]
    if kind == "mlp":
        feats, masks = batch.features[:, b, n], batch.masks[:T][:, b, n]
        lg, v = policy(feats.reshape(-1, feats.shape[-1]), masks.reshape(-1, 5))
        d = Cat(logits=lg.reshape(T, idx.numel(), -1))
        return d.log_prob(acts), d.entropy(), v.reshape(T, -1)
    if kind == "cte":
        lg, v = policy(batch.grid[:T][:, idx], batch.masks[:T][:, idx])
        lp, ent = joint_logp_entropy(lg, acts)
        return lp, ent, v
    lgs, vs = [], []
    for k in range(T // L):
        s = slice(k * L, (k + 1) * L)
        if kind == "lstm":
            g = lambda x: x[s][:, b, n]   # noqa: E731
            f = features_from_channels(g(batch.local_obs), g(batch.goal_delta), g(batch.blocking_prev))
            lg, v, _ = policy.sequence(f, g(batch.masks), g(batch.prev_actions), g(batch.prev_rewards),
                                       batch.resets[s][:, b], (batch.chunk_h[k, idx], batch.chunk_c[k, idx]))
        else:
            g = lambda x: x[s][:, idx]   # noqa: E731
            lg, v, _ = policy.sequence(g(batch.grid), g(batch.masks), g(batch.prev_actions), g(batch.prev_rewards),
                                       g(batch.resets), (batch.chunk_h[k, idx], batch.chunk_c[k, idx]))
        lgs.append(lg)
        vs.append(v)
    lg = torch.cat(lgs)
    if kind == "lstm":
        d = Cat(logits=lg)
        return d.log_prob(acts), d.entropy(), torch.cat(vs)
    lp, ent = joint_logp_entropy(lg, acts)
    return lp, ent, torch.cat(vs)


def column_draws(batch, per_agent, minibatch, generator):
    T = batch.rewards.shape[0]
    n = batch.rewards[0].numel()
    S = max(1, minibatch // T)
    dev = batch.rewards.device
    if per_agent:
        N = batch.rewards.shape[2]
        return [(s * N + torch.arange(N, device=dev)).reshape(-1) for s in per_agent_minibatches(n // N, N, S, dev, generator)]
    perm = draw_permutation(n, dev, generator)
    return [perm[i:i + S] for i in range(0, n, S)]


def loss_of(lp, ent, v, vs, pg, *, vf_coeff, entropy_coeff, num_agents=None):
    T = lp.shape[0]
    mean = (lambda x: x.mean()) if num_agents is None else (lambda x: x.reshape(T, -1, num_agents).mean((0, 1)).sum())  # noqa: E731
    return -mean(lp * pg) + vf_coeff * 0.5 * mean((v - vs) ** 2) - entropy_coeff * mean(ent)


def clip_per_agent_loop(policy, max_norm, N):
    params = [p for p in policy.parameters() if p.grad is not None]
    for j in range(N):
        norm = torch.stack([p.grad[j].norm() for p in params]).norm()
        coef = torch.clamp(max_norm / (norm + 1e-6), max=1.0)
        for p in params:
            p.grad[j].mul_(coef)


def hand_update(kind, policy, opt, batch, *, per_agent=False, generator=None, minibatch=1024, max_minibatches=None,
                L=32, grad_clip=40.0, gamma=0.99, clip_rho=1.0, clip_pg_rho=1.0, vf_coeff=0.5, entropy_coeff=0.01):
    N = batch.rewards.shape[2] if per_agent else None
    for i, idx in enumerate(column_draws(batch, per_agent, minibatch, generator)):
        if max_minibatches is not None and i >= max_minibatches:
            break
        lp, ent, v = forward(kind, policy, batch, idx, L)
        vs, pg = impala.vtrace(lp.detach(), batch.logp, v.detach(), batch.rewards, batch.dones, batch.last_value,
                               columns=idx, gamma=gamma, clip_rho=clip_rho, clip_pg_rho=clip_pg_rho)
        loss = loss_of(lp, ent, v, vs, pg, vf_coeff=vf_coeff, entropy_coeff=entropy_coeff, num_agents=N)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        if per_agent:
            clip_per_agent_loop(policy, grad_clip, N)
        else:
            torch.nn.utils.clip_grad_norm_(policy.parameters(), grad_clip)
        opt.step()
