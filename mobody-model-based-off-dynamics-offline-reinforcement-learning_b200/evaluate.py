"""Policy evaluators (SURVEY.md section 8f rank 4), mirrors of train_mobody.py:53-140 (``eval_policy_batch``: a vector of
environments stepped in lock step) and :142-205 (``eval_policy``).  The environments are the caller's (gym / mujoco are not
part of this image); the policy forward is the CUDA policy kernel, one launch for the whole vector of states per step, and
the optional model check (``eval_trg`` with a dynamics object) is one fused dynamics step over every visited transition.
``eval_policy_in_model`` needs no environment: it scores the policy in the agent's learned target-domain dynamics.
"""
import numpy as np
import torch


def _model_check(dynamics, states, actions, next_states, rewards):
    """train_mobody.py:100-130 / 166-196: one dynamics.step over the visited transitions; prints and returns the two errors."""
    dev = dynamics.model.elites.device
    s, a, ns = (torch.as_tensor(np.asarray(x), dtype=torch.float32, device=dev) for x in (states, actions, next_states))
    r = torch.as_tensor(np.asarray(rewards), dtype=torch.float32, device=dev)
    next_obs, reward, _, info = dynamics.step(s, a, False)
    obs_mse = torch.mean(torch.sqrt(torch.sum((next_obs - ns) ** 2, dim=1)))
    reward_mse = torch.mean((r - reward.squeeze(1)) ** 2)
    both = torch.stack([reward_mse, obs_mse]).cpu()
    print("reward mse", float(both[0]))
    print("obs mse", float(both[1]))
    return float(both[0]), float(both[1])


def eval_policy_batch(policy, env, policy_distribution, eval_episodes=10, eval_cnt=None, dynamics=None, eval_trg=False):
    """train_mobody.py:53-140.  ``env`` is a vector environment of ``eval_episodes`` copies: reset() -> states [E, S],
    step(actions [E, A]) -> (next_states, rewards [E], dones [E], info).  An episode's return counts the rewards up to and
    including its first done step; the loop ends when every copy has finished once."""
    states, actions, next_states, rewards = [], [], [], []
    state = env.reset()
    finished = np.zeros(eval_episodes, dtype=bool)
    done_index = np.full(eval_episodes, 1000, dtype=int)
    reward_all = np.zeros((eval_episodes, 1000))
    it = 0
    while finished.sum() < eval_episodes:
        action = policy.select_action(np.array(state), policy_distribution)
        next_state, reward, done, _ = env.step(action)
        reward_all[:, it] = reward
        live = ~finished                                              # rows still recording (:75-88), incl. the step that ends them
        action2d = np.asarray(action).reshape(eval_episodes, -1)
        states.append(np.asarray(state)[live]); actions.append(action2d[live])
        next_states.append(np.asarray(next_state)[live]); rewards.append(np.asarray(reward)[live])
        ended = live & np.asarray(done, dtype=bool)
        done_index[ended] = it
        finished |= ended
        state = next_state
        it += 1
    avg_reward = sum(reward_all[i, :done_index[i] + 1].sum() for i in range(eval_episodes)) / eval_episodes
    if eval_trg and dynamics is not None:
        _model_check(dynamics, np.concatenate(states), np.concatenate(actions), np.concatenate(next_states), np.concatenate(rewards))
    print("[{}] Evaluation on {} over {} episodes: {}".format(eval_cnt, "target" if eval_trg else "source", eval_episodes, avg_reward))
    return avg_reward


def eval_policy(policy, env, policy_distribution, eval_episodes=10, eval_cnt=None, dynamics=None, eval_trg=False):
    """train_mobody.py:142-205: ``eval_episodes`` sequential episodes of a single environment."""
    states, actions, next_states, rewards = [], [], [], []
    avg_reward = 0.0
    for _ in range(eval_episodes):
        state, done = env.reset(), False
        while not done:
            action = policy.select_action(np.array(state), policy_distribution)
            next_state, reward, done, _ = env.step(action)
            states.append(state); actions.append(action); next_states.append(next_state); rewards.append(reward)
            avg_reward += reward
            state = next_state
    avg_reward /= eval_episodes
    if eval_trg and dynamics is not None:
        _model_check(dynamics, states, actions, next_states, rewards)
    print("[{}] Evaluation on {} over {} episodes: {}".format(eval_cnt, "target" if eval_trg else "source", eval_episodes, avg_reward))
    return avg_reward


def eval_policy_in_model(agent, init_states, horizon=1000, penalized=False, eval_cnt=None):
    """The evaluators' average return with the learned target dynamics standing in for the environment: one episode per start
    state (``init_states`` [N, S], e.g. target-domain dataset states), at most ``horizon`` steps, the policy acting
    deterministically (MOBODY.evaluate_in_model).  Prints in the evaluators' format and returns the average return."""
    res, info = agent.evaluate_in_model(init_states, horizon, penalized=penalized)
    n = int(res["returns"].shape[0])
    print("[{}] Evaluation in the learned target model over {} episodes: {}".format(eval_cnt, n, info["return_mean"]))
    return info["return_mean"]
