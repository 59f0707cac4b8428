import os, sys, numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ia2c_b200.trainer import IA2CTrainer, reference_init
E, N = 1024, 256
init = reference_init(N, 5, seed=3)
keys = ("obs", "act", "reward", "partner_true", "partner_pred", "belief_records", "ep_return", "critic_grad", "critic_params", "actor_grad", "actor_params", "env_state")
for mode in ("auto", "step"):
    for n_ep in (1, 2):
        runs = []
        for rep in range(3):
            tr = IA2CTrainer(E, n_agents=N, init=init, seed=17, rollout_kernel=mode)
            for _ in range(n_ep):
                tr.train_episode()
            torch.cuda.synchronize()
            runs.append({k: getattr(tr, k).detach().cpu().numpy().copy() for k in keys})
            del tr
        bad = [k for k in keys if not (np.array_equal(runs[0][k], runs[1][k]) and np.array_equal(runs[0][k], runs[2][k]))]
        print(mode, "episodes", n_ep, "differing:", bad)
        if bad:
            k = bad[0]
            d = np.argwhere(runs[0][k] != runs[1][k])
            print("   first diffs in", k, d[:5].tolist(), "count", len(d))
