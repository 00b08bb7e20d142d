"""Leaves per tree and iteration (virtual loss): throughput at the headline config (4096 games, 800 sims/move).
ONE_LAUNCH=0 times the per-iteration kernels where the one-launch search would otherwise be picked (K = 1 / 2 / 4)."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from betazero_b200 import env, mcts, net as netmod

B, S = int(os.environ.get("GAMES", "4096")), 800
ONE_LAUNCH = None if os.environ.get("ONE_LAUNCH", "") == "" else os.environ["ONE_LAUNCH"] != "0"  # unset: the default choice
model = netmod.make_net("mlp", seed=0)
me, opp, _ = env.reversi_init(B)

def timed(fn, n=5):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n

for K in [int(x) for x in os.environ.get("LEAVES", "1,2,4,8").split(",")]:
    for G in [int(x) for x in os.environ.get("LANES", "0").split(",")]:
        s = mcts.BatchedMCTS(mcts.TreePools(B, S, n_leaves=K, group_lanes=G), mcts.FusedNetEvaluator(model), graph_unroll=16,
                              one_launch=ONE_LAUNCH)
        s.prepare()
        SK = S - S % K  # K = 3: 798 simulations
        def one():
            s.reset(me, opp)
            s.run(SK)
        ms = timed(one)
        cnt = s.root_policy()[0]
        s.check_errors()
        st = s.stats()
        print(f"leaves={K} lanes={G or 'auto'}{' one-launch' if s.one_launch else ''}: {ms:.2f} ms per {SK}-sim search = {ms / (SK // K) * 1e3:.2f} us/iteration, "
              f"{B * SK / ms / 1e3:.1f} M sims/s; mean depth {st['mean_depth']:.2f}, root visits {int(cnt[0].sum())}, "
              f"max root share {float((cnt.max(1).values.float() / cnt.sum(1).clamp_min(1)).mean()):.3f}")
        del s
        torch.cuda.empty_cache()
