"""Small end-to-end pass over every kernel family for compute-sanitizer (memcheck / racecheck / synccheck)."""
import os, sys, numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from chinesecheckersagent_b200.engine import Engine, BatchedEnv, BatchedMCTS
from chinesecheckersagent_b200.model import ResidualCNN
from chinesecheckersagent_b200.selfplay import BatchedSelfPlay
from chinesecheckersagent_b200.data_generators import BatchedGreedyGenerator
from chinesecheckersagent_b200.arena import BatchedArena, GREEDY
eng = Engine(0)
env = BatchedEnv(300, engine=eng)
env.step_random(24); env.movegen(); env.encode(); env.greedy_candidates()
for variant in ("9", "10"):                                      # both env-step kernels, the default (10) last
    os.environ["CCX_STEP_VARIANT"] = variant
    BatchedEnv(1000, engine=eng).step_random(12, trace_games=40)
    BatchedEnv(70000, engine=eng).step_random(3)                   # > 148 x 448 games: the two-blocks-per-SM instantiation
os.environ.pop("CCX_STEP_VARIANT")
for variant in ("0", "2", "3", "1"):
    os.environ["CCX_GREEDY_VARIANT"] = variant
    g = BatchedEnv(500, engine=eng); g.play_greedy()
os.environ.pop("CCX_GREEDY_VARIANT")
BatchedMCTS(eng, num_itr=12).search(env.state)
BatchedMCTS(eng, num_itr=12, random_ties=True, tie_seed=3).search(env.state, evaluator=1, pre_expand=True)
m = ResidualCNN(engine=eng).load_weights(os.path.join(ROOT, 'tests', 'golden', 'good_model_weights.npz'))
for n in (3, 130):
    x = torch.randint(0, 7, (n, 7, 7, 7), dtype=torch.uint8, device='cuda')
    m.set_kernel('tc'); m.forward(x); m.set_kernel('tc_acc'); m.forward(x); m.set_kernel('simt'); m.forward(x)
m.set_kernel('tc_acc')
for ctx in (0, 1, 2, 3):                                          # accurate trunk: one tile per CTA, and 1-3 contexts sharing the weight slots
    m.eng.call('ccx_net_set_acc_contexts', ctx)
    for n in (5, 700, 1900):                                      # one context with a tile / a partial last round / several rounds
        m.forward(torch.randint(0, 7, (n, 7, 7, 7), dtype=torch.uint8, device='cuda'))
m.set_kernel('tc')
BatchedMCTS(eng, num_itr=6).search_net(env.state[:, :70].contiguous())
g9 = BatchedMCTS(eng, num_itr=9); r9 = env.state[:, :70].contiguous()
for _ in range(3): g9.search_net(r9)          # direct, captured, replayed (CUDA graph of the round loop)
m.set_kernel('tc_acc')
for _ in range(3): g9.search_net(r9)
m.set_kernel('tc')
sp = BatchedSelfPlay(eng, m.evaluate_states, n_slots=33, num_itr=5, max_iters=10)
for _ in range(8): sp.step()
sp.collect()
ring = BatchedSelfPlay(eng, m.evaluate_states, n_slots=33, num_itr=5, max_iters=8, ring=True, random_ties=True)
for _ in range(20): ring.step()                                   # wraps the record ring twice, discards over-long games
ring.collect()
BatchedSelfPlay(eng, m.evaluate_states, n_slots=20, num_itr=4, max_iters=60).play_games(30, max_iterations=40)
gm = BatchedMCTS(eng, num_itr=9, gumbel=True, gumbel_considered=4)    # Gumbel kernels: round trips, fused loop with its graph
gm.search_with(r9, m.evaluate_states, pre_expand=True)
for _ in range(3): gm.search_net(r9)
gsp = BatchedSelfPlay(eng, m.evaluate_states, n_slots=33, num_itr=5, max_iters=10, gumbel=True)
for _ in range(8): gsp.step()
gsp.collect()
from chinesecheckersagent_b200.board import Board
from chinesecheckersagent_b200.MCTS import MCTS, Node
b = Board(engine=eng); b.get_valid_moves(1); b.place(1, (5, 0), (3, 0)); b.check_win()
MCTS(Node(b, 2), m, num_itr=9).search()
BatchedGreedyGenerator(eng).generate(50, random_start=True)
a = BatchedArena(m, GREEDY, 9, num_itr=4)
for _ in range(4): a.step()
torch.cuda.synchronize()
print('sanitize pass done')
