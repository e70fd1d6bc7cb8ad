#!/usr/bin/env python
"""Phase -> source-line regions of the pipeline kernels (for tools/ncu_by_line.py), found by their marker comments so
that they follow edits.  usage: tools/make_regions.py <agent|emit> > regions.txt"""
import os, sys
SRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'layered_safe_marl_b200', 'csrc', 'lsm_kernel_spec.cuh')
lines = open(SRC).read().splitlines()
def at(marker, start=0):
    for i in range(start, len(lines)):
        if marker in lines[i]:
            return i + 1
    raise SystemExit(f"marker not found: {marker}")
AGENT = [('prologue', 'lsm_agent_kernel(const __grid_constant__'), ('P0 prefetch + state load', '---------------- P0: load'),
         ('P0 landmarks + curriculum', 'landmark tables of the group'), ('P1 action decode', '---------------- P1: action decode'),
         ('P1 argmin + filter_resolve', 'np.argmin over the others'), ('P1 integrate', 'everyone has read the pre-integration states'),
         ('P2 theta/speed/obs row', '---------------- P2: goal / reward / done'), ('P2 reach_goal reward', 'reward_reach_goal: navigation_graph_safe.py'),
         ('P2 goal update / tables', 'update_reached_goal_and_done (+ freeze_agent)'), ('P2 other-agents pass / stats', 'one pass over the other agents'),
         ('P2 info state', 'info_callback state: navigation_graph_safe.py'), ('P2 outputs', 'kp.b.reward_individual != nullptr) kp.b.reward_individual'),
         ('P3 reset', '---------------- P3: reset'), ('write-back', '---------------- state write-back'),
         ('record dump', '---------------- emit records -> global memory'), ('end', 'tl_end(kp.timeline, TL_AGENT_END)')]
EMIT = [('prologue + first record prefetch', 'lsm_emit_kernel(const __grid_constant__'), ('loop top: waits / prefetch issue', 'for (int ee = kp.env_begin + blockIdx.x'),
        ('distances', '(a) thresholded distance matrix'), ('masks', '(b) disconnected-entity bit masks'), ('adjacency (mask in place / direct stores)', '(d) adjacency'),
        ('node row builder', '(c) node features: one thread per'), ('node chunks + bulk copy issue', 'bool adj_sent = false;'),
        ('drain', 'every bulk copy issued by this block has finished READING'),
        ('end', 'tl_end(kp.timeline, TL_EMIT_END)')]
tab = AGENT if sys.argv[1] == 'agent' else EMIT
pos = []
cur = 0
for name, marker in tab:
    cur = at(marker, cur)
    pos.append((name, cur))
for (name, a), (_, b) in zip(pos[:-1], pos[1:]):
    print(a, b - 1, name)
