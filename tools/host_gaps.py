import os, sys, time, operator
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from bench import make_gb1_library, make_tokens
from prograph_b200 import graph
from prograph_b200.engine import get_engine
eng = get_engine()
def t(): torch.cuda.synchronize(); return time.perf_counter()
big = "--big" in sys.argv
if big:
    M = make_tokens(1_000_000, 256, "mutational")
    tab = eng.pack(M); lut = graph.distance_lut(tab.words*32, operator.le, 1, False)
    graph.hamming_eps_graph(eng, tab, lut, False, 0, 1, None); del tab; torch.cuda.empty_cache()
G = make_gb1_library(); dev = torch.from_numpy(G).cuda()
lut = None
for it in range(6):
    t0 = t(); tab = eng.pack(dev); t1 = t()
    if lut is None: lut = graph.distance_lut(tab.words*32, operator.le, 1, False)
    a = t(); free = torch.cuda.mem_get_info(); b = t()
    deg, _ = eng.hamming_eps_mean_degree(tab, *graph._eps_sample(160000), tab, lut); c = t()
    keys, edges = eng.hamming_eps_sym(tab, lut, 0, 1, 0, capacity=int(1.5*deg*160000)+(4<<20)); d = t()
    eng.check_edge_budget(edges); e = t()
    csr = eng.edge_keys_to_csr(keys, 160000, tab.words, edges); f = t()
    print(f"it{it}: pack {1e3*(t1-t0):.2f} meminfo {1e3*(b-a):.2f} sample {1e3*(c-b):.2f} sym {1e3*(d-c):.2f} budget {1e3*(e-d):.2f} csr {1e3*(f-e):.2f} total {1e3*(f-t0):.2f} ms", flush=True)
    del keys, csr
