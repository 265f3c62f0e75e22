import sys
sys.path.insert(0, "."); sys.path.insert(0, "tests")
from tgsfilter_b200 import synth
from tgsfilter_b200.engine import FilterEngine
batch = synth.make_config(5, 40000, with_names=False)
for k in (11, 13, 15, 16):
    p = synth.config_params(5); p.kmer = k; p.min_repeat = 5000
    with FilterEngine(p) as eng:
        eng.run(batch); eng.run(batch)
        st = eng.last_stage_ms()
    print("k", k, "kmer stage ms", round(st["kmer"], 3))
