"""K4 stage time on 40 000 HiFi pieces of 15 kb (config[5]) at k = 11 ... 21: k <= 16 runs k_kmer_tag16, k > 16 the
hash kernel k_kmer.  Median and minimum of 5 timed runs after a warm-up.  python profiles/kmer_k_sweep.py"""
import statistics
import sys
sys.path.insert(0, "."); sys.path.insert(0, "tests")
from tgsfilter_b200 import synth
from tgsfilter_b200.engine import FilterEngine
batch = synth.make_config(5, 40000, with_names=False)
for k in (11, 13, 15, 16, 17, 21):
    p = synth.config_params(5); p.kmer = k; p.min_repeat = 5000
    with FilterEngine(p) as eng:
        eng.run(batch)
        ms = []
        for _ in range(5):
            eng.run(batch)
            ms.append(eng.last_stage_ms()["kmer"])
    print("k", k, "kmer stage ms median", round(statistics.median(ms), 3), "min", round(min(ms), 3))
