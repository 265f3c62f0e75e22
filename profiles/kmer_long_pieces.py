"""K4 stage time on ONT-like pieces (config[2] lengths, N50 ~30 kb: most pieces need 2-4 passes of k_kmer_tag16, the few
of more than 65 000 k-mers go to k_kmer_smem at k = 11 and to k_kmer at k = 13) and on HiFi pieces, k = 11 and 13.
Median and minimum of 5 timed runs after a warm-up.  python profiles/kmer_long_pieces.py"""
import statistics
import sys
sys.path.insert(0, "."); sys.path.insert(0, "tests")
from tgsfilter_b200 import synth
from tgsfilter_b200.engine import FilterEngine
for cfg, n in ((2, 20000), (5, 40000)):
    batch = synth.make_config(cfg, n, with_names=False)
    for k in (11, 13):
        p = synth.config_params(cfg); p.kmer = k; p.min_repeat = 50
        with FilterEngine(p) as eng:
            eng.run(batch)
            ms = []
            for _ in range(5):
                eng.run(batch)
                ms.append(eng.last_stage_ms()["kmer"])
        print("config", cfg, "reads", n, "bases", batch.n_bases, "k", k, "kmer stage ms median",
              round(statistics.median(ms), 3), "min", round(min(ms), 3))
