import sys, time
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np
from semadb_b200 import synth
from semadb_b200.vamana import IndexVamana, IndexVectorVamanaParameters
n = int(sys.argv[1]); mb = int(sys.argv[2]) if len(sys.argv) > 2 else 4096
X = synth.sift_shaped(n, 128, 3)
g = IndexVamana("b", IndexVectorVamanaParameters(128), start_vector=synth.start_vector(128, 99))
g.insert_config(1, mb, 16)
t = time.time()
g.insert_batch(np.arange(2, n + 2, dtype=np.uint64), X)
print("built", n, "in", time.time() - t, "s")
ids, d, c = g.search_batch(X[:100], 10, 75)
print("self-recall", (ids[:, 0] == np.arange(2, 102)).mean())
