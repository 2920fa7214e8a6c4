import os, sys, numpy as np
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', '..'))
from nornicdb_b200.knn import KnnIndex
for (n,d,Q,k,metric) in [(40000,64,8,100,'cosine'),(2_000_000,1024,128,100,'dot'),(2_000_000,1024,64,10,'cosine'),(1_000_000,1024,64,10,'cosine'),(5000,256,64,10,'cosine')]:
    ix = KnnIndex(d, metric=metric)
    ix.fill_uniform(n, 7)
    ix.set_path('filter')
    q = np.random.default_rng(1).uniform(-1,1,(Q,d)).astype(np.float32)
    ix.search(q, k)
    print(n,d,Q,k,metric, 'flags', ix.debug_flags())
    ix.release()
