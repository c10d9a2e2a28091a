"""NumPy / SciPy oracle of `sot_b200.cluster.wasserstein_dbscan`'s definition, on a dense neighbour relation."""
import numpy as np
from scipy.sparse import csr_matrix
from scipy.sparse.csgraph import connected_components


def oracle(A, min_samples):
    """labels, core of the definition in `wasserstein_dbscan`'s docstring, for a dense boolean A."""
    R = A.shape[0]
    core = A.sum(1) >= min_samples
    idx = np.nonzero(core)[0]
    sub = A[np.ix_(idx, idx)]
    _, comp = connected_components(csr_matrix(sub | sub.T), directed=False)
    first = {}
    for c, i in zip(comp, idx):
        first.setdefault(c, i)  # idx ascends: the lowest core row of each component
    number = {c: k for k, c in enumerate(sorted(first, key=first.get))}
    labels = np.full(R, -1)
    labels[idx] = [number[c] for c in comp]
    for i in np.nonzero(~core)[0]:
        reach = labels[idx[A[idx, i]]]
        labels[i] = reach.min() if reach.size else -1
    return labels, core, len(number)
