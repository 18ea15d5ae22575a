"""A destroyed context gives back the device memory it allocated.

Every device buffer of a context frees itself when the context is destroyed.  The test creates, uses and destroys
contexts in a loop that reaches the null, pair-table, distance, clustering-null and protein mapping buffers, and
checks that the device's free memory does not fall from cycle to cycle."""
import pytest
import helpers as H

pytestmark = pytest.mark.gpu

CYCLES = 10
# bytes; every null, pair-table, distance and protein partial buffer below holds 1.6 MB or more, so leaking any
# one of them loses at least 16 MB over the cycles
TOLERANCE = 4 << 20


def _setup(ctx, c):
    ctx.set_tree(c["parent"], c["brlen"])
    ctx.set_model(c["Q"], c["pi"], c["rates"], c["probs"])
    ctx.set_alignment(c["codes"], c["code_mask"])


def _cycle(api, dna1, dna2, protein):
    a, b, p = api.Context(), api.Context(), api.Context()
    try:
        _setup(a, dna1)
        a.map()
        a.null_intra("correlation", 3, 50, 4000, K=10)              # 200 000 samples: 1.6 MB per sample array
        a.pairs("correlation")                                        # 179 700 rows in the resident pair table
        a.distance_matrix("correlation", want=False)                  # 600 x 600 matrix
        a.cluster("complete")
        a.cluster_null("correlation", "complete", 5, 0, 4, 10)        # four replicate matrices and dendrograms
        a.mica_null_parametric(7, 4, 2000, K=10)
        _setup(b, dna2)                                               # same topology, another data set
        b.map()
        a.pairs_inter(b, "correlation")
        a.null_inter(b, "correlation", 11, 20, 2000)
        _setup(p, protein)                                            # the protein tensor-core kernels' partials
        p.map()
        p.null_intra("correlation", 13, 10, 1000, K=10)
    finally:
        a.close(); b.close(); p.close()


def test_contexts_give_back_their_device_memory():
    import torch
    from comap_b200 import api
    dna1 = H.random_dna_case(20, 600, 31, mean_brlen=0.08)
    dna2 = H.random_dna_case(20, 450, 31, mean_brlen=0.08)          # same seed -> same topology
    dna2["brlen"] = dna2["brlen"] * 1.5
    protein = H.myoglobin_inputs()
    _cycle(api, dna1, dna2, protein)  # warm-up: lazy module loading and allocator pools
    torch.cuda.synchronize()
    free_before = torch.cuda.mem_get_info()[0]
    for _ in range(CYCLES):
        _cycle(api, dna1, dna2, protein)
    torch.cuda.synchronize()
    free_after = torch.cuda.mem_get_info()[0]
    assert free_before - free_after <= TOLERANCE, \
        "%.1f MB of device memory lost over %d context cycles" % ((free_before - free_after) / 2**20, CYCLES)
