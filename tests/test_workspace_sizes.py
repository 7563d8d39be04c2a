"""b2048_backward_workspace_floats and b2048_backward_tc_layout are host-only: they size the caller's workspace from a
network descriptor and a chunk length.  Every tensor-core family carves its images out of that workspace, so the
values below (recorded from the library) pin which family's layout each shape is sized for."""
import ctypes as C
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "rl-2048-with-reinforce-and-actor-critic_b200", "libb2048.so")

CHUNKS = (4096, 65536, 1 << 20)

# (dims, activation, observations) -> b2048_backward_workspace_floats at each of CHUNKS
WORKSPACE_FLOATS = {
    ((16, 256, 256, 4), "ReLU", "log2"): (4276288, 67436608, 1078001728),
    ((16, 256, 256, 4), "ReLU", "raw"): (4276288, 67436608, 1078001728),
    ((16, 256, 256, 1), "ReLU", "log2"): (4264000, 67240000, 1074856000),
    ((16, 256, 256, 1), "ReLU", "raw"): (4264000, 67240000, 1074856000),
    ((16, 256, 256, 4), "Sigmoid", "log2"): (4276288, 67436608, 1078001728),
    ((272, 256, 128, 64, 4), "ReLU", "onehot"): (3727424, 59023424, 943759424),
    ((16, 64, 192, 64, 128, 4), "ReLU", "log2"): (3719232, 59015232, 943751232),
    ((16, 64, 192, 64, 128, 4), "Sigmoid", "log2"): (18800896, 59015232, 943751232),
    ((16, 96, 4), "ReLU", "log2"): (802880, 12845120, 205520960),     # fp32 kernels only
}

# chunk -> byte offsets of H1, H2, DL2, DL1, A1^T, d3^T and the total (b2048_backward_tc_layout)
TC_LAYOUT = {
    4096: (0, 2097152, 4194304, 6291456, 8388608, 8519680, 8650752),
    65536: (0, 33554432, 67108864, 100663296, 134217728, 136314880, 138412032),
    1 << 20: (0, 536870912, 1073741824, 1610612736, 2147483648, 2181038080, 2214592512),
}


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(LIB):
        import __graft_entry__ as g
        g.build()
    import b2048
    return b2048._lib.load()


def _desc(dims, activation, obs):
    import b2048
    d = b2048._lib.MlpDesc()
    d.n_layers, d.activation, d.obs_mode, d.obs_log2_scale = len(dims) - 1, b2048._lib.ACTV[activation], b2048._lib.OBS[obs], 1.0
    for i, v in enumerate(dims):
        d.dims[i] = v
    for layer in range(d.n_layers):      # never dereferenced: the sizes depend on the shape only
        d.W[layer] = d.b[layer] = 16
    return d


@pytest.mark.parametrize("shape", list(WORKSPACE_FLOATS), ids=lambda s: "-".join(map(str, s[0])) + f"-{s[1]}-{s[2]}")
def test_backward_workspace_floats(lib, shape):
    d = _desc(*shape)
    assert tuple(lib.b2048_backward_workspace_floats(C.byref(d), c) for c in CHUNKS) == WORKSPACE_FLOATS[shape]


@pytest.mark.parametrize("chunk", CHUNKS)
def test_backward_tc_layout(lib, chunk):
    out = (C.c_int64 * 7)()
    assert lib.b2048_backward_tc_layout(chunk, out) == 0
    assert tuple(out) == TC_LAYOUT[chunk]
