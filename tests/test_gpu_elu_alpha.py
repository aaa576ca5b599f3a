"""The ELU select of the tensor-core kernel depends on the layer's alpha.

For 0 <= alpha <= 1 the hidden layers' ELU is max.NaN(z', c*2^-|z'| - c), which equals the ELU only because
alpha*(e^z - 1) >= z for every z <= 0.  For alpha > 1 that inequality fails just below 0 (alpha*(e^z - 1) ~ alpha*z < z),
so those layers must keep the z' < 0 select.  The policies here put most pre-activations where the two differ
(bias -0.4; alpha*(e^z - 1) - z peaks at z = -ln(alpha)), and all-positive output weights add the differences up."""
import numpy as np
import pytest

from go2_onnx_controller_b200 import PolicyBatch, capi, onnx_writer
from oracle import coracle

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(300)]

DIMS = (64, 128, 128, 12)
TOL = {capi.PREC_FP16: 2e-2, capi.PREC_BF16: 1e-1}


def make_policy(path, alpha):
    rng = np.random.default_rng(15)
    ws = [rng.normal(0, 1.0 / np.sqrt(k), (n, k)).astype(np.float32) for k, n in zip(DIMS[:-1], DIMS[1:])]
    ws[-1] = np.abs(ws[-1])
    bs = [np.full(n, -0.4, np.float32) for n in DIMS[1:-1]] + [np.zeros(DIMS[-1], np.float32)]
    onnx_writer.write_policy(str(path), ws, bs, elu_alpha=alpha)
    return ws, bs


def forward_max_form(ws, bs, X, alpha):
    """the policy evaluated with the max form of the ELU whatever alpha is (fp64)"""
    h = X.astype(np.float64)
    for i, (w, b) in enumerate(zip(ws, bs)):
        z = h @ w.astype(np.float64).T + b
        h = np.maximum(z, alpha * np.expm1(-np.abs(z))) if i < len(ws) - 1 else z
    return h


@pytest.mark.parametrize("alpha", [1.5, 1.0])
def test_tensor_core_elu_alpha(torch_cuda, tmp_path, alpha):
    torch = torch_cuda
    path = tmp_path / "elu.onnx"
    ws, bs = make_policy(path, alpha)
    cm = coracle.CModel(str(path))
    rng = np.random.default_rng(1)
    p = PolicyBatch(str(path))
    try:
        assert p.info.tensor_core_path == 1
        for B in (1000, 4096):
            X = rng.normal(0, 1, (B, DIMS[0])).astype(np.float32)
            ref = cm.forward_f64(X, 4)
            wrong = np.abs(forward_max_form(ws, bs, X, alpha) - ref).max()
            # the inputs tell the two selects apart for alpha > 1 (and the max form is the ELU for alpha <= 1)
            assert wrong > 10 * TOL[capi.PREC_FP16] if alpha > 1 else wrong < 1e-9, wrong
            d_obs = torch.from_numpy(X).cuda()
            d_act = torch.full((B, DIMS[-1]), 777.0, device="cuda", dtype=torch.float32)
            for prec in (capi.PREC_FP16, capi.PREC_BF16):
                d_act.fill_(777.0)
                p.infer_device(d_obs.data_ptr(), d_act.data_ptr(), B, prec, 0)
                torch.cuda.synchronize()
                err = np.abs(d_act.cpu().numpy() - ref).max()
                assert err <= TOL[prec], (prec, B, err)
    finally:
        p.close()
