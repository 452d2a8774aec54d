"""Which forward kernel a model gets: the default for each shape, the `*_impl` create options and their
SRS_*_IMPL environment variables, and the errors for a forced variant that does not fit the shape.

Builds models only (small vocabularies); nothing is predicted.
"""
import pytest

from sparrowrecsys_b200._lib import SRS_ERR_INVALID, SrsError
from sparrowrecsys_b200.spec import default_spec
from sparrowrecsys_b200.weights import init_weights

pytestmark = pytest.mark.gpu

RT_NEEDS = "SRS_DIN_IMPL=rt needs 16 < emb_dim <= 32 and hist_len <= 64, or 32 < emb_dim <= 64 and hist_len <= 256"
RTP_NEEDS = "SRS_DIN_IMPL=rtp needs 16 < emb_dim <= 32 and hist_len <= 64"
TC_NEEDS = "SRS_DIN_IMPL=tc needs 16 < emb_dim <= 32 and hist_len <= 128"
EMB_TC_NEEDS = "SRS_EMBMLP_IMPL=tc needs emb_dim <= 12"
FM_TC_NEEDS = "SRS_DEEPFM_IMPL=tc needs 12 < emb_dim <= 16"

# DIN defaults: row tiles for E padded to 32 with T 9..64 and E padded to 64 with T 9..256, the per-pair
# tensor-core kernel for E padded to 32 with T 65..128, CUDA cores otherwise.
_DIN_DEFAULT = {
    16: {},
    32: {9: "din_rt_kernel", 64: "din_rt_kernel", 65: "din_tc_kernel", 128: "din_tc_kernel"},
    48: {T: "din_rt64_kernel" for T in (9, 64, 65, 128, 129, 256)},
    64: {T: "din_rt64_kernel" for T in (9, 64, 65, 128, 129, 256)},
}
DIN_DEFAULTS = [("din", E, T, None, None, _DIN_DEFAULT[E].get(T, "din_kernel"))
                for E in (16, 32, 48, 64) for T in (8, 9, 64, 65, 128, 129, 256, 257)]

# (model, emb_dim, hist_len, create options, environment, expected kernel name or error message)
CASES = DIN_DEFAULTS + [
    ("din", 32, 50, {"din_impl": "rt"}, None, "din_rt_kernel"),
    ("din", 32, 8, {"din_impl": "rt"}, None, "din_rt_kernel"),
    ("din", 64, 200, {"din_impl": "rt"}, None, "din_rt64_kernel"),
    ("din", 16, 50, {"din_impl": "rt"}, None, RT_NEEDS),
    ("din", 32, 65, {"din_impl": "rt"}, None, RT_NEEDS),
    ("din", 64, 257, {"din_impl": "rt"}, None, RT_NEEDS),
    ("din", 32, 50, {"din_impl": "rtp"}, None, "din_rtp_kernel"),
    ("din", 64, 50, {"din_impl": "rtp"}, None, RTP_NEEDS),
    ("din", 32, 65, {"din_impl": "rtp"}, None, RTP_NEEDS),
    ("din", 32, 100, {"din_impl": "tc"}, None, "din_tc_kernel"),
    ("din", 32, 8, {"din_impl": "tc"}, None, "din_tc_kernel"),
    ("din", 32, 50, {"din_impl": "tc"}, None, "din_tc_kernel"),
    ("din", 64, 50, {"din_impl": "tc"}, None, TC_NEEDS),
    ("din", 32, 129, {"din_impl": "tc"}, None, TC_NEEDS),
    ("din", 32, 50, {"din_impl": "cudacore"}, None, "din_kernel"),
    ("din", 64, 300, {"din_impl": "cudacore"}, None, "din_kernel"),
    ("din", 32, 50, {"din_impl": "fastest"}, None, "din_rt_kernel"),
    ("din", 32, 100, {"din_impl": "fastest"}, None, "din_tc_kernel"),
    ("din", 16, 50, {"din_impl": "fastest"}, None, "din_kernel"),
    ("embeddingmlp", 10, 5, None, None, "embmlp_tc_kernel"),
    ("embeddingmlp", 16, 5, None, None, "embmlp_kernel"),
    ("embeddingmlp", 10, 5, {"embmlp_impl": "tc"}, None, "embmlp_tc_kernel"),
    ("embeddingmlp", 16, 5, {"embmlp_impl": "tc"}, None, EMB_TC_NEEDS),
    ("embeddingmlp", 10, 5, {"embmlp_impl": "cudacore"}, None, "embmlp_kernel"),
    ("embeddingmlp", 10, 5, {"embmlp_impl": "fastest"}, None, "embmlp_tc_kernel"),
    ("widendeep", 10, 5, None, None, "embmlp_tc_kernel<wide&deep>"),
    ("widendeep", 20, 5, None, None, "embmlp_kernel<wide&deep>"),
    ("widendeep", 10, 5, {"embmlp_impl": "cudacore"}, None, "embmlp_kernel<wide&deep>"),
    ("widendeep", 20, 5, {"embmlp_impl": "tc"}, None, EMB_TC_NEEDS),
    ("deepfm", 16, 5, None, None, "deepfm_tc_kernel"),
    ("deepfm", 10, 5, None, None, "deepfm_kernel"),
    ("deepfm", 32, 5, None, None, "deepfm_kernel"),
    ("deepfm", 13, 5, {"deepfm_impl": "tc"}, None, "deepfm_tc_kernel"),
    ("deepfm", 10, 5, {"deepfm_impl": "tc"}, None, FM_TC_NEEDS),
    ("deepfm", 16, 5, {"deepfm_impl": "cudacore"}, None, "deepfm_kernel"),
    ("neuralcf", 10, 5, None, None, "ncf_kernel<neural_cf_model_1>"),
    ("twotowers", 10, 5, None, None, "ncf_kernel<two_towers>"),
    ("deepfm_v2", 16, 5, None, None, "deepfm2_kernel"),
    ("dien", 32, 50, None, None, "dien_kernel"),
    # the environment variables select when no option is given; an option takes precedence
    ("din", 32, 50, None, {"SRS_DIN_IMPL": "tc"}, "din_tc_kernel"),
    ("din", 32, 50, {"din_impl": "rt"}, {"SRS_DIN_IMPL": "cudacore"}, "din_rt_kernel"),
    ("din", 32, 50, {"din_impl": "cudacore"}, {"SRS_DIN_IMPL": "tc"}, "din_kernel"),
    ("din", 64, 50, {"din_impl": "cudacore"}, {"SRS_DIN_IMPL": "tc"}, "din_kernel"),
    ("embeddingmlp", 10, 5, None, {"SRS_EMBMLP_IMPL": "cudacore"}, "embmlp_kernel"),
    ("embeddingmlp", 10, 5, {"embmlp_impl": "tc"}, {"SRS_EMBMLP_IMPL": "cudacore"}, "embmlp_tc_kernel"),
    ("deepfm", 16, 5, None, {"SRS_DEEPFM_IMPL": "cudacore"}, "deepfm_kernel"),
    ("deepfm", 16, 5, {"deepfm_impl": "tc"}, {"SRS_DEEPFM_IMPL": "cudacore"}, "deepfm_tc_kernel"),
]

_ENV = ("SRS_DIN_IMPL", "SRS_EMBMLP_IMPL", "SRS_DEEPFM_IMPL")


@pytest.mark.parametrize("model,E,T,options,env,expected", CASES)
def test_kernel_selection(model, E, T, options, env, expected, monkeypatch):
    from sparrowrecsys_b200.model import CTRModel
    for k in _ENV:
        monkeypatch.delenv(k, raising=False)
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    spec = default_spec(model, emb_dim=E, hist_len=T, n_movies=64, n_users=32)
    W = init_weights(spec, E * 1000 + T)
    if expected.startswith("SRS_"):
        with pytest.raises(SrsError) as exc:
            CTRModel(spec, W, device=0, options=options)
        assert exc.value.code == SRS_ERR_INVALID
        assert expected in str(exc.value)
    else:
        with CTRModel(spec, W, device=0, options=options) as m:
            assert m.kernel_name == expected
