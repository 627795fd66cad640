"""A freshly created model (no set_states) starts every cell from the stack's default-constructed state, as a reference
region_model does.  Expected values are the oracle's state structs in the flat ABI order."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

NB = 5  # snow bins of the default hbv_snow / hbv_physical_snow parameter
DEFAULT_STATE = {
    # gamma_snow::state (oracle/sho_core.hpp:498-501) + kirchner.q (oracle/sho_pt_gs_k.hpp:62-66)
    "PTGSKModel": [0.4, 0.1, 30000.0, 1.26, 0.0, 0.0, 0.0, 0.0, 0.1],
    # swe, sca, sp[5], sw[5] (oracle/sho_hbv.hpp:82-84) + kirchner.q (:266-268)
    "PTHSKModel": [0.0] * (2 + 2 * NB) + [0.1],
    # swe, sca, sp[5], sw[5], soil.sm, tank.uz, tank.lz (oracle/sho_hbv.hpp:198, 214, 362-372)
    "HbvStackModel": [0.0] * (2 + 2 * NB) + [0.0, 20.0, 10.0],
    # skaugen::state (oracle/sho_skaugen.hpp:72-75) + kirchner.q (:289-291)
    "PTSSKModel": [4.077, 40.77, 0.0, 0.0, 0.0, 0.0, 0.0, 0.1],
    # hbv_physical_snow::state after distribute() (oracle/sho_hps.hpp:41-50): sp[5], sw[5], albedo[5], iso_pot_energy[5],
    # surface_heat, swe, sca; + kirchner.q (:254-256)
    "PTHPSKModel": [0.0] * (2 * NB) + [0.4] * NB + [0.0] * NB + [30000.0, 0.0, 0.0, 0.1],
}


@pytest.mark.parametrize("cls_name", sorted(DEFAULT_STATE))
def test_fresh_model_state_is_the_default(cls_name):
    import shyft_b200 as sb
    n = 70
    rng = np.random.default_rng(3)
    geo = sb.geo_cell_data_vector(rng.uniform(0, 1e4, n), rng.uniform(0, 1e4, n), rng.uniform(100, 1500, n), area=1e6,
                                  catchment_id=np.repeat([1, 2], n // 2))
    m = getattr(sb, cls_name)(geo)
    want = np.tile(np.array(DEFAULT_STATE[cls_name]), (n, 1))
    assert m.state_size == want.shape[1]
    got = m.get_states()
    assert got.shape == want.shape
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), f"first differing cell row: {got[np.any(got != want, axis=1)][:1]}"
