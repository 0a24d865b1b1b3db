"""CPU checks of the parameter arena and workspace sizes iql_create reports (iql_get_layout; no kernel is launched).

The workspace holds the device tables (per-member scalars, counters, problem descriptors, tensor maps, loss ring, TF32
shadows) and then the per-member activation area; a caller allocates exactly `workspace_bytes`.  The values below
are recorded ones, so a change that moves the parameter arenas or resizes the workspace does so knowingly rather than
as a side effect.  The shapes are the six bench.py workloads (members per
GPU and the default updates per call), the row-split output-layer backward and K-split input-layer weight gradient
(batch 4096 with 1 member, batch 2048 with 4), an FP32-math engine (no shadow tables) and a deterministic policy with
3 hidden layers."""
import pytest

from jsrl_corl_b200.engine import query_layout

# (members, state_dim, action_dim, hidden_dim, n_hidden, batch, deterministic, math_mode, max_steps_per_call)
#   -> (param_floats, q_floats, v_begin, v_end, actor_begin, actor_end, workspace_bytes)
LAYOUTS = {
    "halfcheetah_ens64": ((64, 17, 6, 256, 2, 256, False, "tf32", 320),
                          (289184, 144960, 144960, 216416, 216416, 289184, 606208000)),
    "hopper_ens64": ((64, 11, 3, 256, 2, 256, True, "tf32", 320),
                     (280192, 140864, 140864, 210272, 210272, 280192, 596623360)),
    "hopper_single": ((1, 11, 3, 256, 2, 256, True, "tf32", 1000),
                      (280192, 140864, 140864, 210272, 210272, 280192, 9513984)),
    "antmaze_jsrl": ((1, 29, 8, 256, 3, 256, False, "tf32", 1000),
                     (567200, 284736, 284736, 425056, 425056, 567200, 15138304)),
    "pen_sweep256": ((256, 45, 24, 256, 2, 256, False, "tf32", 320),
                     (332704, 169536, 169536, 248160, 248160, 332704, 2632449280)),
    "stress_4x1024": ((1, 11, 3, 1024, 4, 4096, True, "tf32", 100),
                      (12662912, 6334528, 6334528, 9497696, 9497696, 12662912, 767746560)),
    "split_b4096_1member": ((1, 11, 3, 256, 2, 4096, True, "tf32", 8),
                            (280192, 140864, 140864, 210272, 210272, 280192, 99989760)),
    "split_b2048_4members": ((4, 17, 6, 256, 2, 2048, False, "tf32", 8),
                             (289184, 144960, 144960, 216416, 216416, 289184, 210470400)),
    "fp32_math": ((8, 17, 6, 256, 2, 256, False, "fp32", 16),
                  (289184, 144960, 144960, 216416, 216416, 289184, 46824960)),
    "deterministic_3x256": ((4, 29, 8, 256, 3, 256, True, "tf32", 16),
                            (567168, 284736, 284736, 425056, 425056, 567168, 60498688)),
}


@pytest.mark.parametrize("name", sorted(LAYOUTS))
def test_layout_and_workspace_size_are_pinned(name):
    (S, Sd, A, H, L, B, det, math, k), expected = LAYOUTS[name]
    lay, _ = query_layout(S, Sd, A, H, L, B, det, math_mode=math, max_steps_per_call=k)
    got = (lay.param_floats, lay.q_floats, lay.v_begin, lay.v_end, lay.actor_begin, lay.actor_end, lay.workspace_bytes)
    assert got == expected
