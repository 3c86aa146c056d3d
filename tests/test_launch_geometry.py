"""Launch geometry of hmpc_create (csrc/hmpc_geometry.cuh: launch_geometry): which build of the CTA kernel and of the
warp-per-hopper kernel a configuration launches, with how many threads, how much shared memory and how large a grid.
The CPU tests run the host function through the emulation library for every configuration at B200 limits; the -m gpu
test checks that the library's handles report what the function predicts for the device they run on."""
import itertools

import pytest

from tests.emul import default_config, kernel_builds, launch_geometry

# B200: 148 SMs, 227 KB of shared memory per block (opt-in), 228 KB per SM, 126 MB of L2
B200 = dict(sm_count=148, smem_block=227 * 1024, smem_sm=228 * 1024, l2=126 * 1024 * 1024)
# registers per thread of each warp build (ptxas, sm_100a); hot_path_info reports them on the GPU (test below)
WARP_REGS = {15: 128, 14: 128, 13: 128, 12: 166, 11: 168, 10: 168, 8: 220, 7: 128, 6: 166, 5: 168, 4: 166}
ADMM_REGS = {10: 168, 6: 236}
BATCH = 131072


def geometry(kcap=56, limits=B200, batch=BATCH, **cfg):
    builds = kernel_builds()
    return launch_geometry(default_config(batch=batch, **cfg), kcap, warp_regs=[WARP_REGS[w] for w in builds["warp"]],
                           admm_regs=[ADMM_REGS[w] for w in builds["admm"]], **limits)


def test_register_table_covers_the_builds():
    builds = kernel_builds()
    assert sorted(builds["warp"]) == sorted(WARP_REGS) and sorted(builds["admm"]) == sorted(ADMM_REGS)


@pytest.mark.parametrize("kcap", [56, 48, 40])
def test_every_configuration_fits_its_build(kcap):
    builds = kernel_builds()
    L = B200
    for N, dyn, precision, solver, hot_path in itertools.product(range(3, 65), (2, 3), (0, 1), (0, 1), (0, 1)):
        if precision == 1 and N > 10:
            continue                     # rejected by hmpc_create before any geometry
        g = geometry(kcap, N=N, dyn=dyn, precision=precision, solver=solver, hot_path=hot_path)
        where = (N, dyn, precision, solver, hot_path, kcap)
        assert not g["unsupported"], where
        # CTA kernel: a build of the list with its own thread count, shared memory per block and per SM within the limits
        assert g["threads"] == builds["cta"][g["cta"]], where
        if 6 * N <= 64:
            assert g["cta"] == ("n10_f32" if precision else "n10_f64_admm" if solver else "n10_f64") and g["ws_bytes"] == 0, where
            per_sm = -(-g["grid"] // L["sm_count"])
        else:
            per_sm = {"wide_gmem4": 4, "wide_gmem2": 2}[g["cta"]]
            assert g["ws_bytes"] > 0 and g["ws_bytes"] % g["grid"] == 0, where
        assert g["grid"] == min(BATCH, L["sm_count"] * per_sm), where
        assert g["smem"] + 1024 <= L["smem_block"] and per_sm * (g["smem"] + 1024) <= L["smem_sm"], where
        # warp kernel: exactly the warm-path configurations, a build of the list, sized for the wpc it launches
        warm_path = hot_path == 0 and precision == 0 and N <= 10
        assert bool(g["warp"]) == warm_path, where
        if not warm_path:
            continue
        assert g["kcap"] == kcap and bool(g["admm"]) == bool(solver), where
        assert g["wpc"] in (builds["admm"] if solver else builds["warp"]), where
        assert g["regs"] == (ADMM_REGS if solver else WARP_REGS)[g["wpc"]], where
        ctas = g["warp_per_sm"] // g["wpc"]
        assert ctas * g["wpc"] == g["warp_per_sm"] and ctas >= 1, where
        assert g["warp_smem"] == 8 * g["wdoubles"] * g["wpc"], where          # one slice per launched warp (32 * wpc threads)
        assert g["warp_smem"] + 512 <= L["smem_block"] and ctas * (g["warp_smem"] + 1024) <= L["smem_sm"], where
        assert ctas * 32 * g["wpc"] * ((g["regs"] + 7) & ~7) <= 65536, where
        assert g["warp_grid"] == min(-(-BATCH // g["wpc"]), L["sm_count"] * ctas), where
        assert g["group"] == (0 if solver else g["wpc"] + 256), where


def test_cta_build_by_horizon():
    """N <= 10: shared-memory matrices; N > 10: four 128-thread CTAs per SM while 4 x 148 workspaces fit the L2, then
    two 256-thread CTAs."""
    for N in range(3, 65):
        for dyn in (2, 3):
            want = "n10_f64" if N <= 10 else "wide_gmem4" if N <= 24 else "wide_gmem2"
            assert geometry(N=N, dyn=dyn)["cta"] == want, (N, dyn)
    assert geometry(N=10, solver=1)["cta"] == "n10_f64_admm" and geometry(N=10, precision=1)["cta"] == "n10_f32"


def test_warp_build_by_horizon_and_kcap():
    picks = {56: {3: 14, 4: 13, 5: 13, 6: 13, 7: 13, 8: 12, 9: 12, 10: 12}, 40: {N: 15 for N in range(3, 11)}}
    for kcap, want in picks.items():
        for N, wpc in want.items():
            g = geometry(kcap, N=N)
            assert (g["wpc"], g["warp_per_sm"]) == (wpc, wpc), (kcap, N, g)
            assert geometry(kcap, N=N, solver=1)["wpc"] == 10, (kcap, N)


def test_small_shared_memory_is_refused_not_undersized():
    """A device whose SM holds fewer than two of the N > 10 CTAs has no build: hmpc_create returns HMPC_ERR_UNSUPPORTED."""
    small = dict(B200, smem_sm=100 * 1024)
    assert geometry(N=40, limits=small)["unsupported"]
    assert not geometry(N=10, limits=small)["unsupported"]


@pytest.mark.gpu
def test_handles_report_the_predicted_warp_geometry(monkeypatch):
    import torch

    from hopper_mpc_inertial_b200.batch import BatchMpc
    p = torch.cuda.get_device_properties(0)
    limits = dict(sm_count=p.multi_processor_count, smem_block=p.shared_memory_per_block_optin,
                  smem_sm=p.shared_memory_per_multiprocessor, l2=p.L2_cache_size)
    B = 4096
    for kcap, solver, N in itertools.product((56, 40), (0, 1), range(3, 11)):
        monkeypatch.setenv("HMPC_WARP_KCAP", str(kcap))
        info = BatchMpc(B, N=N, device=0, solver=solver).hot_path_info()
        g = geometry(kcap, limits=limits, batch=B, N=N, solver=solver)
        assert (info["warps_per_sm"], info["kcap"], info["regs"]) == (g["warp_per_sm"], g["kcap"], g["regs"]), (kcap, solver, N, info, g)
