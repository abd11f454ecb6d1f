"""CPU: every kernel instantiation in genpc_b200/libgenpc_b200.so has an entry in KERNELS, and every entry names a kernel that
still exists.  An entry says why the instantiation is trusted:

- "tests/<file>.py::<test>": a test that runs it and compares its result with the oracle (or, for an internal stage, the
  result of the call it belongs to);
- "helper": cub and set-up kernels whose output is checked only through the call that uses them;
- "not compared: <why>": a kernel that no test compares yet (a known gap, stated).

A new kernel, template instantiation or threshold therefore has to be placed here.  tools/kernel_coverage.py runs the GPU
suite under torch.profiler and lists the instantiations that no test launched, to keep the table honest."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "genpc_b200", "libgenpc_b200.so")
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"


def kernel_key(name):
    """Demangled kernel name (cu++filt's or the profiler's spelling) -> 'ns::kernel<args>' without casts, spaces, return type
    or parameter list; cub kernels lose their versioned namespace and template arguments."""
    s = re.sub(r"\(bool\)0", "false", name)
    s = re.sub(r"\(bool\)1", "true", s)
    s = re.sub(r"\((?:unsigned )?(?:int|long|char|short)\)", "", s)
    s = s.replace(" ", "")
    s = re.sub(r"^void(?=\w*::)", "", s)
    depth = 0
    for i, ch in enumerate(s):
        if ch == "<":
            depth += 1
        elif ch == ">":
            depth -= 1
        elif ch == "(" and depth == 0:
            s = s[:i]
            break
    if s.startswith("cub::"):
        s = re.sub(r"<.*", "", re.sub(r"CUB_\w+::", "", s))
    return s


def library_kernels(lib=LIB):
    """Keys of every kernel in the library's SASS (cuobjdump -sass, names demangled by cu++filt)."""
    out = subprocess.run([CUOBJDUMP, "-sass", lib], capture_output=True, text=True, check=True).stdout
    mangled = sorted(set(re.findall(r"Function : (\S+)", out)))
    filt = os.path.join(os.path.dirname(CUOBJDUMP), "cu++filt")
    filt = filt if os.path.exists(filt) else (shutil.which("cu++filt") or "c++filt")
    dem = subprocess.run([filt], input="\n".join(mangled) + "\n", capture_output=True, text=True, check=True).stdout.split("\n")
    return {kernel_key(d) for d in dem[:len(mangled)]}


CG = "tests/test_chamfer_gpu.py::"
PRU = "tests/test_chamfer_prune.py::"
LARGE = "tests/test_chamfer_large_clouds.py::"
HF = "tests/test_chamfer_host_feed.py::"
FPS = "tests/test_fps.py::"
EMD = "tests/test_emd.py::"
REG = "tests/test_registration.py::"
DSP = "tests/test_dispatch_paths.py::"
DEPTH = "tests/test_depth.py::test_depth_gpu_bit_exact"
GRID = PRU + "test_grid_scan_bit_exact"
NOT_COMPARED = "not compared: "

KERNELS = {
    # cub's radix sort inside the grid scan (nn_grid.cuh); its order is checked through the scan's results
    "cub::EmptyKernel": "helper",
    "cub::DeviceRadixSortExclusiveSumKernel": "helper",
    "cub::DeviceRadixSortHistogramKernel": "helper",
    "cub::DeviceRadixSortOnesweepKernel": "helper",
    "cub::DeviceRadixSortSingleTileKernel": "helper",
    # Chamfer: exhaustive, symmetric, pruned and grid scans, epilogue, gradients
    "genpc::nn_scan_kernel<1>": CG + "test_backward_vs_oracle",
    "genpc::nn_scan_kernel<2>": DSP + "test_partial_scan_two_queries_per_thread_merges_to_the_oracle",
    "genpc::nn_scan_kernel<4>": "tests/test_sharded.py::test_partial_scans_merge_to_the_single_gpu_result",
    "genpc::nn_unpack_kernel": CG + "test_backward_vs_oracle",
    "genpc::nn_sym_kernel<2>": DSP + "test_chamfer_sym_kernel_two_rows_per_thread_vs_oracle",
    "genpc::nn_sym_kernel<4>": "tests/test_c1_scan.py::test_c1_on_gpu_vs_oracle_and_golden",
    "genpc::nn_sym_balanced_kernel<2>": CG + "test_forward_bit_exact_vs_oracle",
    "genpc::nn_sym_balanced_kernel<4>": CG + "test_forward_bit_exact_vs_oracle",
    "genpc::nn_sym_gated_kernel<2>": DSP + "test_host_fed_forward_two_rows_per_thread_vs_oracle",
    "genpc::nn_sym_gated_kernel<4>": HF + "test_host_fed_forward_bit_exact",
    "genpc::nn_sym_epilogue_kernel<false>": CG + "test_nan_and_inf_points_stay_in_range",
    "genpc::nn_sym_epilogue_kernel<true>": "tests/test_c1_scan.py::test_c1_on_gpu_vs_oracle_and_golden",
    "genpc::nn_bin_sort_kernel<1>": PRU + "test_exact_ties_and_degenerate_geometry",
    "genpc::nn_bin_sort_kernel<2>": PRU + "test_sort_cluster_layouts_bit_exact",
    "genpc::nn_bin_sort_kernel<3>": PRU + "test_sort_cluster_layouts_bit_exact",
    "genpc::nn_bin_sort_kernel<4>": PRU + "test_sort_cluster_layouts_bit_exact",
    "genpc::nn_bin_sort_kernel<8>": PRU + "test_sort_cluster_layouts_bit_exact",
    "genpc::nn_prune_kernel<1>": CG + "test_full_c2_bit_exact_vs_oracle_and_reference",
    "genpc::nn_prune_kernel<2>": PRU + "test_exact_ties_and_degenerate_geometry",
    "genpc::nn_prune_kernel<4>": DSP + "test_registration_c3_pruned_sym_finish512_vs_oracle",
    "genpc::nn_prune_kernel<8>": PRU + "test_pruned_scan_bit_exact_on_awkward_shapes",
    "genpc::nn_prune_kernel<16>": DSP + "test_registration_pruned_clouds_above_16384_points_vs_oracle",
    "genpc::nn_prune_coop_kernel<1>": PRU + "test_pruned_scan_bit_exact_on_awkward_shapes",
    "genpc::nn_prune_coop_kernel<2>": PRU + "test_sort_cluster_layouts_bit_exact",
    "genpc::nn_prune_coop_kernel<4>": PRU + "test_fused_loss_step_with_the_pruned_scan",
    "genpc::nn_prune_coop_kernel<8>": CG + "test_full_c2_bit_exact_vs_oracle_and_reference",
    "genpc::nn_prune_coop_kernel<16>": PRU + "test_pruned_scan_bit_exact_on_awkward_shapes",
    "genpc::prune_rearm_kernel": HF + "test_host_fed_forward_bit_exact",
    "genpc::grid_init_kernel": GRID,
    "genpc::grid_bbox_kernel": GRID,
    "genpc::grid_key_kernel": GRID,
    "genpc::grid_gather_kernel": GRID,
    "genpc::grid_boxes_kernel<false>": GRID,
    "genpc::grid_boxes_kernel<true>": GRID,
    "genpc::grid_decide_kernel": PRU + "test_large_clouds_take_the_grid_scan_by_default",
    "genpc::nn_prune2_kernel<1,false>": GRID,
    "genpc::nn_prune2_kernel<1,true>": PRU + "test_probe_hands_non_overlapping_large_clouds_to_the_exhaustive_kernels",
    "genpc::nn_prune2_kernel<2,false>": PRU + "test_large_clouds_take_the_grid_scan_by_default",
    "genpc::nn_prune2_kernel<2,true>": PRU + "test_large_clouds_take_the_grid_scan_by_default",
    "genpc::nn_prune2_kernel<4,false>": PRU + "test_large_clouds_take_the_grid_scan_by_default",
    "genpc::nn_prune2_kernel<4,true>": PRU + "test_large_clouds_take_the_grid_scan_by_default",
    "genpc::nn_prune2_kernel<8,false>": LARGE + "test_c5_full_size_default_path",
    "genpc::nn_prune2_kernel<8,true>": LARGE + "test_c5_full_size_default_path",
    "genpc::nn_prune2_kernel<16,false>": LARGE + "test_grid_scan_superblock_register_edges",
    "genpc::nn_prune2_kernel<16,true>": LARGE + "test_grid_scan_superblock_register_edges",
    "genpc::chamfer_grad_kernel<false,false>": CG + "test_unaligned_pointers_take_the_scalar_paths",
    "genpc::chamfer_grad_kernel<false,true>": DSP + "test_fused_loss_backward_with_unaligned_gradient_arrays",
    "genpc::chamfer_grad_kernel<true,false>": CG + "test_backward_vs_oracle",
    "genpc::chamfer_grad_kernel<true,true>": CG + "test_fused_forward_c_abi",
    "genpc::chamfer_loss_kernel": CG + "test_fused_forward_c_abi",
    # EMD
    "genpc::emd_auction_kernel<0,5>": EMD + "test_emd_gpu_bit_exact_vs_oracle",
    "genpc::emd_auction_kernel<4,3>": EMD + "test_emd_gpu_bit_exact_vs_oracle",
    "genpc::emd_auction_kernel<8,3>": EMD + "test_emd_gpu_bit_exact_vs_oracle",
    "genpc::emd_auction_kernel<16,3>": EMD + "test_emd_pruned_bid_equals_exhaustive_bid_on_adversarial_inputs",
    "genpc::emd_sort_kernel": EMD + "test_emd_pruned_bid_equals_exhaustive_bid_on_adversarial_inputs",
    "genpc::emd_grad_kernel": DSP + "test_emd_batch_512_more_clouds_than_ctas",
    # FPS
    "genpc::fps_reg_kernel<1,true>": FPS + "test_fps_gpu_bit_exact",
    "genpc::fps_reg_kernel<2,true>": FPS + "test_fps_gpu_bit_exact",
    "genpc::fps_reg_kernel<4,true>": FPS + "test_fps_gpu_ties_and_api",
    "genpc::fps_reg_kernel<8,false>": FPS + "test_fps_single_cta_shared_memory_and_l1_forms",
    "genpc::fps_reg_kernel<16,false>": FPS + "test_fps_single_cta_shared_memory_and_l1_forms",
    "genpc::fps_reg_kernel<32,false>": DSP + "test_fps_batches_beyond_the_clusters",
    "genpc::fps_smem_kernel<8>": FPS + "test_fps_single_cta_shared_memory_and_l1_forms",
    "genpc::fps_smem_kernel<16>": FPS + "test_fps_single_cta_shared_memory_and_l1_forms",
    "genpc::fps_gmem_kernel": DSP + "test_fps_fusion_size_gmem_kernel_vs_oracle_and_float64",
    "genpc::fps_cluster_kernel<1,8,false>": FPS + "test_fps_cluster_kernel_bit_exact",
    "genpc::fps_cluster_kernel<2,8,false>": FPS + "test_fps_cluster_kernel_bit_exact",
    "genpc::fps_cluster_kernel<4,8,false>": FPS + "test_fps_cluster_kernel_bit_exact",
    "genpc::fps_cluster_kernel<8,8,true>": FPS + "test_fps_cluster_kernel_bit_exact",
    "genpc::fps_cluster_kernel<12,8,true>": FPS + "test_fps_cluster_kernel_bit_exact",
    "genpc::fps_cluster_kernel<18,8,true>": FPS + "test_fps_cluster_kernel_bit_exact",
    "genpc::fps_cluster_kernel<1,16,false>": FPS + "test_fps_cluster_kernel_bit_exact",
    "genpc::fps_cluster_kernel<2,16,false>": FPS + "test_fps_cluster_kernel_bit_exact",
    "genpc::fps_cluster_kernel<4,16,false>": DSP + "test_fps_both_sides_of_the_cluster_limit",
    "genpc::fps_cluster_kernel<6,16,false>": FPS + "test_fps_cluster_kernel_bit_exact",
    "genpc::fps_cluster_kernel<9,16,false>": FPS + "test_fps_cluster_kernel_bit_exact",
    # registration
    "genpc::register_step_kernel<1>": REG + "test_step_loss_and_gradient_vs_oracle",
    "genpc::register_step_kernel<2>": DSP + "test_registration_small_problem_kernels_vs_oracle",
    "genpc::register_step_kernel<4>": DSP + "test_registration_small_problem_kernels_vs_oracle",
    "genpc::register_persistent_kernel<1,256>": DSP + "test_registration_small_problem_kernels_vs_oracle",
    "genpc::register_persistent_kernel<1,512>": REG + "test_persistent_small_registration_equals_launch_per_iteration",
    "genpc::register_persistent_kernel<1,1024>": REG + "test_trajectory_vs_oracle",
    "genpc::register_persistent_kernel<2,1024>": DSP + "test_registration_small_problem_kernels_vs_oracle",
    "genpc::register_persistent_kernel<4,1024>": DSP + "test_registration_small_problem_kernels_vs_oracle",
    "genpc::register_sym_scan_kernel<2>": DSP + "test_registration_sym_scan_two_rows_per_thread_vs_oracle",
    "genpc::register_sym_scan_kernel<4>": DSP + "test_registration_c3_pruned_sym_finish512_vs_oracle",
    "genpc::register_finish_kernel<128>": DSP + "test_registration_single_cloud_four_starts_finish128_vs_oracle",
    "genpc::register_finish_kernel<256>": DSP + "test_registration_8_scans_exhaustive_sym_finish256_vs_oracle",
    "genpc::register_finish_kernel<512>": DSP + "test_registration_c3_pruned_sym_finish512_vs_oracle",
    "genpc::register_sims_kernel": DSP + "test_registration_c3_pruned_sym_finish512_vs_oracle",
    "genpc::icp_step_kernel": "tests/test_reg_xyz.py::test_icp_step_kernel_matches_the_torch_formulation",
    "genpc::knn_mean_kernel<1>": DSP + "test_knn_mean_distance_every_list_size",
    # mesh sampling, depth rendering
    "genpc::mesh_face_area_kernel": "tests/test_mesh_glb.py::test_sampler_kernel_bit_exact_vs_oracle",
    "genpc::mesh_sample_kernel": "tests/test_mesh_glb.py::test_sampler_kernel_bit_exact_vs_oracle",
    "genpc::project_kernel": DEPTH,
    "genpc::uv_kernel": DEPTH,
    "genpc::zsplat_kernel": DEPTH,
    "genpc::zresolve_kernel": DEPTH,
    "genpc::unproject_kernel": DEPTH,
}
KERNELS.update({f"genpc::knn_mean_kernel<{k}>": DSP + "test_knn_mean_distance_every_list_size" for k in range(2, 33)})


@pytest.fixture(scope="module")
def kernels():
    if not os.path.exists(CUOBJDUMP):
        pytest.skip("cuobjdump not available")
    if not os.path.exists(LIB):
        from genpc_b200.csrc import build

        build.build()
    return library_kernels()


def test_kernel_key_reads_both_spellings():
    assert kernel_key("void genpc::fps_reg_kernel<(int)32, (bool)0>(const float *, int, int, int, int *, float *)") == \
        "genpc::fps_reg_kernel<32,false>"
    assert kernel_key("void genpc::fps_reg_kernel<32, false>(float const*, int, int, int, int*, float*)") == \
        "genpc::fps_reg_kernel<32,false>"
    assert kernel_key("genpc::register_sims_kernel(genpc::RegArgs, genpc::Similarity *)") == "genpc::register_sims_kernel"
    assert kernel_key("void cub::CUB_200802_SM_1000::EmptyKernel<void>()") == "cub::EmptyKernel"


def test_every_kernel_has_an_entry_and_every_entry_a_kernel(kernels):
    missing = sorted(kernels - set(KERNELS))
    stale = sorted(set(KERNELS) - kernels)
    assert not missing, f"kernels without an entry in KERNELS: {missing}"
    assert not stale, f"entries in KERNELS whose kernel no longer exists: {stale}"


def test_entries_name_existing_tests_or_a_reason():
    for k, v in KERNELS.items():
        if v == "helper" or v.startswith(NOT_COMPARED):
            continue
        path, _, name = v.partition("::")
        assert path.startswith("tests/") and name, (k, v)
        with open(os.path.join(ROOT, path)) as f:
            assert re.search(r"^def " + re.escape(name) + r"\(", f.read(), re.M), (k, v)
