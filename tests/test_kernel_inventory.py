"""CPU test: every kernel the library launches (every post_launch name in kokorox_b200/csrc/*.cu) is either checked by
an op-level test against a reference, or carries a written exemption.  A new kernel cannot land without one of the two,
and a mapped test that is renamed or removed fails here."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "kokorox_b200", "csrc")

OPS = "tests/test_ops_gpu.py"
SIG = "tests/test_signal_ops_gpu.py"

# kernel name -> op-level tests ("file::test") that compare it with a reference
TESTED = {
    "conv_f32": [f"{OPS}::test_conv1d_matches_torch", f"{OPS}::test_conv_prologue_epilogue_fusions"],
    "conv_tc": [f"{OPS}::test_tc_conv_matches_torch_on_bf16_operands", f"{OPS}::test_tc_conv_transpose_phases"],
    "conv_tc_tf32x3": [f"{OPS}::test_split_tf32_gemm_is_fp32_grade", f"{OPS}::test_split_fp16_gemm_is_fp32_grade"],
    "apply_bf16": [f"{OPS}::test_tc_conv_matches_torch_on_bf16_operands", f"{OPS}::test_tc_conv_fused_prologue_epilogue"],
    "apply_tf32": [f"{OPS}::test_split_tf32_gemm_is_fp32_grade"],
    "apply_f16x2": [f"{OPS}::test_split_fp16_gemm_is_fp32_grade"],
    "im2col_bf16": [f"{OPS}::test_im2col_fast_kernel_is_bit_identical"],
    "arb_conv": [f"{OPS}::test_fused_arb_conv", f"{OPS}::test_fused_arb_conv_bf16_residual_stream"],
    "post_conv": [f"{SIG}::test_post_conv_matches_float64_reference"],
    "attention": [f"{OPS}::test_attention_matches_torch", f"{OPS}::test_attention_tcgen05_matches_torch_and_mma_sync"],
    "attn_prep": [f"{OPS}::test_attention_tcgen05_matches_torch_and_mma_sync"],
    "lstm": [f"{OPS}::test_lstm_matches_torch", f"{OPS}::test_lstm_ragged_batch_groups"],
    "layernorm": [f"{OPS}::test_layernorm_kernels"],
    "colstats": [f"{OPS}::test_instance_norm_adain_coefficients", f"{OPS}::test_pointwise_conv_with_statistics"],
    "adain_coef": [f"{OPS}::test_instance_norm_adain_coefficients"],
    "pointwise_conv_stats": [f"{OPS}::test_pointwise_conv_with_statistics"],
    "add_rows_stats": [f"{SIG}::test_add_rows_stats"],
    "pool_up": [f"{SIG}::test_pool_up_kernels"],
    "pool_up_bf16": [f"{SIG}::test_pool_up_kernels"],
    "duration": [f"{SIG}::test_durations_ties_and_specials", f"{SIG}::test_durations_speeds_and_cap"],
    "dur_scan": [f"{SIG}::test_length_regulator_exact"],
    "expand_idx": [f"{SIG}::test_length_regulator_exact"],
    "gather_rows": [f"{SIG}::test_length_regulator_exact", f"{SIG}::test_durations_ties_and_specials"],
    "curve_conv": [f"{SIG}::test_curve_conv_matches_float64"],
    "sine_phase": [f"{SIG}::test_sine_source_matches_oracle", f"{SIG}::test_sine_source_ragged_batch"],
    "sine_source": [f"{SIG}::test_sine_source_matches_oracle", f"{SIG}::test_sin_reduced_bound_at_large_phases",
                    f"{SIG}::test_production_noise_is_standard_normal", f"{SIG}::test_production_noise_is_uncorrelated",
                    f"{SIG}::test_production_noise_is_keyed_by_sample_not_batch_slot"],
    "stft": [f"{SIG}::test_stft_matches_float64"],
    "istft": [f"{SIG}::test_istft_matches_float64", f"{SIG}::test_istft_pcm16_twin"],
    "resample": ["tests/test_resample_gpu.py::test_resample_kernel_matches_resample_poly"],
    "loud_energy": ["tests/test_loudness_gpu.py::test_kernels_match_reference"],
    "loud_peak": ["tests/test_loudness_gpu.py::test_kernels_match_reference", "tests/test_limiter_gpu.py::test_kernels_match_reference"],
    "loud_gain": ["tests/test_loudness_gpu.py::test_kernels_match_reference"],
    "lim_envelope": ["tests/test_limiter_gpu.py::test_kernels_match_reference"],
    "lim_trim": ["tests/test_limiter_gpu.py::test_kernels_match_reference"],
    "loud_short": ["tests/test_loudness_range_gpu.py::test_kernels_match_reference"],
    "loud_range": ["tests/test_loudness_range_gpu.py::test_kernels_match_reference"],
    "flac_analyze": ["tests/test_flac_gpu.py::test_kernel_matches_reference_encoder"],
    "flac_scan": ["tests/test_flac_gpu.py::test_kernel_matches_reference_encoder"],
    "flac_pack": ["tests/test_flac_gpu.py::test_kernel_matches_reference_encoder"],
    "mp3_encode": ["tests/test_mp3_gpu.py::test_kernel_matches_the_reference_encoder"],
}

# kernel name -> why it has no op-level test
EXEMPT = {
    "copy_row": "plain row copy (the reflection pad of the second up-sampling); a wrong row is gross at model level",
    "copy_cols": "plain column copy between activation tensors; any error is gross at model level",
    "bcast_cols": "plain broadcast of a per-item vector over the item's rows; any error is gross at model level",
    "embed_rows": "plain table row gather; any error is gross at model level",
    "add_rows": "elementwise fp32 a + b of the fp32 configuration (add_rows_stats is its tested twin); gross at model level",
    "albert_embed": "three table rows summed and a LayerNorm; compared with the oracle's `bert` stage in "
                    "tests/test_parity_gpu.py::test_stagewise_parity_teacher_forced",
    "mix_styles": "voice-table mix, bit-identical to the host mix in tests/test_parity_gpu.py::test_device_voice_table_and_mix_styles",
}


def launched_names():
    """Every kernel name passed to post_launch: string literals, and the prefix before '[' of names formatted into a
    buffer (snprintf(nm, ..., "arb_conv[c%d ...]") then post_launch(nm, ...))."""
    names = {}
    for f in sorted(os.listdir(CSRC)):
        if not f.endswith(".cu"):
            continue
        src = open(os.path.join(CSRC, f)).read()
        for m in re.finditer(r'post_launch\(\s*"([^"]+)"', src):
            names.setdefault(m.group(1), f)
        for m in re.finditer(r'post_launch\(\s*(\w+)\s*,', src):
            var = m.group(1)
            for fm in re.finditer(r'snprintf\(\s*' + re.escape(var) + r'\s*,[^,]+,\s*"([^"\[%]+)', src):
                names.setdefault(fm.group(1).strip(), f)
    return names


def test_kernel_names_are_found():
    names = launched_names()
    assert {"arb_conv", "conv_f32", "conv_tc", "conv_tc_tf32x3", "istft", "sine_source", "mp3_encode"} <= set(names)
    assert not any("[" in n or "%" in n for n in names)


def test_every_launched_kernel_is_tested_or_exempt():
    names = launched_names()
    unmapped = sorted(n for n in names if n not in TESTED and n not in EXEMPT)
    assert not unmapped, f"kernels without an op-level test or a written exemption: {unmapped} ({[names[n] for n in unmapped]})"
    assert not set(TESTED) & set(EXEMPT)
    stale = sorted(set(TESTED) - set(names)) + sorted(set(EXEMPT) - set(names))
    assert not stale, f"mapped names no kernel launches any more: {stale}"


def test_mapped_tests_exist():
    missing = []
    for tests in TESTED.values():
        for t in tests:
            path, name = t.split("::")
            src = open(os.path.join(ROOT, path)).read()
            if not re.search(r"^def " + re.escape(name) + r"\(", src, re.M):
                missing.append(t)
    for why in EXEMPT.values():
        for t in re.findall(r"(tests/\w+\.py)::(\w+)", why):
            src = open(os.path.join(ROOT, t[0])).read()
            if not re.search(r"^def " + re.escape(t[1]) + r"\(", src, re.M):
                missing.append("::".join(t))
    assert not missing, f"mapped tests that do not exist: {missing}"
