// build.rs -- builds librm_b200.so from the vendored sources (engine/rm_b200/ = this repository's
// `include/` and `rusty_marcher_b200/csrc/`) with nvcc for sm_100a and links the crate against it.
// Needs CUDA >= 12.8 (nvcc that knows compute_100a).  Set NVCC to override the compiler.
use std::{env, path::PathBuf, process::Command};

fn main() {
    let out = PathBuf::from(env::var("OUT_DIR").unwrap());
    let src = PathBuf::from("rm_b200/rusty_marcher_b200/csrc");
    let lib = out.join("librm_b200.so");
    let status = Command::new(env::var("NVCC").unwrap_or_else(|_| "nvcc".into()))
        .args(&[
            "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
            "-fmad=false", // FP32 FMAs are explicit in the kernels; the f64 validation kernels must never fuse
            "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math", "-shared", "-o",
        ])
        .arg(&lib)
        .args(
            ["rm_api.cu", "rm_kernels.cu", "rm_lens.cu", "rm_area.cu", "rm_rough.cu", "rm_motion.cu", "rm_distributed.cu", "rm_indirect.cu", "rm_path.cu", "rm_scene.cpp", "rm_bvh.cpp", "rm_host.cpp"]
                .iter()
                .map(|f| src.join(f)),
        )
        .status()
        .expect("nvcc not found: the render path has no CPU fallback");
    assert!(status.success(), "nvcc failed building librm_b200.so");
    println!("cargo:rustc-link-search=native={}", out.display());
    println!("cargo:rustc-link-lib=dylib=rm_b200");
    println!("cargo:rustc-env=LD_RUN_PATH={}", out.display());
    println!("cargo:rerun-if-changed=rm_b200");
}
