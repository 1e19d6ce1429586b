// Compiles the CUDA core for sm_100a with nvcc (the same command line as rs_pathtracing_b200/build.py)
// and links the resulting shared library.  RT_B200_CSRC points at rs_pathtracing_b200/csrc.
use std::{env, path::PathBuf, process::Command};

fn main() {
    let out = PathBuf::from(env::var("OUT_DIR").unwrap());
    let csrc = PathBuf::from(env::var("RT_B200_CSRC").unwrap_or_else(|_| "../../rs_pathtracing_b200/csrc".into()));
    let lib = out.join("librt_b200.so");
    let status = Command::new(env::var("NVCC").unwrap_or_else(|_| "nvcc".into()))
        .args(["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
               "-fmad=false",                       // the parity contract: no a*b+c contraction
               "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math",
               "-diag-suppress", "20014", "-shared", "-cudart", "static", "-o"])
        .arg(&lib)
        .arg(csrc.join("rt_core.cu"))              // C ABI, raygen / extend / shade / resolve / assemble / tonemap
        .arg(csrc.join("rt_march_kernels.cu"))     // k_march_filter, k_march
        .status()
        .expect("nvcc not found");
    assert!(status.success(), "nvcc failed");
    println!("cargo:rustc-link-search=native={}", out.display());
    println!("cargo:rustc-link-lib=dylib=rt_b200");
    println!("cargo:rerun-if-changed={}", csrc.display());
    println!("cargo:rerun-if-env-changed=RT_B200_CSRC");
}
