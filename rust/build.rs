//! Compiles the CUDA sources of the path with nvcc for sm_100a and links them into the crate.
//! No Triton, no multi-backend dispatch, no CPU fallback: without nvcc the build fails.
use std::{env, path::PathBuf, process::Command};

const SOURCES: [&str; 10] = ["ndi_api.cu", "ndi_eval.cu", "ndi_bin.cu", "ndi_sweep.cu", "ndi_grid.cu", "ndi_spline.cu", "ndi_rowsplit.cu", "ndi_partition.cu", "ndi_integral.cu", "ndi_hermite.cu"];

fn main() {
    let out = PathBuf::from(env::var("OUT_DIR").unwrap());
    let csrc = PathBuf::from(env::var("CARGO_MANIFEST_DIR").unwrap()).join("../ndarray_interp_b200/csrc");
    let nvcc = env::var("NVCC").unwrap_or_else(|_| "nvcc".into());
    let mut objects = Vec::new();
    for src in SOURCES {
        let obj = out.join(src.replace(".cu", ".o"));
        let status = Command::new(&nvcc)
            .args(["-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo"])
            // parity: no FMA contraction, IEEE division, denormals kept (the defaults of the last three)
            .args(["-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false"])
            .args(["-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-c"])
            .arg(csrc.join(src))
            .arg("-o")
            .arg(&obj)
            .status()
            .expect("nvcc not found: this crate has no CPU fallback");
        assert!(status.success(), "nvcc failed on {src}");
        println!("cargo:rerun-if-changed={}", csrc.join(src).display());
        objects.push(obj);
    }
    let lib = out.join("libndi_b200.a");
    let status = Command::new("ar").arg("crs").arg(&lib).args(&objects).status().expect("ar");
    assert!(status.success());
    println!("cargo:rustc-link-search=native={}", out.display());
    println!("cargo:rustc-link-lib=static=ndi_b200");
    let cuda = env::var("CUDA_HOME").unwrap_or_else(|_| "/usr/local/cuda".into());
    println!("cargo:rustc-link-search=native={cuda}/lib64");
    println!("cargo:rustc-link-lib=dylib=cudart");
    println!("cargo:rustc-link-lib=dylib=stdc++");
    for h in ["ndi_device.cuh", "ndi_spline.cuh", "ndi_internal.h"] {
        println!("cargo:rerun-if-changed={}", csrc.join(h).display());
    }
}
