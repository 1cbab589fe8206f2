// build.rs -- compiles the sm_100a kernels with nvcc and links them into the dawnsearch binary
// (north_star (1): "a new Rust crate in src/index ... calls CUDA through a thin C-ABI FFI layer built by
// build.rs with nvcc for sm_100a").  Replaces the `usearch` crate's own build.rs (Cargo.lock:3755-3762).
//
// UNCOMPILED IN THIS REPO: the build image has no cargo/rustc.  What IS checked here, on every CPU test run
// (tests/test_rust_shim.py): the source list below equals `SRCS` of dawnsearch_b200/csrc/Makefile, the nvcc
// flags equal the Makefile's `NVCCFLAGS` (minus -Xptxas -v), every `extern "C"` name in gpu_index.rs is
// declared in include/dawn_index.h and exported by the built library, and the link line matches the Makefile's.
use std::{env, path::PathBuf, process::Command};

// keep in sync with SRCS in dawnsearch_b200/csrc/Makefile (enforced by tests/test_rust_shim.py)
const SRCS: &[&str] = &[
    "dawn_index.cu", "scan_topk.cu", "finalize.cu", "ingest.cu", "gemm_topk.cu", "gemm_i8.cu", "i8_tensor.cu",
    "dawn_front.cu", "dawn_multi.cu", "remove.cu",
];
// keep in sync with NVCCFLAGS in dawnsearch_b200/csrc/Makefile.  -ffp-contract=off matters: the host mirrors
// of src/search/vector.rs:181-197 (dawn_front.cu) must not fuse a*b+c, Rust never does.
const NVCCFLAGS: &[&str] = &[
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "-Xcompiler", "-ffp-contract=off",
];

fn main() {
    let out = PathBuf::from(env::var("OUT_DIR").unwrap());
    // DAWN_CSRC lets the dawnsearch workspace vendor the kernels anywhere; default = this repository's layout
    let csrc = PathBuf::from(env::var("DAWN_CSRC").unwrap_or_else(|_| "../dawnsearch_b200/csrc".into()));
    let nvcc = env::var("NVCC").unwrap_or_else(|_| "nvcc".into());
    let mut objs = Vec::new();
    for s in SRCS {
        let obj = out.join(s.replace(".cu", ".o"));
        let ok = Command::new(&nvcc).args(NVCCFLAGS).arg("-c").arg(csrc.join(s)).arg("-o").arg(&obj)
            .status().expect("nvcc not found").success();
        assert!(ok, "nvcc failed on {s}");          // no CPU fallback: a failed CUDA build fails the crate
        println!("cargo:rerun-if-changed={}", csrc.join(s).display());
        objs.push(obj);
    }
    println!("cargo:rerun-if-changed={}", csrc.join("dawn_common.cuh").display());
    println!("cargo:rerun-if-changed={}", csrc.join("../../include/dawn_index.h").display());
    let lib = out.join("libdawn_b200.a");
    let _ = std::fs::remove_file(&lib);
    assert!(Command::new("ar").arg("crs").arg(&lib).args(&objs).status().unwrap().success());
    let cuda = env::var("CUDA_HOME").unwrap_or_else(|_| "/usr/local/cuda".into());
    println!("cargo:rustc-link-search=native={}", out.display());
    println!("cargo:rustc-link-lib=static=dawn_b200");
    println!("cargo:rustc-link-search=native={cuda}/lib64");
    println!("cargo:rustc-link-lib=static=cudart_static");
    // NCCL (dawn_multi.cu: ncclCommInitAll / ncclAllGather) is bound at run time with dlopen("libnccl.so.2"), so that a
    // process which already maps an NCCL keeps using that one; -ldl below is all the link line needs for it.
    println!("cargo:rustc-link-lib=dylib=stdc++");
    println!("cargo:rustc-link-lib=dylib=pthread");
    println!("cargo:rustc-link-lib=dylib=dl");
    println!("cargo:rustc-link-lib=dylib=rt");
}
