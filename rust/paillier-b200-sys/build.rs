// Builds the CUDA library from source with the `cc` crate (nvcc, sm_100a only) — what north_star calls the "cc-built .cu" — or,
// with PB200_LIB_DIR set, links a libpaillier_b200.so that was built elsewhere (python -m paillier_halo2_b200.build).
//
// NOT RUN IN THIS REPOSITORY'S BUILD ENVIRONMENT (no Rust toolchain there): the flags below are the ones
// paillier_halo2_b200/build.py uses, which is what the tests and the bench exercise.
use std::env;
use std::path::PathBuf;

fn main() {
    println!("cargo:rerun-if-env-changed=PB200_LIB_DIR");
    if let Ok(dir) = env::var("PB200_LIB_DIR") {
        println!("cargo:rustc-link-search=native={}", dir);
        println!("cargo:rustc-link-lib=dylib=paillier_b200");
        println!("cargo:rustc-link-arg=-Wl,-rpath,{}", dir);
        return;
    }
    let root = PathBuf::from(env::var("CARGO_MANIFEST_DIR").unwrap()).join("../..");
    let csrc = root.join("paillier_halo2_b200/csrc");
    let sources = ["capi.cu", "simple64_kernels.cu", "block28_kernels.cu", "cells.cu", "inverse_kernels.cu"];
    let mut build = cc::Build::new();
    build
        .cuda(true)
        .cudart("shared")
        .flag("-std=c++17")
        .flag("-O3")
        .flag("-lineinfo")
        // sm_100a only: no PTX fallback for other architectures, no multi-backend dispatch
        .flag("-gencode")
        .flag("arch=compute_100a,code=sm_100a")
        .include(root.join("include"));
    for s in sources {
        let p = csrc.join(s);
        println!("cargo:rerun-if-changed={}", p.display());
        build.file(p);
    }
    for h in ["block28.cuh", "simple64.cuh", "engine.hpp", "cells.hpp", "host_bigint.hpp"] {
        println!("cargo:rerun-if-changed={}", csrc.join(h).display());
    }
    println!("cargo:rerun-if-changed={}", root.join("include/paillier_b200.h").display());
    build.compile("paillier_b200");
    println!("cargo:rustc-link-lib=dylib=cudart");
    println!("cargo:rustc-link-lib=dylib=stdc++");
}
