// build.rs of the `bbs_plus` crate with the B200 batch engine: drives nvcc over the CUDA kernel library and links it.
// No CPU fallback and no multi-backend dispatch: without the CUDA toolkit the build fails, without a B200 every batch call
// returns BBS_E_CUDA.
//
// Source layout expected next to Cargo.toml (the north star's "new cuda/ kernel library"):
//     cuda/csrc/*.cu, *.cuh, *.inc     = bbs_sign_b200/csrc of the engine's repository
//     cuda/include/bbs_b200.h          = include/bbs_b200.h
// (`BBS_B200_CUDA_DIR` overrides the directory, e.g. to point at a checkout of the engine.)
// The recipe is the engine's own Makefile: one object per (kernel group, curve) so the compile is parallel.
use std::{env, path::PathBuf, process::Command, thread};

const GROUPS: [&str; 10] = ["ctx", "h2s", "verify", "pairing", "sign", "signitem", "proof", "proofitem", "rlc", "selftest"];

fn nvcc(args: &[String]) {
    let nvcc = env::var("NVCC").unwrap_or_else(|_| "nvcc".into());
    let status = Command::new(&nvcc)
        .args(args)
        .status()
        .unwrap_or_else(|e| panic!("{nvcc} not found ({e}): the bbs_plus batch API needs the CUDA toolkit (>= 12.8, sm_100a)"));
    assert!(status.success(), "nvcc failed: {args:?}");
}

fn main() {
    let out = PathBuf::from(env::var("OUT_DIR").unwrap());
    let root = env::var("BBS_B200_CUDA_DIR")
        .map(PathBuf::from)
        .unwrap_or_else(|_| PathBuf::from(env::var("CARGO_MANIFEST_DIR").unwrap()).join("cuda"));
    let src = root.join("csrc");
    let inc = root.join("include");
    assert!(src.join("capi.cu").exists(), "CUDA sources not found under {}", src.display());
    let common: Vec<String> = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC"]
        .iter().map(|s| s.to_string()).chain([format!("-I{}", inc.display())]).collect();

    // (source, extra define, object)
    let mut jobs: Vec<(PathBuf, Option<&'static str>, PathBuf)> = vec![(src.join("capi.cu"), None, out.join("capi.o"))];
    for g in GROUPS {
        jobs.push((src.join(format!("tu_{g}.cu")), Some("-DBBS_TU_BLS"), out.join(format!("tu_{g}_bls.o"))));
        jobs.push((src.join(format!("tu_{g}.cu")), Some("-DBBS_TU_BN"), out.join(format!("tu_{g}_bn.o"))));
    }
    let handles: Vec<_> = jobs.iter().cloned().map(|(cu, def, obj)| {
        let mut args = common.clone();
        if let Some(d) = def { args.push(d.to_string()); }
        args.extend(["-c".to_string(), "-o".to_string(), obj.display().to_string(), cu.display().to_string()]);
        thread::spawn(move || nvcc(&args))
    }).collect();
    for h in handles { h.join().expect("nvcc job panicked"); }

    let lib = out.join("libbbs_b200.so");
    let mut link: Vec<String> = vec!["-gencode".into(), "arch=compute_100a,code=sm_100a".into(), "-shared".into(),
                                     "-o".into(), lib.display().to_string()];
    link.extend(jobs.iter().map(|(_, _, o)| o.display().to_string()));
    nvcc(&link);

    println!("cargo:rustc-link-search=native={}", out.display());
    println!("cargo:rustc-link-lib=dylib=bbs_b200");
    println!("cargo:rustc-link-lib=dylib=cudart");
    println!("cargo:rerun-if-changed={}", root.display());
    println!("cargo:rerun-if-env-changed=BBS_B200_CUDA_DIR");
    println!("cargo:rerun-if-env-changed=NVCC");
}
