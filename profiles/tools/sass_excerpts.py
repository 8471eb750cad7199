#!/usr/bin/env python3
"""Writes profiles/r2_sass_<kernel>.txt: excerpts of the shipped library's SASS (cuobjdump -sass libfp8_b200.so) around
the instructions that prove what each hot kernel is made of -- the tcgen05 MMA loop (UTCQMMA), TMA loads / stores
(UTMALDG / UTMASTG), tensor-memory loads (LDTM), bulk copies (UBLKCP), the cast inner loops (F2FP), the GEMV's warp MMAs.
Runs here (no GPU needed):   python profiles/tools/sass_excerpts.py"""
import os, re, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
LIB = os.path.join(ROOT, "fp8-mps-metal_b200", "libfp8_b200.so")
OUT = os.path.join(ROOT, "profiles")

# (output name, regex on the demangled function name, [mnemonic regexes to excerpt around], context lines)
KERNELS = [
    ("gemm_tcgen05_256x256_pair", r"fp8_gemm_tcgen05_kernel<256, 2, 0>", [r"UTCQMMA", r"UTMALDG", r"LDTM", r"UTCBAR", r"STG\.E\.128"], 6),
    ("gemm_tcgen05_push_256x256_pair", r"fp8_gemm_tcgen05_kernel<256, 2, 2>", [r"UTMASTG", r"UTCQMMA", r"LDTM", r"STS\.128", r"UTMACMDFLUSH|DEPBAR|UTMACCTL"], 6),
    ("gemm_splitk_x4", r"fp8_gemm_splitk_kernel<4>", [r"UTCQMMA", r"UBLKCP|UBLKRED|UBLK", r"LDTM", r"UCGABAR", r"MAPA|UMAPA"], 5),
    ("gemv_fhfma_m1", r"fp8_gemv_kernel<1, 4>", [r"FHFMA", r"LDG\.E\.128", r"ACQBULK|GRIDDEP"], 5),
    ("dequant_ldg_f16", r"fp8_to_wide_kernel<1, false, 512, 8, 0>", [r"F2FP", r"LDG", r"STG"], 4),
    ("encode_bf16", r"wide_to_fp8_kernel<2, false, 512, 4, 32>", [r"F2FP", r"LDG\.E\.(ENL2\.)?256|LDG", r"STG"], 4),
]


def main():
    sass = subprocess.run(["cuobjdump", "-sass", LIB], stdout=subprocess.PIPE, text=True, check=True).stdout
    blocks = re.split(r"\n\s*Function : ", sass)
    names = [b.split("\n", 1)[0].strip() for b in blocks[1:]]
    dem = subprocess.run(["c++filt"] + names, stdout=subprocess.PIPE, text=True).stdout.splitlines()
    for out_name, fn_re, pats, ctx in KERNELS:
        hit = [i for i, d in enumerate(dem) if re.search(fn_re, d)]
        if not hit:
            print("not found:", fn_re)
            continue
        i = hit[0]
        lines = [l for l in blocks[i + 1].split("\n") if re.search(r"/\*[0-9a-f]{4}\*/", l)]
        code = [re.sub(r"\s*/\* 0x[0-9a-f]+ \*/\s*$", "", l).rstrip() for l in lines]
        counts = {}
        for l in code:
            m = re.search(r"\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", l)
            if m:
                op = m.group(1).split(".")[0]
                counts[op] = counts.get(op, 0) + 1
        with open(os.path.join(OUT, f"r2_sass_{out_name}.txt"), "w") as f:
            f.write(f"# {dem[i]}\n# {len(code)} SASS instructions; from `cuobjdump -sass fp8-mps-metal_b200/libfp8_b200.so` (sm_100a)\n")
            f.write("# opcode histogram (top 24): " + ", ".join(f"{k} {v}" for k, v in sorted(counts.items(), key=lambda kv: -kv[1])[:24]) + "\n")
            for pat in pats:
                idx = [k for k, l in enumerate(code) if re.search(pat, l)]
                f.write(f"\n## {pat}: {len(idx)} instruction(s)\n")
                shown = -1
                n_ex = 0
                for k in idx:
                    if k <= shown:
                        continue
                    lo, hi = max(0, k - ctx), min(len(code), k + ctx + 1)
                    f.write("\n".join(code[lo:hi]) + "\n   ...\n")
                    shown = hi
                    n_ex += 1
                    if n_ex >= 2:
                        break
        print("wrote", f"profiles/r2_sass_{out_name}.txt", dem[i][:90])


if __name__ == "__main__":
    main()
