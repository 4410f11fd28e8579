"""cuobjdump -sass excerpts of the hot kernels of the built library -> profiles/r<round>_sass_*.txt (runs without a GPU).

    python scripts/sass_listings.py [SUBSTRING]    (only the listings whose tag contains SUBSTRING)"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROF = os.path.join(ROOT, "profiles")
so = os.path.join(ROOT, "colosseum_b200", "_lib", "libcolosseum_b200.so")
syms = subprocess.run(["cuobjdump", "-elf", so], capture_output=True, text=True).stdout
for tag, pat in (("backup_kernel_f32_max_vec_warp", r"_ZN4colo13backup_kernelIfLi0ELb1ELb0EEEv\w+?(?=_param|\s|$)"),
                 ("backup_tma_kernel_max_8", r"_ZN4colo17backup_tma_kernelILi0ELi8EEEv\w+?(?=_param|\s|$)"),
                 ("gs_solve_tma_kernel_f32", r"_ZN4colo19gs_solve_tma_kernelIfEEv\w+?(?=_param|\s|$)"),
                 ("env_step_kary_lean_kernel_4", r"_ZN4colo25env_step_kary_lean_kernelILi4ELb0EEEv\w+?(?=_param|\s|$)"),
                 ("env_step_kary_lean_kernel_4_compact", r"_ZN4colo25env_step_kary_lean_kernelILi4ELb1EEEv\w+?(?=_param|\s|$)"),
                 ("hitting_umma_kernel_128", r"_ZN4colo19hitting_umma_kernelILi128ELb0EEEv\w+?(?=_param|\s|$)"),
                 ("hitting_umma_kernel_128_multicast", r"_ZN4colo19hitting_umma_kernelILi128ELb1EEEv\w+?(?=_param|\s|$)"),
                 ("env_step_breaks_lean_kernel_2", r"_ZN4colo27env_step_breaks_lean_kernelILi2ELb0EEEv\w+?(?=_param|\s|$)"),
                 ("env_step_dense_kary_kernel_breaks_2",
                  r"_ZN4colo26env_step_dense_kary_kernelIfLi1ELb0ELi2EEEv\w+?(?=_param|\s|$)")):
    if len(sys.argv) > 1 and sys.argv[1] not in tag:
        continue
    rnd = "r3" if "breaks" in tag else "r2"
    m = re.search(pat, syms)
    if not m:
        print("symbol not found:", tag)
        continue
    sass = subprocess.run(["cuobjdump", "-sass", "-fun", m.group(0), so], capture_output=True, text=True).stdout
    body = [l for l in sass.splitlines() if re.match(r"\s+/\*[0-9a-f]{4,}\*/", l)]
    hist = collections.Counter()
    for l in body:
        t = re.sub(r"^\s*/\*[0-9a-f]+\*/\s*", "", l).split()
        op = t[1] if t[0].startswith("@") else t[0]
        hist[op.split(".")[0].rstrip(";")] += 1
    with open(os.path.join(PROF, f"{rnd}_sass_{tag}.txt"), "w") as f:
        f.write(f"# cuobjdump -sass -fun {m.group(0)} libcolosseum_b200.so  ({len(body)} instructions)\n# mnemonic histogram: "
                + ", ".join(f"{k} {v}" for k, v in hist.most_common(24)) + "\n")
        f.write("\n".join(re.sub(r"\s+/\* 0x[0-9a-f]+ \*/\s*$", "", l) for l in body) + "\n")
    print(tag, len(body), dict(hist.most_common(8)))
