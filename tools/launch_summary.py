"""Cut ONE hot-path pass out of an ncu launch list (ncu --metrics gpu__time_duration.sum --csv --log-file X.csv ...) and
write profiles/<tag>_launches_<what>.csv (every launch) + profiles/<tag>_launches_<what>_summary.csv (per-kernel totals).

    python tools/launch_summary.py gpurun_out/r1h_launches.csv r1h step "<command that produced it>"

`step`: the launches from one step_advance_kernel up to (not including) the next one = one cfg-2 denoise step (graph replay)."""
import collections, csv, re, sys

src, tag, what, cmd = sys.argv[1], sys.argv[2], sys.argv[3], sys.argv[4]
rows = [r for r in csv.reader(l for l in open(src) if l.startswith('"'))]
h = rows[0]
ki, vi = h.index("Kernel Name"), h.index("Metric Value")
L = []
for r in rows[1:]:
    n = re.sub(r"\(.*$", "", re.sub(r"^void ", "", r[ki]))
    n = re.sub(r"<unnamed>::|\(anonymous namespace\)::|halo::|sweep::|stencil::|vqtc::", "", n)
    L.append((n, float(r[vi].replace(",", "")) / 1000.0))
if what == "decode":   # one quantize + decode pass: from the last vq_kernel launch to the decoder's head (stencil) launch after it
    a = max(i for i, (n, _) in enumerate(L) if n.startswith("vq_kernel") or n.startswith("vq_tc_kernel"))
    b = min(i for i, (n, _) in enumerate(L) if i > a and "conv_stencil" in n)
    seq = L[a:b + 1]
else:
    marks = [i for i, (n, _) in enumerate(L) if n.startswith("step_advance")]
    assert len(marks) >= 2, "need two step_advance launches in the list"
    # the last cfg-2 step: bench.py also replays cfg-4 steps (level-0 self-attention: flash_attn_kernel<64, ...>) later in the run
    segs = [L[a:b] for a, b in zip(marks, marks[1:]) if not any(n.startswith("flash_attn_kernel<64") for n, _ in L[a:b]) and b - a > 100]
    seq = segs[-1]
with open(f"profiles/{tag}_launches_{what}.csv", "w") as f:
    f.write(f"# {tag}: {cmd}\n# " + ("one cfg-3 quantize + decode pass (B=16): vq_kernel .. the decoder's head" if what == "decode" else
            "one cfg-2 denoise step (graph replay): every launch from one step_advance to the next (the update runs in out.conv's epilogue)") + "; cold-cache, serialised times\n")
    f.write("index,kernel,us\n")
    for i, (n, u) in enumerate(seq):
        f.write(f'{i},"{n}",{u:.3f}\n')
tot = sum(u for _, u in seq)
agg = collections.OrderedDict()
for n, u in seq:
    a = agg.setdefault(n, [0, 0.0]); a[0] += 1; a[1] += u
with open(f"profiles/{tag}_launches_{what}_summary.csv", "w") as f:
    f.write(f"# {tag}: per-kernel totals of one " + ("cfg-3 quantize + decode pass" if what == "decode" else "cfg-2 step") + " under ncu (cold-cache, serialised; compare SHARES)\n")
    f.write("# conv_halo_kernel<BLOCK_N, TD, NS, NB, TPS, STAGED, PAIR, CG2, FUSE_UPD>; conv_halo_up_kernel<BLOCK_N, NS, NB, PAIR>; conv_igemm_kernel<BLOCK_N, NSTAGE, KSPLIT>\n")
    f.write("kernel,launches,total_us,share\n")
    for n, (c, u) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
        f.write(f'"{n}",{c},{u:.1f},{u / tot:.4f}\n')
    f.write(f"TOTAL,{len(seq)},{tot:.1f},1.0\n")
print(open(f"profiles/{tag}_launches_{what}_summary.csv").read())
