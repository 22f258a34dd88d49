import csv, io, os, subprocess, sys
rep=sys.argv[1]
raw = subprocess.run(["ncu","-i",rep,"--page","source","--csv","--print-source","cuda,sass","--kernel-name","regex:k_inflate_fast"],capture_output=True,text=True).stdout
rows=list(csv.reader(io.StringIO(raw)))
cur=None;hdr=None
lines={}
for r in rows:
    if len(r)==2 and r[0]=="File Path": cur=r[1].split("/")[-1]; continue
    if r and r[0]=="Line No": hdr=r; i_s=hdr.index("# Samples"); i_e=hdr.index("Instructions Executed"); continue
    if hdr is None or len(r)<len(hdr) or r[0]=="": continue
    try: s=int(r[i_s]); e=int(r[i_e])
    except: continue
    if cur=="inflate_fast.cuh":
        a=lines.setdefault(int(r[0]),[0,0]); a[0]+=s; a[1]+=e
    else:
        a=lines.setdefault(-1,[0,0]); a[0]+=s; a[1]+=e
# find phase boundaries by grepping the source
src=open(os.path.join(os.path.dirname(os.path.abspath(__file__)),'..','archive_b200','csrc','inflate_fast.cuh')).read().split('\n')
marks=[]
def find(s):
    for i,l in enumerate(src):
        if s in l: return i+1
    return None
ph=[("helpers(br/lookup)",1,find("FP_DEV void fp_fetch_next")),
    ("fetch_next",find("FP_DEV void fp_fetch_next"),find("FP_DEV void fp_parse_header")),
    ("parse_header",find("FP_DEV void fp_parse_header"),find("FP_DEV void fp_plan_lanes")),
    ("plan",find("FP_DEV void fp_plan_lanes"),find("k_inflate_fast(const")),
    ("kernel prologue/loop top",find("k_inflate_fast(const"),find("// ---------------- tables")),
    ("tables",find("// ---------------- tables"),find("// ---------------- pass A:")),
    ("pass A",find("// ---------------- pass A:"),find("// ---------------- pass A2")),
    ("pass A2",find("// ---------------- pass A2"),find("// ---------------- the chain")),
    ("chain",find("// ---------------- the chain"),find("// ---------------- pass A3")),
    ("A3+scan",find("// ---------------- pass A3"),find("// ---------------- pass C")),
    ("pass C",find("// ---------------- pass C"),find("// ======================= the unit's blocks are decoded")),
    ("post/fetch",find("// ======================= the unit's blocks are decoded"),find("// ---------------- LZ77")),
    ("LZ77",find("// ---------------- LZ77"),find("// ---------------- output:")),
    ("output",find("// ---------------- output:"),len(src)+1)]
ts=sum(v[0] for v in lines.values()); te=sum(v[1] for v in lines.values())
print("total samples",ts,"inst",te)
for name,a,b in ph:
    s=sum(v[0] for k,v in lines.items() if a<=k<b); e=sum(v[1] for k,v in lines.items() if a<=k<b)
    print(f"{name:28s} samples {100*s/ts:5.1f}%  inst {100*e/te:5.1f}%  ({e/16384:9.0f} warp-inst/unit)")
s,e=lines.get(-1,[0,0]); print(f"{'other files(intrinsics)':28s} samples {100*s/ts:5.1f}%  inst {100*e/te:5.1f}%")
print()
a=find("// ---------------- LZ77"); b=find("// ---------------- output:")
for k in sorted(lines):
    if a<=k<b and lines[k][1]>0:
        print(f"{k:5d} inst {lines[k][1]/16384:8.0f}/unit  samples {100*lines[k][0]/ts:4.1f}%  {src[k-1].strip()[:90]}")
