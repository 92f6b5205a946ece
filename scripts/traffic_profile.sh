#!/bin/bash
# DRAM bytes of every kernel of one multiply+relin pass, L2 state preserved between kernels. usage: traffic_profile.sh <tag>
TAG=$1
python scripts/traffic_case.py > gpurun_out/${TAG}_plain.log 2>&1 &&
ncu --cache-control none --clock-control none --metrics dram__bytes_read.sum,dram__bytes_write.sum -k regex:'k_' --csv --log-file gpurun_out/${TAG}_traffic.csv python scripts/traffic_case.py > gpurun_out/${TAG}_ncu.log 2>&1
python - <<PY
import csv
rows=[r for r in csv.reader(l for l in open("gpurun_out/${TAG}_traffic.csv") if not l.startswith("=="))]
h=rows[0]; ki,mi,ui,vi=h.index("Kernel Name"),h.index("Metric Name"),h.index("Metric Unit"),h.index("Metric Value")
tot={}; 
for r in rows[1:]:
    k=r[ki].split("(")[0].replace("fheb::",""); v=float(r[vi].replace(",",""))*{"byte":1,"Kbyte":1e3,"Mbyte":1e6,"Gbyte":1e9}[r[ui]]
    tot[k]=tot.get(k,0)+v
n=1184*2
print("${TAG}: DRAM KB/op per kernel:", {k: round(v/n/1e3) for k,v in tot.items()}, "total KB/op", round(sum(tot.values())/n/1e3))
PY
