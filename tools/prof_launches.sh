set -x
ncu --metrics gpu__time_duration.sum --clock-control none -c 300 --csv --log-file gpurun_out/launches_r01g.csv python bench.py --steps 2 --warmup 3 --no-cpu-baseline > gpurun_out/ncu_g.log 2>&1
python - <<'E'
import subprocess, os, json
env=dict(os.environ); env["LD_LIBRARY_PATH"]="oracle/_ref:mnn_b200:"+env.get("LD_LIBRARY_PATH","")
for plug in (0,1):
    e=dict(env)
    if plug: e["REFDUMP_PLUGIN"]=os.path.abspath("oracle/_ref/libmnn_b200_plugin.so")
    r=subprocess.run(["oracle/_ref/refdump","bench","tests/golden/mbv2_int8.mnn","32","32","3","20"],env=e,capture_output=True,text=True)
    print("plugin" if plug else "cpu", [l for l in r.stdout.splitlines() if l.startswith("{")], r.stderr[-300:])
E
