# usage: bash tools/job_test_bench.sh <tag> [pytest args...]   -- GPU suite, then the bench line under the driver's arguments
cd "${GRAFT_REPO_ROOT:-/root/repo}"
tag=$1; shift
timeout 900 python -m pytest tests -m gpu -x -q "$@" > gpurun_out/${tag}_gputest.log 2>&1; tail -4 gpurun_out/${tag}_gputest.log
show() {
python - "$1" <<PY
import json, sys
d = json.load(open(sys.argv[1]))
print(sys.argv[1], "ms/step %.4f" % d["ms_per_step"], "value %.1fM" % (d["value"] / 1e6), "e2e %.1fM" % (d["e2e"]["value"] / 1e6),
      {k: round(v * 1e3, 1) for k, v in d["roofline"]["phase_ms"].items()}, "frac %.3f" % d["roofline"]["frac"])
PY
}
python bench.py --steps 20 --warmup 5 --no-cpu-baseline --no-extra > gpurun_out/${tag}_bench.json 2> gpurun_out/${tag}_bench.err || tail -5 gpurun_out/${tag}_bench.err
show gpurun_out/${tag}_bench.json
python bench.py --steps 200 --warmup 10 --no-cpu-baseline --no-extra > gpurun_out/${tag}_bench200.json 2> gpurun_out/${tag}_bench200.err || tail -5 gpurun_out/${tag}_bench200.err
show gpurun_out/${tag}_bench200.json
