#!/bin/bash
# Dense keys (DNG_DENSE) measured: the card, the dense-key GPU tests, output
# parity of the two arms (bench.py --dump-outputs), then alternating bench runs
# of DNG_DENSE=0 and 1 (and one each of the variants 3 = hashed path inline,
# 5 = lanes of a counter added up first).
#   tools/gpu_dense_ab.sh [OUTDIR]     (default: a new temporary directory)
cd "$(dirname "$0")/.."
out=${1:-$(mktemp -d)}
echo "outputs: $out"
mkdir -p $out
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $out/gpu.txt
cat $out/gpu.txt
timeout 900 python -m pytest tests/test_dense_keys.py -x -q -m gpu > $out/t_dense.log 2>&1
echo "dense tests rc=$?"; tail -3 $out/t_dense.log
for d in 0 1; do
	DNG_DENSE=$d timeout 600 python bench.py --gpus 1 --steps 10 --warmup 3 \
	    --dump-outputs $out/dump$d > $out/dump$d.json 2> $out/dump$d.err
	echo "dump $d rc=$?"
done
diff -r $out/dump0 $out/dump1 > /dev/null && echo "dumps identical" || echo "DUMPS DIFFER"
for r in 1 2 3; do
	for d in 0 1; do
		DNG_DENSE=$d timeout 600 python bench.py --gpus 1 --steps 10 \
		    --warmup 3 > $out/b${d}_$r.json 2> $out/b${d}_$r.err
		echo "bench dense=$d run=$r rc=$?"
	done
done
for d in 3 5; do
	DNG_DENSE=$d timeout 600 python bench.py --gpus 1 --steps 10 --warmup 3 \
	    --cfg-steps 0 > $out/b${d}_1.json 2> $out/b${d}_1.err
	echo "bench dense=$d rc=$?"
done
