for cfg in "QCE_CHECKSUM_PER_COL=0 QCE_CHECKSUM_WAVES=1" "QCE_CHECKSUM_PER_COL=0 QCE_CHECKSUM_WAVES=2" "QCE_CHECKSUM_PER_COL=0 QCE_CHECKSUM_WAVES=3" "QCE_CHECKSUM_PER_COL=0 QCE_CHECKSUM_WAVES=4" "QCE_CHECKSUM_PER_COL=0 QCE_CHECKSUM_WAVES=5" "QCE_CHECKSUM_PER_COL=1 QCE_CHECKSUM_WAVES=3"; do
  env $cfg python bench.py --config c2 --steps 6 --warmup 3 --no-cpu-baseline > gpurun_out/ck.json 2> gpurun_out/ck.err
  python -c "
import json; d=json.load(open('gpurun_out/ck.json')); k=d['roofline']['kernels_ms_per_step']; print('$cfg', round(d['ms_per_step'],3), 'checksum', k.get('checksum'), d['parity']['full_vs_checker'])"
done
