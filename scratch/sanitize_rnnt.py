"""Small RNNT pass for compute-sanitizer (memcheck / racecheck): tiny RNNT model (2 LSTM layers), a ragged batch
with a T' = 1 clip and frames that reach max_symbols (blank bias 11), through pk_transcribe_batch and pk_decode.
    compute-sanitizer --tool memcheck python scratch/sanitize_rnnt.py"""
import os, sys, tempfile
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'oracle'), os.path.join(ROOT, 'tests')]
os.environ.setdefault('PK_GRAPH', '0')
import __graft_entry__ as ge
pkg = ge.load_package()
from parakeet_cpp_b200 import synth
import rnnt_oracle as RO
td = tempfile.mkdtemp()
wp = os.path.join(td, 'tiny_rnnt.safetensors')
synth.save_safetensors(wp, synth.make_weights(RO.make_tiny_rnnt_config(), seed=3, blank_bias=11.0))
e = pkg.Engine(pkg.make_tiny_rnnt_config(), wp, 0)
pcms = [synth.make_audio(32000, 21), synth.make_audio(20000, 22), synth.make_audio(400, 23)]
print('rnnt', [len(t) for t in e.transcribe_batch(pcms, pkg.Decoder.RNNT)], 'truncated', e.truncated_count())
encs = e.encode(e.mel(pcms))
print('rnnt decode', [len(t) for t in e.decode(encs, pkg.Decoder.RNNT)])
e.close()
print('done')
