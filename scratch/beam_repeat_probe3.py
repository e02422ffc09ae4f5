import os, sys, collections
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from handwritten_math_ocr_api_b200 import FormulaRecognitionModel
from handwritten_math_ocr_api_b200.layout import ModelConfig
from handwritten_math_ocr_api_b200.synthetic import synth_images, synth_state_dict
cfg = ModelConfig()
m = FormulaRecognitionModel(cfg.vocab_size)
m.load_state_dict(synth_state_dict(cfg, seed=0))
N = int(sys.argv[1]); NIMG = int(sys.argv[2]); BEAM = int(sys.argv[3]); SPL = int(sys.argv[4]) if len(sys.argv) > 4 else 0
GREEDY = BEAM == 0
if GREEDY:
    BEAM = 1
if SPL:
    m.set_option("steps_per_launch", SPL)
imgs = synth_images(8, seed=99).cuda().repeat((NIMG + 7) // 8, 1, 1, 1)[:NIMG].contiguous()
feats = m.encoder(imgs)
per_image = [collections.Counter() for _ in range(NIMG)]
for rep in range(N):
    if GREEDY:
        sc = m.generate(encoder_out=feats, max_len=70, return_logprobs=True)[2].sum(1)
    elif BEAM == 1:     # beam 1 through the beam kernel: n-best returns the scores generate() does not
        sc = m.generate_nbest(encoder_out=feats, beam_size=1, max_len=70)[1][:, 0]
    else:
        sc = m.generate(encoder_out=feats, max_len=70, beam_size=BEAM)[3]
    for i, v in enumerate(sc.tolist()):
        per_image[i][v] += 1
multi = [(i, dict(c)) for i, c in enumerate(per_image) if len(c) > 1]
print(f"{'greedy kernel ' if GREEDY else ''}beam {BEAM} images {NIMG} spl {SPL}: images with more than one score value: {len(multi)} of {NIMG}; deviating runs: {sum(sum(c.values()) - max(c.values()) for _, c in [(i, per_image[i]) for i in range(NIMG)])}")
