"""Command-line / YAML configuration surface of the hot path.

Same flags, defaults and destinations as the reference's global ``parser``
(engine/config/__init__.py:6-260); only options that the feature-bank training path can act on are
validated.  As in the reference, YAML sweep files inject keys through ``argparse.Namespace`` and thus
bypass ``choices`` (that is how ``text_type: gpt3_cupl`` works there), so ``choices`` are advisory.
"""
import argparse

from . import defaults

DATASETS = ["imagenet", "caltech101", "dtd", "eurosat", "fgvc_aircraft", "food101", "oxford_flowers",
            "oxford_pets", "stanford_cars", "sun397", "ucf101", "imagenetv2", "imagenet_sketch", "imagenet_a",
            "imagenet_r"]

parser = argparse.ArgumentParser()
_add = parser.add_argument

# directories
_add("--data_dir", type=str, default=defaults.DATA_DIR, help="where the dataset is saved")
_add("--indices_dir", type=str, default=defaults.FEW_SHOT_DIR, help="where the (few-shot) indices are saved")
_add("--description_dir", type=str, default=defaults.DESCRIPTION_DIR, help="where the text descriptions are saved")
_add("--feature_dir", type=str, default=defaults.FEATURE_DIR, help="where pre-extracted features live")
_add("--result_dir", type=str, default=defaults.RESULT_DIR, help="where to save experiment results")
# dataset
_add("--dataset", type=str, default="fgvc_aircraft", help="dataset name")
_add("--train-shot", type=int, default=1, help="number of train shots (-1 = full data)")
_add("--max-val-shot", type=int, default=4, help="val shots = min(max_val_shot, train_shot)")
_add("--seed", type=int, default=1, help="seed number")
# encoders (only their names / feature widths matter here; extraction is offline)
_add("--clip-encoder", type=str, default="RN50", help="CLIP encoder the banks were extracted with")
_add("--vision-model", type=str, default="", help="vision encoder the image bank was extracted with")
_add("--language-model", type=str, default="", help="language encoder the text bank was extracted with")
_add("--descriptor_type", type=str, default=None)
_add("--text-augmentation", type=str, default="vanilla")
_add("--image-augmentation", type=str, default="crop", help="crop | flip (deterministic views only)")
_add("--batch-size", type=int, default=32, help="batch size for evaluation")
_add("--num-workers", type=int, default=4,
     help="kept for the sampler RNG protocol: >0 draws the permutation when the iterator is built")
# training
_add("--text_shot", default=None, help="text rows per class: int, 'average' or None (all)")
_add("--custom-name", default="", help="custom name for the experiment save_dir")
_add("--modality", type=str, default="image", choices=["crossmodal", "image", "text"])
_add("--classifier_init", type=str, default="zeroshot", choices=["zeroshot", "random"])
_add("--text_type", type=str, default="hand_crafted")
_add("--logit", type=float, default=4.60517, help="logit scale (exp(logit) is the inverse softmax temperature)")
_add("--hyperparams", type=str, default="linear", help="hyperparams sweep preset")
_add("--eval_test", action="store_true", default=False)
_add("--alpha", type=float, default=0.0, help="weight of the text loss during crossmodal training")
_add("--flip_projection", type=bool, default=False)
_add("--common_dim", type=int, default=0, help="common dimension")
# additions of this implementation
_add("--dp-sampler", type=str, default="global", choices=["global", "sharded"],
     help="data-parallel runs (torchrun): 'global' = every rank draws the reference's global permutation and takes its "
          "slice of each batch (bit-exact order); 'sharded' = every rank owns a strided row shard of the banks and "
          "shuffles it itself (the sampler cost drops by the number of ranks)")
_add("--precision", type=str, default="auto", choices=["auto", "fp32", "bf16"],
     help="fp32 = exact SIMT kernels, bf16 = tcgen05 tensor-core kernels, auto = by batch size")
_add("--sweep-batched", action="store_true", default=False,
     help="train the hyper-parameter combinations of the sweep in lock step on one GPU (one step of all heads = four "
          "launches) instead of one after the other; every combination gets its own seeded sampler stream")
_add("--sweep-batched-adapter", action="store_true", default=False,
     help="--sweep-batched, and the combinations whose heads have an image adapter or learnable temperatures (preset "
          "'linear') also train in lock step (five launches per step of all heads) instead of one after the other")
_add("--grad-diagnostics", action="store_true", default=False,
     help="log the reference's gradient probes (train/grad_direction_sim, img_grad_norm, txt_grad_norm, "
          "grad_agreement_rate): every step for batched sweep groups, at evaluation cadence for single runs")
