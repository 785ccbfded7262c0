"""CPU restatement of the unimodal DINO step for the LeNet-style CentralNet encoders (ImageEncoderCentral, SpectrogramEncoderCentral).
TEST INFRASTRUCTURE ONLY.  The step itself is tests/unimodal_dino_ref.py::unimodal_dino_step; this module supplies the two encoders
and registers them in its kind table (unimodal_dino_ref.UNIMODAL_KINDS) on import, so that UniModalDinoState(kind="image_central" |
"spectrogram_central") and unimodal_dino_step work for them.  The encoder forwards are the pinned oracle.dino_ref.central_image_features
/ central_audio_features under the `encoder` prefix; their layer code is checked against the reference's goldens through multi_central.
The parameter specs include the unused fc1 / fc2 classifier heads, so that EMA and checkpoints can be compared."""
import unimodal_dino_ref as U
from oracle import dino_ref as R


def _central_branch_spec(branch, O):
    """One branch of oracle.dino_ref.central_encoder_spec under `encoder.`, in the module's declaration order:
    encoder.0.{conv,bn}{k}, the unused encoder.0.fc1 / fc2, encoder.1 = Linear(flat, O)."""
    pre = f"{branch}_encoder."
    return [("encoder." + n[len(pre):], s) for n, s in R.central_encoder_spec(O, O) if n.startswith(pre)]


def central_image_spec(O=256):
    return _central_branch_spec("image", O)


def central_audio_spec(O=256):
    return _central_branch_spec("audio", O)


def central_image_bn_names():
    return ["encoder.0.bn1", "encoder.0.bn2"]


def central_audio_bn_names():
    return [f"encoder.0.bn{k}" for k in (1, 2, 3, 4)]


def image_central_encoder(img, p, buf, train=True):
    """ImageEncoderCentral.forward: dino_ref.central_image_features(pre="encoder") -- two conv5 blocks, flatten, encoder.1."""
    return R.central_image_features(img, p, buf, pre="encoder", train=train)


def spectrogram_central_encoder(spec, p, buf, train=True):
    """SpectrogramEncoderCentral.forward: dino_ref.central_audio_features(pre="encoder") -- four conv5 blocks, flatten, encoder.1."""
    return R.central_audio_features(spec, p, buf, pre="encoder", train=train)


# kind -> (encoder parameter spec, BatchNorm names, encoder forward), the layout of unimodal_dino_ref.UNIMODAL_KINDS
CENTRAL_KINDS = {"image_central": (central_image_spec, central_image_bn_names, image_central_encoder),
                 "spectrogram_central": (central_audio_spec, central_audio_bn_names, spectrogram_central_encoder)}
U.UNIMODAL_KINDS.update(CENTRAL_KINDS)
