"""Hyper-parameters of the RecNet hot path.

Attribute names and default values follow the reference's ``config.py`` (TrainConfig, config.py:27-93;
EvalConfig, config.py:160-173) so that code written against ``from config import TrainConfig as C`` keeps
working; everything that only served the reference's data loading, logging and checkpoint naming is left
out (out of scope, SURVEY.md section 2).  Additions: ``precision``, ``optimizer_impl`` and the two ``*_attn_softmax`` switches.
"""


class TrainConfig:
    # --- model selection (config.py:28-33) ---
    model = "RecNet"
    corpus = "MSVD"
    encoder_model = "InceptionV4"
    decoder_model = "GRU"            # [ "LSTM", "GRU" ]  (reference default; published runs used LSTM)
    reconstructor_model = "LSTM"     # [ "LSTM", "GRU" ]
    device = "cuda"

    # --- B200 additions ---
    precision = "bf16"               # "bf16": tcgen05 GEMMs, fp32 accumulate/state; "fp32": FFMA parity build
    optimizer_impl = "recnet"        # "recnet": optim.ClipAdam (own fused clip + Adam kernels, measured 21 us/step faster);
    #                                  "torch": torch.optim.Adam(fused, capturable) + clip_grad_norm_.  RECNET_OPTIMIZER overrides.

    # --- batch / vocabulary (config.py:48-56) ---
    min_count = 5
    caption_max_len = 30
    batch_size = 100
    init_word2idx = {'<PAD>': 0, '<SOS>': 1, '<EOS>': 2}

    # --- embedding (config.py:57-59) ---
    embedding_size = 468
    embedding_dropout = 0.5
    embedding_scale = 1

    # --- encoder features (config.py:62-63) ---
    encoder_output_size = 1536
    encoder_output_len = 28

    # --- decoder (config.py:66-71) ---
    decoder_n_layers = 1
    decoder_hidden_size = 512
    decoder_attn_size = 128
    decoder_dropout = 0.5
    decoder_out_dropout = 0.5
    decoder_teacher_forcing_ratio = 1.0
    decoder_attn_softmax = False     # B200 addition: True = the paper's softmax attention; False = the reference's mean (SURVEY.md 0.1)

    # --- reconstructor (config.py:74-82) ---
    use_recon = True
    reconstructor_type = "local"     # [ "global", "local" ]
    reconstructor_n_layers = 1
    reconstructor_hidden_size = 1536
    reconstructor_decoder_dropout = 0.5
    reconstructor_dropout = 0.5
    reconstructor_attn_size = 128
    reconstructor_attn_softmax = False   # B200 addition, local reconstructor only: as decoder_attn_softmax

    # --- optimisation (config.py:85-94) ---
    n_iterations = 100000
    decoder_learning_rate = 1e-5
    reconstructor_learning_rate = 1e-6
    decoder_weight_decay = 1e-5
    reconstructor_weight_decay = 1e-5
    decoder_use_amsgrad = True
    reconstructor_use_amsgrad = False
    use_gradient_clip = True
    gradient_clip = 50.0

    # --- search (config.py:97) ---
    search_methods = ["greedy", ("beam", 5)]


class EvalConfig:
    corpus = "MSVD"
    encoder_model = "InceptionV4"
    device = "cuda"
