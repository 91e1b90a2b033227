"""EF model of the 3-stage LCT system (basic_vqa/models_lct.py:9-267): PC-DARTS image encoder (the search network, on the
sm_100a kernels) + question LSTM (seeded with the image embedding) + fusion head, with the question decoder that
`generate()`s the pseudo questions.  Same class / attribute / state_dict names and registration order as the reference
(note QstEncoder.fc1 / fc2 are swapped with respect to darts_vqa/vqa_model.py)."""
import torch
import torch.nn as nn

import config
import pcd_ops
from pcd_ops import decode_question, linear_3xtf32, lstm_forward, vocab_cross_entropy
from pcdarts.model_search import Network


def _copy_dropout(src, dst):
    """model.new() builds fresh modules; carry the dropout probabilities over (they are configuration, not state)."""
    probs = {n: m.p for n, m in src.named_modules() if isinstance(m, nn.Dropout)}
    for n, m in dst.named_modules():
        if isinstance(m, nn.Dropout) and n in probs:
            m.p = probs[n]


class ImgEncoder(nn.Module):
    def __init__(self, embed_size, vqa_model=None, init_ch=16, layers=4):
        super().__init__()
        self.darts = Network(init_ch, embed_size, layers) if vqa_model is None else Network(init_ch, embed_size, layers, vqa_model)
        self.fc = nn.Linear(self.darts.output_ch * self.darts.output_size ** 2, embed_size)

    def forward(self, image):
        feat = linear_3xtf32(self.darts(image), self.fc.weight, self.fc.bias)
        return feat.div(feat.norm(p=2, dim=1, keepdim=True).detach())


class QstEncoder(nn.Module):
    def __init__(self, qst_vocab_size, word_embed_size, embed_size, num_layers, hidden_size, deterministic=True,
                 temperature=0.1, max_length=30, beam_size=1, end_token=None, length_penalty=0.0,
                 top_k=0, top_p=1.0):
        super().__init__()
        self.hidden_size = hidden_size
        self.deterministic = deterministic
        self.temperature = temperature
        self.max_length = max_length
        self.beam_size = beam_size          # > 1: deterministic decoding by beam search; generate() returns the best beam
        self.end_token = end_token          # set (<end> = 3): words after it are <pad> = 0, and the decode stops early
        self.length_penalty = length_penalty    # beams with end_token: ranked by log-probability / length^length_penalty
        self.top_k = top_k                  # sampling (deterministic=False) only: draw among the top_k most likely words (0: all)
        self.top_p = top_p                  # sampling only: draw within the nucleus of probability top_p (1: all)
        self.word2vec = nn.Embedding(qst_vocab_size, word_embed_size)
        self.tanh = nn.Tanh()
        self.lstm = nn.LSTM(word_embed_size, hidden_size, num_layers)
        self.fc1 = nn.Linear(2 * num_layers * hidden_size, embed_size)
        self.fc2 = nn.Linear(hidden_size, qst_vocab_size)
        self.softmax = nn.Softmax(dim=2)
        nn.init.xavier_uniform_(self.fc1.weight.data)
        nn.init.xavier_uniform_(self.fc2.weight.data)
        nn.init.zeros_(self.fc1.bias)
        nn.init.zeros_(self.fc2.bias)

    def forward(self, question, image_embedding, return_states=False):
        self.lstm.flatten_parameters()
        h0 = image_embedding.view(1, -1, self.hidden_size)
        # alpha-only passes (pcd_ops.weight_grads(False)): nothing behind the word embedding is differentiated, so the LSTM's
        # input-gradient GEMM is not asked for either
        with torch.set_grad_enabled(torch.is_grad_enabled() and pcd_ops.weight_grads_enabled()):
            words = self.tanh(self.word2vec(question)).transpose(0, 1)          # T x B x E (teacher forcing)
        out, (hidden, cell) = lstm_forward(self.lstm, words, h0, h0)
        feat = torch.cat((hidden, cell), 2).transpose(0, 1)
        feat = linear_3xtf32(self.tanh(feat.reshape(feat.size(0), -1)), self.fc1.weight, self.fc1.bias)
        states = self.tanh(out.transpose(0, 1))
        if return_states:
            return feat, states
        return feat, linear_3xtf32(states, self.fc2.weight, self.fc2.bias)

    def next_word_loss(self, states, question):
        targets = torch.cat((question[:, 1:], question.new_full((question.size(0), 1), -100)), dim=1)
        return vocab_cross_entropy(states, self.fc2.weight, self.fc2.bias, targets)

    def sample(self, prob):
        if self.deterministic:
            return torch.argmax(prob, 2)
        soft = self.softmax(prob / self.temperature)
        return torch.multinomial(soft[:, 0, :], 1)

    def generate(self, image_embedding):
        """Greedy / sampled / beam-search 30-step decode from <start> = 2 (models_lct.py:124-157); the word choice is not
        differentiable."""
        batch = len(image_embedding)
        h0 = image_embedding.reshape(batch, self.hidden_size)
        qst = decode_question(h0, self.lstm, self.word2vec, self.fc2, self.max_length, self.deterministic, self.temperature,
                              self.beam_size, self.end_token, self.length_penalty, self.top_k, self.top_p)
        if qst is not None:
            return qst
        # sampled decoding outside the kernel's envelope: the reference's module loop (torch.multinomial)
        self.lstm.flatten_parameters()
        h = image_embedding.view(1, -1, self.hidden_size)
        state = (h, h)
        word = torch.full((batch, 1), 2, dtype=torch.long, device=image_embedding.device)
        current = self.tanh(self.word2vec(word)).transpose(0, 1)
        qst = torch.zeros((batch, self.max_length), dtype=torch.long, device=image_embedding.device)
        for t in range(self.max_length):
            out, state = self.lstm(current, state)
            pred = self.sample(self.fc2(self.tanh(out.transpose(0, 1))))
            current = self.word2vec(pred).transpose(0, 1)       # models_lct.py:152: no tanh after the first word
            qst[:, t] = pred[:, 0]
        return qst


class VqaModel(nn.Module):
    def __init__(self, embed_size, qst_vocab_size, ans_vocab_size, word_embed_size, num_layers, hidden_size, pretrained=True):
        super().__init__()
        if config.ARCH_TYPE != 'darts':
            raise NotImplementedError("the fixed (VGG19) EF encoder is outside the PC-DARTS path; use models.VqaModel-style stock modules")
        self.img_encoder = ImgEncoder(embed_size, self)
        self.qst_encoder = QstEncoder(qst_vocab_size, word_embed_size, embed_size, num_layers, hidden_size)
        self.tanh = nn.Tanh()
        self.dropout = nn.Dropout(0.5)
        self.fc1 = nn.Linear(embed_size, ans_vocab_size)
        self.fc2 = nn.Linear(ans_vocab_size, ans_vocab_size)
        self.criterion = nn.CrossEntropyLoss()
        self.embed_size = embed_size
        self.qst_vocab_size = qst_vocab_size
        self.ans_vocab_size = ans_vocab_size
        self.word_embed_size = word_embed_size
        self.num_layers = num_layers
        self.hidden_size = hidden_size

    def _answer(self, img_feature, qst_feature):
        z = self.dropout(self.tanh(torch.mul(img_feature, qst_feature)))
        z = self.dropout(self.tanh(linear_3xtf32(z, self.fc1.weight, self.fc1.bias)))
        return linear_3xtf32(z, self.fc2.weight, self.fc2.bias)

    def forward(self, img, qst):
        img_feature = self.img_encoder(img)
        qst_feature, qst_out = self.qst_encoder(qst, img_feature)
        return self._answer(img_feature, qst_feature), qst_out

    def generate(self, img):
        img_feature = self.img_encoder(img)
        qst = self.qst_encoder.generate(img_feature)
        qst_feature, _ = self.qst_encoder(qst, img_feature, return_states=True)
        return qst, self._answer(img_feature, qst_feature)

    def genotype(self):
        return self.img_encoder.darts.genotype()

    def arch_parameters(self):
        return self.img_encoder.darts.arch_parameters()

    def _loss(self, images, questions, labels, qst_only=False):
        """models_lct.py:253-260.  `qst_only` is not part of the reference signature: the darts_vqa-flavour Architect that
        get_architect returns under SKIP_STAGE2 passes it (always False there); True keeps only the next-word loss."""
        img_feature = self.img_encoder(images)
        qst_feature, states = self.qst_encoder(questions, img_feature, return_states=True)
        qst_loss = self.qst_encoder.next_word_loss(states, questions)
        if qst_only:
            return qst_loss
        return self.criterion(self._answer(img_feature, qst_feature), labels) + qst_loss

    def new(self):
        twin = VqaModel(self.embed_size, self.qst_vocab_size, self.ans_vocab_size, self.word_embed_size, self.num_layers,
                        self.hidden_size)
        twin.img_encoder.darts = self.img_encoder.darts.new()
        _copy_dropout(self, twin)
        # the unrolled twin generates ArchitectLct's pseudo questions: it decodes the way this model was configured to
        for name in ("deterministic", "temperature", "max_length", "beam_size", "end_token", "length_penalty", "top_k", "top_p"):
            setattr(twin.qst_encoder, name, getattr(self.qst_encoder, name))
        return twin.to(config.DEVICE)
