"""VQA model around the PC-DARTS image encoder — B200 drop-in for darts_vqa/vqa_model.py.

VqaModel(embed_size, qst_vocab_size, ans_vocab_size, word_embed_size, num_layers, hidden_size,
img_encoder_type='darts') keeps the reference's sub-module names (img_encoder.darts / img_encoder.fc /
qst_encoder.{word2vec,lstm,fc1,fc2} / fc1 / fc2), construction order (so a seeded init matches the
reference's) and methods: forward, generate, new, _loss, genotype, arch_parameters,
save/load_arch_parameters.

The image encoder's search network runs on the fused sm_100a kernels (pcdarts/model_search.py).  The
question LSTM, the embedding, the small fusion head and the losses are ordinary dense fp32 torch ops
on the same device (SURVEY.md §8f ranks fusing the vocabulary projection as the next step).  The VGG
encoder of the reference (`img_encoder_type='vgg'`) is outside this path and not provided.
"""
import torch
import torch.nn as nn

import config
import pcd_ops
from pcd_ops import decode_question, linear_3xtf32, lstm_forward, vocab_cross_entropy
from pcdarts.model_search import Network


class DartsEncoder(nn.Module):
    """Search network -> Linear(256*7*7, embed) -> x / ||x||_2.detach()  (vqa_model.py:47-66)."""

    def __init__(self, embed_size, init_ch=16, layers=4):
        super().__init__()
        self.darts = Network(init_ch, embed_size, layers)
        self.fc = nn.Linear(self.darts.output_ch * self.darts.output_size ** 2, embed_size)

    def forward(self, image):
        feat = linear_3xtf32(self.darts(image), self.fc.weight, self.fc.bias)      # 12544 -> 512 on the tensor cores (split-K)
        return feat.div(feat.norm(p=2, dim=1, keepdim=True).detach())


class DerivedEncoder(DartsEncoder):
    """The network DERIVED from a searched genotype (pcdarts/model.py NetworkDerived) -> Linear -> x / ||x||_2.detach(): the
    image encoder of the VQA model trained after the search.  The network sits under the same attribute name, `darts`."""

    def __init__(self, embed_size, network):
        nn.Module.__init__(self)
        self.darts = network
        self.fc = nn.Linear(network.output_ch * network.output_size ** 2, embed_size)


def get_img_encoder(img_encoder_type, embed_size):
    if img_encoder_type == 'darts':
        return DartsEncoder(embed_size)
    if img_encoder_type == 'derived':
        raise ValueError("a derived image encoder is built from a search model: vqa_model.derive_vqa(search_model)")
    if img_encoder_type == 'vgg':
        raise NotImplementedError("the VGG19 encoder (vqa_model.py:8-45) is outside the PC-DARTS search path")
    raise Exception(f'Unrecognized encoder type: {img_encoder_type}')


class QstEncoder(nn.Module):
    """Embedding -> tanh -> LSTM seeded with the image embedding -> question feature + per-step vocabulary
    logits (vqa_model.py:77-196; QstEncoderBase and QstEncoder merged, names unchanged)."""

    def __init__(self, qst_vocab_size, word_embed_size, embed_size, num_layers, hidden_size,
                 deterministic=True, temperature=0.1, max_length=30, beam_size=1, end_token=None, length_penalty=0.0):
        super().__init__()
        self.hidden_size = hidden_size
        self.deterministic = deterministic
        self.temperature = temperature
        self.max_length = max_length
        self.beam_size = beam_size          # > 1: deterministic decoding by beam search; generate() returns the best beam
        self.end_token = end_token          # set (<end> = 3): words after it are <pad> = 0, and the decode stops early
        self.length_penalty = length_penalty    # beams with end_token: ranked by log-probability / length^length_penalty
        self.word2vec = nn.Embedding(qst_vocab_size, word_embed_size)
        self.tanh = nn.Tanh()
        self.lstm = nn.LSTM(word_embed_size, hidden_size, num_layers)
        self.fc1 = nn.Linear(hidden_size, qst_vocab_size)
        self.softmax = nn.Softmax(dim=2)
        nn.init.xavier_uniform_(self.fc1.weight.data)
        nn.init.zeros_(self.fc1.bias)
        self.fc2 = nn.Linear(2 * num_layers * hidden_size, embed_size)
        nn.init.xavier_uniform_(self.fc2.weight.data)
        nn.init.zeros_(self.fc2.bias)

    def forward(self, question, image_embedding, return_states=False):
        self.lstm.flatten_parameters()
        h0 = image_embedding.view(1, -1, self.hidden_size)
        # alpha-only passes (pcd_ops.weight_grads(False)): nothing behind the word embedding is differentiated, so the LSTM's
        # input-gradient GEMM is not asked for either
        with torch.set_grad_enabled(torch.is_grad_enabled() and pcd_ops.weight_grads_enabled()):
            words = self.tanh(self.word2vec(question)).transpose(0, 1)          # T x B x E (teacher forcing)
        out, (hidden, cell) = lstm_forward(self.lstm, words, h0, h0)      # persistent recurrence kernels + tcgen05 GEMMs
        feat = torch.cat((hidden, cell), 2).transpose(0, 1)
        feat = linear_3xtf32(self.tanh(feat.reshape(feat.size(0), -1)), self.fc2.weight, self.fc2.bias)
        states = self.tanh(out.transpose(0, 1))                              # B x T x H, input of the vocabulary projection
        if return_states:
            return feat, states
        # vocabulary projection (35 GFLOP at B=64): tcgen05 tensor cores, fp32-accurate 3xTF32 split
        return feat, linear_3xtf32(states, self.fc1.weight, self.fc1.bias)

    def next_word_loss(self, states, question):
        """CE(fc1(states)[:, :-1], question[:, 1:]) (vqa_model.py:356-358), projection and loss fused: the last time step
        is masked out instead of sliced away."""
        targets = torch.cat((question[:, 1:], question.new_full((question.size(0), 1), -100)), dim=1)
        return vocab_cross_entropy(states, self.fc1.weight, self.fc1.bias, targets)

    def sample(self, prob):
        if self.deterministic:
            return torch.argmax(prob, 2)
        soft = self.softmax(prob / self.temperature)
        return torch.multinomial(soft[:, 0, :], 1)

    def generate(self, image_embedding):
        """Greedy / sampled / beam-search 30-step decode from the <start> token (index 2)  (vqa_model.py:103-136)."""
        batch = len(image_embedding)
        h0 = image_embedding.reshape(batch, self.hidden_size)
        qst = decode_question(h0, self.lstm, self.word2vec, self.fc1, self.max_length, self.deterministic, self.temperature,
                              self.beam_size, self.end_token, self.length_penalty)
        if qst is not None:
            return qst
        # sampled decoding outside the kernel's envelope is the reference's module loop (torch.multinomial), as is any other
        # falsy `deterministic` with an overridden sample()
        self.lstm.flatten_parameters()
        h = image_embedding.view(1, -1, self.hidden_size)
        state = (h, h)
        word = torch.full((batch, 1), 2, dtype=torch.long, device=image_embedding.device)
        current = self.tanh(self.word2vec(word)).transpose(0, 1)
        qst = torch.zeros((batch, self.max_length), dtype=torch.long, device=image_embedding.device)
        for t in range(self.max_length):
            out, state = self.lstm(current, state)
            pred = self.sample(self.fc1(self.tanh(out.transpose(0, 1))))
            current = self.word2vec(pred).transpose(0, 1)
            qst[:, t] = pred[:, 0]
        return qst


class VqaModelBase(nn.Module):
    def __init__(self, embed_size, qst_vocab_size, ans_vocab_size, word_embed_size, num_layers, hidden_size,
                 img_encoder_type='vgg'):
        super().__init__()
        self.embed_size = embed_size
        self.qst_vocab_size = qst_vocab_size
        self.ans_vocab_size = ans_vocab_size
        self.word_embed_size = word_embed_size
        self.num_layers = num_layers
        self.hidden_size = hidden_size
        self.criterion = nn.CrossEntropyLoss()
        self.img_encoder_type = img_encoder_type
        self.img_encoder = get_img_encoder(img_encoder_type, embed_size)
        # the contract is fp32 (rel 1e-4): keep cuDNN's LSTM off TF32 (torch enables it by default)
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False

    def genotype(self):
        return self.img_encoder.darts.genotype()

    def arch_parameters(self):
        return self.img_encoder.darts.arch_parameters()

    def save_arch_parameters(self, save_path):
        if self.img_encoder_type == 'darts':
            self.img_encoder.darts.save_arch_parameters(save_path)

    def load_arch_parameters(self, load_path):
        if self.img_encoder_type == 'darts':
            self.img_encoder.darts.load_arch_parameters(load_path)


class VqaModel(VqaModelBase):
    """Question and answer heads on the shared image embedding (vqa_model.py:279-364)."""

    def __init__(self, embed_size, qst_vocab_size, ans_vocab_size, word_embed_size, num_layers, hidden_size,
                 img_encoder_type='vgg'):
        super().__init__(embed_size, qst_vocab_size, ans_vocab_size, word_embed_size, num_layers, hidden_size,
                         img_encoder_type)
        self.qst_encoder = QstEncoder(qst_vocab_size, word_embed_size, embed_size, num_layers, hidden_size)
        self.tanh = nn.Tanh()
        self.dropout = nn.Dropout(0.5)
        self.fc1 = nn.Linear(embed_size, ans_vocab_size)
        self.fc2 = nn.Linear(ans_vocab_size, ans_vocab_size)

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
        qst_feature, _ = self.qst_encoder(qst, img_feature)
        return qst, self._answer(img_feature, qst_feature)

    def new(self):
        twin = VqaModel(self.embed_size, self.qst_vocab_size, self.ans_vocab_size, self.word_embed_size,
                        self.num_layers, self.hidden_size, self.img_encoder_type)
        twin.img_encoder.darts = self.img_encoder.darts.new()
        twin.to(config.DEVICE)
        return twin

    def _loss(self, images, questions, labels, qst_only=False):
        """vqa_model.py:351-364; same value and gradients as CE on `self(images, questions)`, but the question logits stay
        inside the fused projection + cross-entropy op."""
        return self._loss_staged(images, questions, labels, qst_only)[0]

    def _loss_staged(self, images, questions, labels, qst_only=False):
        """(loss, image embedding): the embedding is the only tensor through which the loss depends on the image encoder, so
        a data-parallel backward can be cut there (pcd_dist.staged_grads: the all-reduce of the question-encoder / head
        gradients runs while the search network's backward is still computing)."""
        img_feature = self.img_encoder(images)
        qst_feature, states = self.qst_encoder(questions, img_feature, return_states=True)
        qst_loss = self.qst_encoder.next_word_loss(states, questions)
        if qst_only:
            return qst_loss, img_feature
        return self.criterion(self._answer(img_feature, qst_feature), labels) + qst_loss, img_feature


def derive_vqa(search_model, layers=None):
    """A freshly initialised VqaModel with the dimensions of `search_model` whose image encoder is the network its genotype
    describes (pcdarts.model.derive; `layers` overrides the depth).  As in DARTS, the derived network is trained from
    scratch: nothing but the genotype is taken over.  genotype() returns it, arch_parameters() is empty.  new() (the unrolled
    twin of an architecture search) does not apply."""
    from pcdarts.model import derive
    m = VqaModel(search_model.embed_size, search_model.qst_vocab_size, search_model.ans_vocab_size,
                 search_model.word_embed_size, search_model.num_layers, search_model.hidden_size, img_encoder_type='darts')
    m.img_encoder = DerivedEncoder(search_model.embed_size, derive(search_model.img_encoder.darts, layers))
    m.img_encoder_type = 'derived'
    device = next(search_model.parameters()).device
    return m.to(device)
