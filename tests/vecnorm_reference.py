"""float64 numpy restatement of SB3 1.8 VecNormalize as tb_set_vecnorm states it (include/tennisbot_b200.h): RunningMeanStd with
Chan's update_from_moments, the per-env discounted returns, and the two normalisation formulas.  The batch moments are taken in
float64 from the float32 values (SB3's np.mean of a float32 array sums in float32; the library deliberately does not)."""
import numpy as np


class RunningMeanStd:
    def __init__(self, shape=(), epsilon=1e-4):
        self.mean = np.zeros(shape, np.float64)
        self.var = np.ones(shape, np.float64)
        self.count = float(epsilon)

    def update(self, x):
        x = np.asarray(x, np.float64)
        self.update_from_moments(x.mean(axis=0), x.var(axis=0), x.shape[0])

    def update_from_moments(self, batch_mean, batch_var, batch_count):
        delta = batch_mean - self.mean
        tot = self.count + batch_count
        new_mean = self.mean + delta * batch_count / tot
        m2 = self.var * self.count + batch_var * batch_count + np.square(delta) * self.count * batch_count / tot
        self.mean, self.var, self.count = new_mean, m2 / tot, tot


def normalize(x, mean, var, epsilon, clip):
    """clip((x - mean) / sqrt(var + epsilon), -clip, clip) in float64, rounded once to float32."""
    return np.clip((np.asarray(x, np.float64) - mean) / np.sqrt(var + epsilon), -clip, clip).astype(np.float32)


class VecNormalizeRef:
    def __init__(self, num_envs, obs_dim, training=True, norm_obs=True, norm_reward=True, clip_obs=10.0, clip_reward=10.0,
                 gamma=0.99, epsilon=1e-8, record=None):
        self.training, self.norm_obs, self.norm_reward = training, norm_obs, norm_reward
        self.clip_obs, self.clip_reward, self.gamma, self.epsilon = clip_obs, clip_reward, gamma, epsilon
        self.obs_rms, self.ret_rms = RunningMeanStd((obs_dim,)), RunningMeanStd(())
        self.returns = np.zeros(num_envs, np.float64)
        if record is not None:
            self.load(record)

    def reset(self, obs, mask=None):
        """A reset of the envs in mask (all if None): returns zeroed; a full reset folds its observation when training."""
        if mask is None:
            self.returns[:] = 0.0
            if self.training and self.norm_obs:
                self.obs_rms.update(obs)
        else:
            self.returns[np.asarray(mask, bool)] = 0.0

    def step(self, next_obs, reward, done):
        """VecNormalize.step_wait after the env step: the statistics updates; returns the normalised reward."""
        if self.training and self.norm_obs:
            self.obs_rms.update(next_obs)
        if self.training:
            self.returns = self.returns * self.gamma + np.asarray(reward, np.float32)
            self.ret_rms.update(self.returns)
        r = self.normalize_reward(reward)
        self.returns[np.asarray(done, bool)] = 0.0
        return r

    def normalize_obs(self, obs):
        if not self.norm_obs:
            return np.asarray(obs, np.float32)
        return normalize(obs, self.obs_rms.mean, self.obs_rms.var, self.epsilon, self.clip_obs)

    def normalize_reward(self, reward):
        if not self.norm_reward:
            return np.asarray(reward, np.float32)
        return normalize(reward, 0.0, self.ret_rms.var, self.epsilon, self.clip_reward)

    def record(self):
        """The statistics in tb_get_vecnorm's layout (TB_VECNORM_WORDS)."""
        o, r = self.obs_rms, self.ret_rms
        return np.concatenate([o.mean, o.var, [o.count, float(r.mean), float(r.var), r.count]])

    def load(self, rec):
        rec = np.asarray(rec, np.float64)
        od = (rec.size - 4) // 2
        self.obs_rms.mean, self.obs_rms.var, self.obs_rms.count = rec[:od].copy(), rec[od:2 * od].copy(), float(rec[2 * od])
        self.ret_rms.mean, self.ret_rms.var, self.ret_rms.count = float(rec[2 * od + 1]), float(rec[2 * od + 2]), float(rec[2 * od + 3])


def record_formula(rec, obs_dim, raw_obs, epsilon, clip_obs):
    """The normalised observation the library computes from a raw float32 observation and a record."""
    rec = np.asarray(rec, np.float64)
    return normalize(raw_obs, rec[:obs_dim], rec[obs_dim:2 * obs_dim], epsilon, clip_obs)
